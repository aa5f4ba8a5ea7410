// Warp-specialised tcgen05 / TMEM / TMA pipeline shared by the encoder GEMMs and the CIR
// search kernel (sm_100a only).
//
//   D[128 x BN] (fp32, TMEM)  =  A[128 x K] (bf16, K-major)  *  B[BN x K]^T (bf16, K-major)
//
// One persistent CTA per SM, 8 warps:
//   warp 0      TMA producer   (one lane): global -> 128B-swizzled smem ring, mbarrier tx
//   warp 1      MMA issuer     (one lane): tcgen05.mma kind::f16, M=128, N=BN, K=16 x4 / stage
//   warp 2      TMEM allocator (2*BN fp32 columns = two accumulator buffers)
//   warps 4..   epilogue       Epi::kWarps = 4 or 8 warps; warp w reads TMEM lanes 32*(w%4)..+31
//                              (hardware rule), so with 8 warps two warps share a row quarter
//                              and split the tile's columns: tcgen05.ld + Epi::tile()
// Three barrier rings: smem full/empty (TMA <-> MMA), TMEM full/empty (MMA <-> epilogue).
// The tile sequence comes from a Sched object that all roles evaluate identically.
//
// CL == 1: a single CTA issues its own M = 128 MMAs on a whole B tile.
// CL == 2: a CTA PAIR (cluster of 2, tcgen05 cta_group::2).  The two CTAs own consecutive M
// tiles (256 rows together) and the same B tile (n0); the even CTA issues M = 256 MMAs, each CTA
// supplies its own 128 rows of A and HALF of the B tile from its own shared memory and receives
// its 128 accumulator rows in its own TMEM.  Against two independent CTAs (or a multicast
// cluster, which still parks the whole B tile in both CTAs) this cuts the shared-memory traffic
// per SM from 192 B/clk (96 operand reads + 96 TMA fills at full tensor rate, above the 128 B/clk
// the SM can move) to 128 B/clk, and the stage footprint from 48 KB to 32 KB (6 stages).  (A
// multicast cluster was ahead for the search kernel while it was HBM / power bound, 1004 vs 940
// TFLOP/s at 10 M rows; with the pacing window of SchedSearch the pair is 3 % ahead.)
// The Sched must give both CTAs of a pair the same tile count and n0.
#pragma once
#include <cuda.h>

#include "ptx.cuh"

namespace ofx {

constexpr int kBM = 128;       // accumulator rows per CTA tile (UMMA M, cta_group::1)
constexpr int kBK = 64;        // bf16 elements per smem row = 128 B = one swizzle span
constexpr int kUmmaK = 16;     // K per tcgen05.mma for 16-bit inputs
constexpr int kEpiWarp0 = 4;   // first epilogue warp (warp % 4 selects the TMEM lane quarter)

template <int BN, int STAGES, int CL = 1>
struct TcCfg {
    static constexpr int kABytes = kBM * kBK * 2;
    static constexpr int kBBytes = BN / CL * kBK * 2;   // pair: each CTA holds half of the B tile
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kStages = STAGES;
    static constexpr int kTmemCols = 2 * BN;  // power of two for BN in {64,128,256}
    static constexpr int kRingBytes = kStages * kStageBytes;
    static constexpr int kBarBytes = 1024;  // barriers + tmem slot; keeps the epilogue smem 1024-byte aligned (TMA swizzle)
};

template <int BN, int STAGES, class Epi, int CL = 1>
constexpr int tc_smem_bytes() {
    return 1024 /*alignment slack*/ + TcCfg<BN, STAGES, CL>::kRingBytes + TcCfg<BN, STAGES, CL>::kBarBytes +
           Epi::kSmemBytes;
}

// Sched concept:
//   struct Params;  __device__ Sched(const Params&, int cta, int n_cta);
//   __device__ bool next();          advance to the next tile of this CTA
//   int m0, n0;                      tile origin (rows of A, rows of B)
//   static constexpr bool kPrefetch; int pf_n0;   optional: B tile to prefetch into L2 (-1 = none)
//   static constexpr bool kThrottle; void throttle();   optional: producer-side pacing hook, called once per tile
// Epi concept:
//   struct Params; static constexpr int kSmemBytes;
//   static constexpr int kWarps;   4 or 8 epilogue warps
//   __device__ void begin(const Params&, const Sched&, int ewarp, int lane, uint8_t* smem);
//   __device__ void end(const Params&, int lane);   after the last tile (e.g. drain bulk stores)
//   __device__ void pre_tile(const Params&, const Sched&, int ewarp, int lane, uint8_t* smem);
//                                   called before waiting for the tile's accumulator
//   __device__ void tile(const Params&, const Sched&, uint32_t tmem_acc /*lane quarter applied*/,
//                        int ewarp /*0..kWarps-1: quarter = ewarp & 3, column group = ewarp >> 2*/,
//                        int lane, uint8_t* epi_smem);
//   (an object per epilogue thread: state such as running top-k thresholds lives in it)
//   using Operand = __half;        optional: fp16 A and B (kind::f16 with F16 inputs); bf16 without it
template <class Epi>
constexpr int tc_threads() { return 128 + 32 * Epi::kWarps; }

template <class Epi, class = void>
struct TcOperand { using type = __nv_bfloat16; };
template <class Epi>
struct TcOperand<Epi, std::void_t<typename Epi::Operand>> { using type = typename Epi::Operand; };

// Debug instrumentation (OFX_TC_PROF=1, gemm.cu): per-CTA cycle counters of the MMA warp
// {total, wait smem-full, wait tmem-empty} and of epilogue warp 0 {total, wait tmem-full}.
__device__ long long* g_tc_prof = nullptr;

template <int BN, int STAGES, int CL, class Sched, class Epi>
__global__ void __launch_bounds__(128 + 32 * Epi::kWarps, 1)
tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
          const typename Sched::Params sp, const __grid_constant__ typename Epi::Params ep,
          const int num_k_blocks) {
    static_assert(CL == 1 || CL == 2, "CL = 1 (single CTA) or 2 (CTA pair)");
    using Cfg = TcCfg<BN, STAGES, CL>;
    constexpr bool kPair = CL == 2;
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte aligned bases
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* s_a = smem;
    uint8_t* s_b = smem + Cfg::kStages * Cfg::kABytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kRingBytes);
    uint64_t* full = bars;                       // [kStages]
    uint64_t* empty = bars + Cfg::kStages;       // [kStages]
    uint64_t* tmem_full = bars + 2 * Cfg::kStages;       // [2]
    uint64_t* tmem_empty = bars + 2 * Cfg::kStages + 2;  // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * Cfg::kStages + 4);
    uint8_t* epi_smem = smem + Cfg::kRingBytes + Cfg::kBarBytes;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t crank = CL > 1 ? cluster_ctarank() : 0u;   // pair: 0 = leader (issues the MMAs)
    constexpr int kBRowsPerCta = BN / CL;  // rows of the B tile this CTA fetches

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < Cfg::kStages; ++i) {
            mbar_init(&full[i], 1);     // pair: the leader's collects the bytes of both CTAs
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tmem_full[i], 1);
            mbar_init(&tmem_empty[i], Epi::kWarps * (kPair ? 2 : 1));  // one arrive per epilogue warp (pair: of both CTAs, on the leader's)
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        if constexpr (kPair) tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
        else tmem_alloc(tmem_slot, Cfg::kTmemCols);
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();  // peers' barriers are initialised before any remote use
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            Sched sched(sp, blockIdx.x, gridDim.x);
            int stage = 0;
            uint32_t phase = 0;
            while (sched.next()) {
                if constexpr (Sched::kThrottle) sched.throttle();
                for (int kb = 0; kb < num_k_blocks; ++kb) {
                    if constexpr (Sched::kPrefetch) {
                        // designated CTAs pull a LATER B tile of the sweep into L2 (this CTA's rows of it)
                        if (sched.pf_n0 >= 0)
                            tma_prefetch_l2_2d(&tm_b, kb * kBK, sched.pf_n0 + static_cast<int>(crank) * kBRowsPerCta);
                    }
                    mbar_wait(&empty[stage], phase ^ 1);
                    if constexpr (!kPair) {
                        mbar_arrive_expect_tx(&full[stage], Cfg::kStageBytes);
                        tma_load_2d(s_a + stage * Cfg::kABytes, &tm_a, &full[stage], kb * kBK, sched.m0);
                        tma_load_2d(s_b + stage * Cfg::kBBytes, &tm_b, &full[stage], kb * kBK, sched.n0);
                    } else {
                        // both CTAs' bytes are accounted on the leader's barrier
                        if (crank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::kStageBytes);
                        const uint32_t bar = mapa_shared(smem_u32(&full[stage]), 0);
                        tma_load_2d_pair(s_a + stage * Cfg::kABytes, &tm_a, bar, kb * kBK, sched.m0, kEvictNormal);
                        tma_load_2d_pair(s_b + stage * Cfg::kBBytes, &tm_b, bar, kb * kBK,
                                         sched.n0 + static_cast<int>(crank) * kBRowsPerCta, kEvictNormal);
                    }
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        // The whole warp walks the schedule (warp-uniform control flow and addresses keep the
        // descriptors in uniform registers); one elected lane issues the tcgen05 instructions
        // back to back.  A lane-0-only loop costs ~20 issue slots per MMA in address traffic
        // between the vector and uniform register files.
        if (!kPair || crank == 0) {
            constexpr uint32_t idesc = umma_idesc_16<typename TcOperand<Epi>::type>(kPair ? 2 * kBM : kBM, BN);
            constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO, version, SW128
            const uint32_t a_lo0 = ((smem_u32(s_a) & 0x3FFFF) >> 4) | (1u << 16);
            const uint32_t b_lo0 = ((smem_u32(s_b) & 0x3FFFF) >> 4) | (1u << 16);
            auto desc = [](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
            Sched sched(sp, blockIdx.x, gridDim.x);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            long long* prof = g_tc_prof;
            long long t0 = clock64(), t_full = 0, t_te = 0, tq;
            while (sched.next()) {
                if (prof) { tq = clock64(); mbar_wait(&tmem_empty[acc], acc_phase ^ 1); t_te += clock64() - tq; }
                else mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < num_k_blocks; ++kb) {
                    if (prof) { tq = clock64(); mbar_wait(&full[stage], phase); t_full += clock64() - tq; }
                    else mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + stage * (Cfg::kABytes >> 4);
                    const uint32_t b_lo = b_lo0 + stage * (Cfg::kBBytes >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < kBK / kUmmaK; ++k) {
                            if constexpr (kPair)
                                umma_bf16_pair(d_tmem, desc(a_lo + k * (kUmmaK * 2 >> 4)), desc(b_lo + k * (kUmmaK * 2 >> 4)),
                                               idesc, (kb | k) != 0 ? 1u : 0u);
                            else
                                umma_bf16(d_tmem, desc(a_lo + k * (kUmmaK * 2 >> 4)), desc(b_lo + k * (kUmmaK * 2 >> 4)),
                                          idesc, (kb | k) != 0 ? 1u : 0u);
                        }
                        // frees the smem slot (in both CTAs of a pair) when the MMAs retire
                        if constexpr (kPair) umma_commit_pair(&empty[stage], 0b11);
                        else umma_commit(&empty[stage]);
                    }
                    __syncwarp();
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
                if (elect_one()) {                                // accumulator complete -> epilogue(s)
                    if constexpr (kPair) umma_commit_pair(&tmem_full[acc], 0b11);
                    else umma_commit(&tmem_full[acc]);
                }
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if (prof && lane == 0) {
                prof[blockIdx.x * 8 + 0] = clock64() - t0; prof[blockIdx.x * 8 + 1] = t_full; prof[blockIdx.x * 8 + 2] = t_te;
            }
        }
    } else if (warp >= kEpiWarp0) {
        // ------------------------------------------------------------ epilogue
        const int ewarp = warp - kEpiWarp0;
        const int quarter = warp & 3;
        Sched sched(sp, blockIdx.x, gridDim.x);
        int acc = 0;
        uint32_t acc_phase = 0;
        Epi epi;
        epi.begin(ep, sched, ewarp, lane, epi_smem);
        long long* prof = g_tc_prof;
        long long t0 = clock64(), t_tf = 0, tq;
#ifdef OFX_DEBUG
        long long tl_start = t0, tl_busy = 0, tl_wait0 = 0;    // per-unit timeline of CTA 0 (search schedules only)
        int tl_n = 0;
#endif
        while (sched.next()) {
#ifdef OFX_DEBUG
            if constexpr (Sched::kPrefetch) {
                if (prof && blockIdx.x == 0 && ewarp == 0 && lane == 0 && sched.first && sched.it == 0) {
                    const long long now = clock64();
                    if (tl_n > 0 && tl_n <= 40) {
                        prof[1200 + 3 * (tl_n - 1)] = now - tl_start;
                        prof[1200 + 3 * (tl_n - 1) + 1] = tl_busy;
                        prof[1200 + 3 * (tl_n - 1) + 2] = t_tf - tl_wait0;
                    }
                    tl_start = now; tl_busy = 0; tl_wait0 = t_tf; ++tl_n;
                }
            }
            const long long tl_t = clock64();
#endif
            epi.pre_tile(ep, sched, ewarp, lane, epi_smem);   // e.g. start fetching the residual tile
            if (prof) { tq = clock64(); mbar_wait(&tmem_full[acc], acc_phase); t_tf += clock64() - tq; }
            else mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_acc = tmem_base + acc * BN + (static_cast<uint32_t>(quarter * 32) << 16);
            epi.tile(ep, sched, t_acc, ewarp, lane, epi_smem);
#ifdef OFX_DEBUG
            tl_busy += clock64() - tl_t;
#endif
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (kPair) mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty[acc]), 0));
                else mbar_arrive(&tmem_empty[acc]);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        epi.end(ep, lane);
#ifdef OFX_DEBUG
        if constexpr (Sched::kPrefetch) {
            if (prof && blockIdx.x == 0 && ewarp == 0 && lane == 0 && tl_n > 0 && tl_n <= 40) {
                prof[1200 + 3 * (tl_n - 1)] = clock64() - tl_start;
                prof[1200 + 3 * (tl_n - 1) + 1] = tl_busy;
                prof[1200 + 3 * (tl_n - 1) + 2] = t_tf - tl_wait0;
                prof[1199] = tl_n;
            }
        }
#endif
        if (prof && ewarp == 0 && lane == 0) {
            prof[blockIdx.x * 8 + 4] = clock64() - t0; prof[blockIdx.x * 8 + 5] = t_tf;
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();  // no CTA leaves while a peer may still signal its barriers
    if (warp == 2) {
        tc_fence_after();
        if constexpr (kPair) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
        else tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
}

}  // namespace ofx
