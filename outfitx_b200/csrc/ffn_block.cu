// Fused feed-forward block of one encoder layer (d_model 512), one kernel:
//
//     x  <-  x + W2 . mish(W1 . LN2(x) + b1) + b2            (rows of the token matrix, in place)
//
// i.e. torch.nn.TransformerEncoderLayer's `x = x + _ff_block(norm2(x))` (pre-LN slow path,
// torch/nn/modules/transformer.py:950,980-982) as the reference builds it at
// /root/reference/src/models/outfit_x.py:32-45 (activation = F.mish, d_ffn 2024 zero-padded to 2048).
// The 2048-wide hidden activation never leaves the SM: it goes TMEM -> registers (bias + mish)
// -> shared memory (bf16 or fp16, the operand type; UMMA operand layout) -> second GEMM.  HBM traffic per token is one
// fp32 row in and one out (4 KB) instead of the 16 KB of LN + two separate GEMMs.
//
// Work decomposition: a CTA PAIR (cluster of 2, tcgen05 cta_group::2) owns 128 consecutive
// token rows, 64 per CTA.  With M = 128 across the pair an accumulator of 64 rows x N columns
// occupies 128 TMEM lanes x N/2 columns per CTA, so the full-width output (64 x 512 fp32 =
// 256 columns) and two 64 x 256 hidden-chunk accumulators (2 x 128 columns) fit the 512 TMEM
// columns together -- with cta_group::1 (128 rows per CTA) the output tile alone fills TMEM.
// Weight tiles are split across the pair (each CTA loads half of the N rows of every B tile),
// so every weight byte crosses L2 -> SM once per 128 token rows.
//
// Per tile the hidden dimension is swept in chunks of 256 units:
//   G1(c): acc1[c&1] = H . W1[c]^T          8 k-blocks of 64, N = 256
//   E (c): U[c&1] = bf16(mish(acc1 + b1))   epilogue warps, TMEM -> smem
//   G2(c): acc2 += U[c&1] . W2[:, c]^T      4 k-blocks of 64, 2 x (N = 256)
// issued as G1(0) G1(1) | G1(2) G2(0) | G1(3) G2(1) | ... : as soon as E(c) has drained acc1[c&1]
// the NEXT-BUT-ONE first GEMM goes in front of G2(c), so the epilogue of a chunk has three GEMM
// phases (~10k cycles) to finish instead of two, and H is released three phases before the tile
// ends (the LayerNorm prologue of the next tile needs that time).  Because G2(c) is now issued
// after G1(c+2), "acc1[c&1] is full again" no longer implies "G2(c) has read U[c&1]": E(c+2)
// waits for an explicit u_free[c&1] commit before it overwrites U.
//
// Warp roles (16 warps): 0 TMA producer (weights), 1 MMA issuer (leader CTA only), 2 TMEM
// allocator, 4-11 epilogue (mish chunks, then the residual epilogue), 12-15 LayerNorm warps: the
// prologue (x rows -> H in the swizzled K-major operand layout) and, when h_next is given, norm1 of
// the NEXT encoder layer on the rows the residual epilogue has just written (x_done barrier), so
// that no LayerNorm kernel runs between two layers.  Registers are re-partitioned with setmaxnreg:
// warps 0-3 give 48 per thread back, the epilogue warpgroups run with 152.
//
// What bounds it (measured, see DESIGN.md section 4): shared-memory bandwidth.  An M=128 pair MMA
// reads 96 B/clk of operands while TMA refills the weight ring at 64 B/clk; every byte the
// epilogues move through shared memory on top of that is paid for by the tensor pipe.
#include <cuda.h>
#include <stdlib.h>

#include "encoder_ops.h"
#include "ptx.cuh"

namespace ofx {
namespace ffnb {

constexpr int DM = 512;               // d_model (K of GEMM 1, N of GEMM 2)
constexpr int KB1 = DM / 64;          // k-blocks of GEMM 1
constexpr int CH = 256;               // hidden units per chunk (N of GEMM 1)
constexpr int KB2 = CH / 64;          // k-blocks of GEMM 2 per chunk
constexpr int ROWS = 64;              // token rows per CTA
constexpr int TILE = 2 * ROWS;        // token rows per CTA pair
constexpr int KBLK_BYTES = ROWS * 128;        // one 64-row x 64-element bf16 operand block
constexpr int H_BYTES = KB1 * KBLK_BYTES;     // 64 KB
constexpr int U_BYTES = KB2 * KBLK_BYTES;     // 32 KB
constexpr int SUB_BYTES = 128 * 128;          // one weight sub-tile: 128 rows x 64 K per CTA
constexpr int STAGE_BYTES = 2 * SUB_BYTES;    // ring stage = two sub-tiles = 8 MMAs per barrier wait
constexpr int NSTAGE = 3;
constexpr int BAR_BYTES = 512;
constexpr int SMEM_BYTES = 1024 + H_BYTES + 2 * U_BYTES + NSTAGE * STAGE_BYTES + BAR_BYTES;
constexpr int NTHREADS = 512;
constexpr int EPI_WARP0 = 4, N_EPI_WARPS = 8, LN_WARP0 = 12, N_LN_WARPS = 4;
constexpr uint32_t TM_ACC1 = 0, TM_ACC2 = 256;  // TMEM columns

struct Params {
    float* x;               // (rows, 512) fp32 residual stream, updated in place
    int rows;               // host-side row count (upper bound when rows_dev != nullptr)
    const int* rows_dev;    // optional device-side row count
    const float* ln_w;      // LayerNorm 2
    const float* ln_b;
    const float* b1;        // (n_chunks * 256) fp32, zero beyond d_ffn
    const float* b2;        // (512)
    int n_chunks;           // padded d_ffn / 256
    void* h_next;           // optional (rows, 512) 16-bit (the operand type): LayerNorm 1 of the NEXT layer applied to the new x
    const float* lnn_w;     // its affine terms
    const float* lnn_b;
    int debug;              // OFX_FFN_DEBUG bit mask, timing experiments only (results are WRONG with 1 / 256 / 512):
                            // 1 skip mish, 8 dump cycle counters, 256 skip the residual loads, 512 skip the x stores
    long long* prof;        // debug bit 3: per-pair cycle counters (16 per pair: MMA-warp waits; with
                            // -DOFX_FFN_EPROF also the phases of epilogue warp 0)
};

__device__ __forceinline__ float mish_fast(float x) {
    // x * n / (n + 2), n = w (w + 2), w = e^x   (see gemm.cu)
    float w, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(w) : "f"(fminf(x, 40.f) * 1.4426950408889634f));
    const float n = fmaf(w, w, w + w);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(n + 2.f));
    return x * n * r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// T: the 16-bit operand type (__nv_bfloat16 or __half) of H, U, the weights and h_next
template <class T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
ffn_block_kernel(const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_w2,
                 const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* s_h = smem;
    uint8_t* s_u = smem + H_BYTES;                       // U[0], U[1]
    uint8_t* s_w = smem + H_BYTES + 2 * U_BYTES;         // weight ring
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_w + NSTAGE * STAGE_BYTES);
    uint64_t* w_full = bars;                    // [NSTAGE]  leader's are used (tx from both CTAs)
    uint64_t* w_empty = bars + NSTAGE;          // [NSTAGE]  per CTA (multicast commit)
    uint64_t* acc1_full = bars + 2 * NSTAGE;    // [2]       per CTA (multicast commit)
    uint64_t* u_full = acc1_full + 2;           // [2]       leader's: 16 epilogue-warp arrivals
    uint64_t* u_free = u_full + 2;              // [2]       per CTA (multicast commit): G2 has read U[b]
    uint64_t* acc2_full = u_free + 2;           //           per CTA (multicast commit)
    uint64_t* acc2_empty = acc2_full + 1;       //           leader's: 16 arrivals
    uint64_t* h_full = acc2_empty + 1;          //           leader's: 8 LN-warp arrivals
    uint64_t* h_empty = h_full + 1;             //           per CTA (multicast commit)
    uint64_t* x_done = h_empty + 1;             //           per CTA: 8 epilogue-warp arrivals, new x rows are in global memory
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x_done + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();          // 0 = leader
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const int n_rows = p.rows_dev ? min(*p.rows_dev, p.rows) : p.rows;
    const int n_tiles = (n_rows + TILE - 1) / TILE;
    const int nch = p.n_chunks;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_w1);
        tma_prefetch_desc(&tm_w2);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < NSTAGE; ++i) {
            mbar_init(&w_full[i], 1);
            mbar_init(&w_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&acc1_full[i], 1);
            mbar_init(&u_full[i], 2 * N_EPI_WARPS);
            mbar_init(&u_free[i], 1);
        }
        mbar_init(acc2_full, 1);
        mbar_init(acc2_empty, 2 * N_EPI_WARPS);
        mbar_init(h_full, 2 * N_LN_WARPS);
        mbar_init(h_empty, 1);
        mbar_init(x_done, N_EPI_WARPS);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // Register re-partitioning (setmaxnreg, per warpgroup of 4 warps): the producer / MMA / allocator
    // warpgroup hands 48 registers per thread back, the two epilogue warpgroups take 24 more each (bias
    // vectors + a TMEM slab + the prefetched residual rows do not fit 128 without spilling into the mish loop).
    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;" ::: "memory");
    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (weights)
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const int r128 = static_cast<int>(rank) * 128;
            // one ring stage = two 128-row x 64-K sub-tiles
            auto put2 = [&](const CUtensorMap* tm, int i0, int o0, int i1, int o1) {
                mbar_wait(&w_empty[stage], phase ^ 1);
                if (rank == 0) mbar_arrive_expect_tx(&w_full[stage], 2 * STAGE_BYTES);   // both CTAs' bytes
                const uint32_t bar = mapa_shared(smem_u32(&w_full[stage]), 0);
                tma_load_2d_pair(s_w + stage * STAGE_BYTES, tm, bar, i0, o0, kEvictLast);
                tma_load_2d_pair(s_w + stage * STAGE_BYTES + SUB_BYTES, tm, bar, i1, o1, kEvictLast);
                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
            };
            auto g1 = [&](int c) {   // W1 rows of chunk c, k-blocks (2j, 2j+1)
                for (int j = 0; j < KB1 / 2; ++j)
                    put2(&tm_w1, (2 * j) * 64, c * CH + r128, (2 * j + 1) * 64, c * CH + r128);
            };
            auto g2 = [&](int c) {   // W2 columns of chunk c, k-block kb, output halves 0 / 1
                for (int kb = 0; kb < KB2; ++kb)
                    put2(&tm_w2, c * CH + kb * 64, r128, c * CH + kb * 64, 256 + r128);
            };
            for (int t = pair; t < n_tiles; t += n_pairs) {
                g1(0);
                if (nch > 1) g1(1);
                for (int c = 0; c < nch; ++c) {
                    if (c + 2 < nch) g1(c + 2);
                    g2(c);
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (leader only)
        // The whole warp runs the loop (warp-uniform control flow and addresses, so the
        // descriptors live in uniform registers); one elected lane issues the tcgen05 ops.
        // Measured: a UTCHMMA blocks its issuer until the tensor pipe accepts it (the queue is
        // about one deep), and an M=128 / N=256 pair MMA runs for only 64 cycles, so whatever the
        // issuing thread does between MMAs is tensor-pipe idle time.  Hence 8 MMAs per ring
        // stage, and the mbarrier poll for the NEXT stage is issued before this stage's MMAs so
        // that its ~100-cycle latency overlaps them.
        if (rank == 0) {
            constexpr uint32_t idesc = umma_idesc_16<T>(128, 256);
            constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO, version, SW128
            const uint32_t h_lo = ((smem_u32(s_h) & 0x3FFFF) >> 4) | (1u << 16);
            const uint32_t u_lo = ((smem_u32(s_u) & 0x3FFFF) >> 4) | (1u << 16);
            const uint32_t w_lo = ((smem_u32(s_w) & 0x3FFFF) >> 4) | (1u << 16);
            auto desc = [](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
            int stage = 0;
            uint32_t phase = 0, tphase = 0, uph0 = 0, uph1 = 0;
            uint32_t ready = 0;     // result of the early poll of w_full[stage]
            long long t_w = 0, t_u = 0, t_h = 0, t_a2 = 0, t0 = clock64(), tq;
            long long t_uc[3] = {0, 0, 0};     // u_full wait of chunk 0, chunk 1, last chunk
#define PROF_WAIT(acc, stmt) do { if (p.prof) { tq = clock64(); stmt; acc += clock64() - tq; } else { stmt; } } while (0)
            // waits for ring stage `stage`, polls the next one, returns this stage's B descriptor base
            auto acquire = [&](int& ns, uint32_t& nph, uint32_t& nready) -> uint32_t {
                if (!ready) PROF_WAIT(t_w, mbar_wait(&w_full[stage], phase));
                tc_fence_after();
                ns = stage + 1; nph = phase;
                if (ns == NSTAGE) { ns = 0; nph ^= 1; }
                nready = mbar_try_wait(&w_full[ns], nph) ? 1u : 0u;
                return w_lo + stage * (STAGE_BYTES >> 4);
            };
            auto g1 = [&](int c) {
                const uint32_t d = tmem_base + TM_ACC1 + (c & 1) * 128;
                for (int j = 0; j < KB1 / 2; ++j) {
                    int ns; uint32_t nph, nready;
                    const uint32_t b = acquire(ns, nph, nready);
                    const uint32_t a = h_lo + (2 * j) * (KBLK_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int sub = 0; sub < 2; ++sub)
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma_bf16_pair(d, desc(a + sub * (KBLK_BYTES >> 4) + 2 * k),
                                               desc(b + sub * (SUB_BYTES >> 4) + 2 * k), idesc,
                                               (j | sub | k) != 0 ? 1u : 0u);
                        umma_commit_pair(&w_empty[stage], 0b11);
                    }
                    __syncwarp();
                    stage = ns; phase = nph; ready = nready;
                }
                if (elect_one()) {
                    umma_commit_pair(&acc1_full[c & 1], 0b11);
                    if (c == nch - 1) umma_commit_pair(h_empty, 0b11);   // H may be refilled
                }
                __syncwarp();
            };
            auto wait_u = [&](int c) {     // E(c) done: U[c&1] is ready and acc1[c&1] has been drained
                const long long before = t_u;
                if (c & 1) { PROF_WAIT(t_u, mbar_wait(&u_full[1], uph1)); uph1 ^= 1; }
                else       { PROF_WAIT(t_u, mbar_wait(&u_full[0], uph0)); uph0 ^= 1; }
                if (p.prof) {
                    if (c == 0) t_uc[0] += t_u - before;
                    else if (c == 1) t_uc[1] += t_u - before;
                    else if (c == nch - 1) t_uc[2] += t_u - before;
                }
                tc_fence_after();
            };
            auto g2 = [&](int c) {
                const uint32_t ub = u_lo + (c & 1) * (U_BYTES >> 4);
                for (int kb = 0; kb < KB2; ++kb) {
                    int ns; uint32_t nph, nready;
                    const uint32_t b = acquire(ns, nph, nready);
                    const uint32_t a = ub + kb * (KBLK_BYTES >> 4);
                    if (elect_one()) {
#pragma unroll
                        for (int half = 0; half < 2; ++half)
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma_bf16_pair(tmem_base + TM_ACC2 + half * 128, desc(a + 2 * k),
                                               desc(b + half * (SUB_BYTES >> 4) + 2 * k), idesc,
                                               (c | kb | k) != 0 ? 1u : 0u);
                        umma_commit_pair(&w_empty[stage], 0b11);
                    }
                    __syncwarp();
                    stage = ns; phase = nph; ready = nready;
                }
                if (elect_one()) umma_commit_pair(&u_free[c & 1], 0b11);   // U[c&1] may be overwritten once these retire
                __syncwarp();
            };
            for (int t = pair; t < n_tiles; t += n_pairs) {
                PROF_WAIT(t_h, mbar_wait(h_full, tphase));
                tc_fence_after();
                g1(0);
                if (nch > 1) g1(1);
                for (int c = 0; c < nch; ++c) {
                    wait_u(c);
                    if (c + 2 < nch) g1(c + 2);
                    if (c == 0) {   // the previous tile's output has left TMEM
                        PROF_WAIT(t_a2, mbar_wait(acc2_empty, tphase ^ 1));
                        tc_fence_after();
                    }
                    g2(c);
                }
                if (elect_one()) umma_commit_pair(acc2_full, 0b11);
                __syncwarp();
                tphase ^= 1;
            }
            if (p.prof && lane == 0) {
                long long* o = p.prof + pair * 16;
                o[0] = clock64() - t0; o[1] = t_w; o[2] = t_u; o[3] = t_h; o[4] = t_a2;
                o[5] = t_uc[0]; o[6] = t_uc[1]; o[7] = t_uc[2];
            }
#undef PROF_WAIT
        }
    }
    } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + N_EPI_WARPS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 152;" ::: "memory");
        // ------------------------------------------------------------ epilogue warps
        const int q = warp & 3;                       // TMEM lane quarter
        const int ch = (warp - EPI_WARP0) >> 2;       // which 64 of the accumulator's 128 columns
        const int row_l = (q & 1) * 32 + lane;        // token row within this CTA's 64
        const int nhalf = q >> 1;                     // N half held by lanes 64..127
        const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
        const int kblk = nhalf * 2 + ch;              // k-block of U this thread's 64 values form
        const uint32_t u_row = kblk * KBLK_BYTES + (row_l >> 3) * 1024 + (row_l & 7) * 128;
        const int sw = row_l & 7;
        const uint32_t ufull0 = mapa_shared(smem_u32(&u_full[0]), 0);
        const uint32_t ufull1 = mapa_shared(smem_u32(&u_full[1]), 0);
        const uint32_t a2empty = mapa_shared(smem_u32(acc2_empty), 0);
        // staging for the residual epilogue: this warp's own 32-row x 128-byte block of U[1] (free from
        // acc2_full until these warps themselves run chunk 1 of the next tile; U[0] is NOT free: chunk 0
        // of the next tile is worked in between the residual slabs, see below)
        uint8_t* stg = s_u + U_BYTES + kblk * KBLK_BYTES + (q & 1) * 4096;
        const int sub_row = lane >> 3, chunk = lane & 7;
        // barrier parities as bit masks (indexable arrays would live in local memory): bit b = buffer b
        uint32_t a1ph = 0, ufph = 3, tphase = 0;
        // debug bit 3: where epilogue warp 0 of the leader spends its cycles
        // (compile with -DOFX_FFN_EPROF: the seven 64-bit counters cost registers the mish loop needs)
#ifdef OFX_FFN_EPROF
        const bool eprof = p.prof && rank == 0 && warp == EPI_WARP0;
        long long e_wa1 = 0, e_wuf = 0, e_mish = 0, e_wa2 = 0, e_res = 0, e_mish0 = 0, eq = 0;
        long long r_tmem = 0, r_stage = 0, r_add = 0, r_store = 0;
#define EPROF_BEGIN() do { if (eprof) eq = clock64(); } while (0)
#define EPROF_END(acc) do { if (eprof) { const long long now = clock64(); acc += now - eq; eq = now; } } while (0)
#else
#define EPROF_BEGIN() do { } while (0)
#define EPROF_END(acc) do { } while (0)
#endif
        // E(c): U[c&1] = bf16(mish(acc1[c&1] + b1)) for this warp's 32 rows x 64 hidden units
        auto mish_chunk = [&](int c) {
            const int b = c & 1;
            EPROF_BEGIN();
            // bias of this thread's 64 hidden units (warp-uniform addresses).  With ~224 KB of
            // shared memory there is next to no L1, so these are L2 round trips: slab 0's are
            // issued before the barrier wait, slab 1's while slab 0 is being computed.
            const float4* bias4 = reinterpret_cast<const float4*>(p.b1 + c * CH + nhalf * 128 + ch * 64);
            float4 bv0[8], bv1[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) bv0[i] = __ldg(bias4 + i);
            mbar_wait(&acc1_full[b], (a1ph >> b) & 1);
            a1ph ^= 1u << b;
            tc_fence_after();
            EPROF_END(e_wa1);
            uint8_t* dst = s_u + b * U_BYTES + u_row;
            auto slab = [&](int s, const float4 (&bv)[8], const uint32_t (&raw)[32]) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t w[4];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const float4 bb = bv[2 * j + h];
                        float v0 = __uint_as_float(raw[8 * j + 4 * h + 0]) + bb.x;
                        float v1 = __uint_as_float(raw[8 * j + 4 * h + 1]) + bb.y;
                        float v2 = __uint_as_float(raw[8 * j + 4 * h + 2]) + bb.z;
                        float v3 = __uint_as_float(raw[8 * j + 4 * h + 3]) + bb.w;
                        if (!(p.debug & 1)) { v0 = mish_fast(v0); v1 = mish_fast(v1); v2 = mish_fast(v2); v3 = mish_fast(v3); }
                        w[2 * h] = pack2_16<T>(v0, v1);
                        w[2 * h + 1] = pack2_16<T>(v2, v3);
                    }
                    *reinterpret_cast<uint4*>(dst + (((s * 4 + j) ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
                }
            };
            uint32_t raw[32];
            tmem_ld_32x32(t_lane + TM_ACC1 + b * 128 + ch * 64, raw);
#pragma unroll
            for (int i = 0; i < 8; ++i) bv1[i] = __ldg(bias4 + 8 + i);
            tmem_ld_wait();
            // the previous use of U[b] (two chunks ago) must have been read by its G2; the very
            // first wait on each buffer passes (fresh barrier, parity 1)
            EPROF_END(e_mish);
            mbar_wait(&u_free[b], (ufph >> b) & 1);
            ufph ^= 1u << b;
            EPROF_END(e_wuf);
            slab(0, bv0, raw);
            tmem_ld_32x32(t_lane + TM_ACC1 + b * 128 + ch * 64 + 32, raw);
            tmem_ld_wait();
            slab(1, bv1, raw);
            fence_proxy_async();     // generic-proxy smem writes -> visible to the UMMA (async proxy)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(b ? ufull1 : ufull0);
#ifdef OFX_FFN_EPROF
            if (eprof) { const long long now = clock64(); e_mish += now - eq; if (c == 0) e_mish0 += now - eq; }
#endif
        };
        for (int t = pair; t < n_tiles; t += n_pairs) {
#pragma unroll 1
            for (int c = 0; c < nch; ++c) mish_chunk(c);
            // ---- residual epilogue: x <- x + acc2 + b2 for this warp's 32 rows x 128 columns, in 4 slabs of
            // 32 columns (TMEM -> registers -> swizzled staging block -> row-major, coalesced).  It sits between
            // the last GEMM of this tile and the first mish chunk of the next one, whose first GEMMs are already
            // running.  Measured (OFX_FFN_DEBUG=8, -DOFX_FFN_EPROF): ~10k cycles per tile, and it stays ~10k
            // whether the rows travel as per-thread LDG / STG, as TMA bulk stores, or by TMA in both directions
            // with the add done in place in the staging block -- every variant was built and timed within 1 %.
            // The common factor is shared-memory bandwidth: GEMM 1 of the next tile reads operands at 96 B/clk
            // while TMA refills the weight ring at 64 B/clk, which is more than the 128 B/clk the SM has, so
            // whatever the epilogue moves through shared memory is paid for by the tensor pipe one for one.  The
            // cheapest form therefore wins: one staging round trip (256 KB per CTA and tile), residual rows
            // prefetched one slab ahead in registers.
            const long long row0 = static_cast<long long>(t) * TILE + rank * ROWS + (q & 1) * 32;
            auto slab_c0 = [&](int sl) { return (sl >> 1) * 256 + nhalf * 128 + ch * 64 + (sl & 1) * 32; };
            const int rows_valid = n_rows - static_cast<int>(row0) - sub_row;   // row 4i+sub_row live iff 4i < rows_valid
            auto slab_col = [&](int sl) { return slab_c0(sl) + chunk * 4; };
            float4 res[8], b4;
            auto load_res = [&](int sl) {     // residual rows and output bias of slab sl
                const float* xp = p.x + (row0 + sub_row) * DM + slab_col(sl);
                b4 = __ldg(reinterpret_cast<const float4*>(p.b2 + slab_col(sl)));
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    res[i] = (4 * i < rows_valid && !(p.debug & 256)) ? ldg128(xp + static_cast<long long>(4 * i) * DM)
                                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            };
            load_res(0);
            EPROF_BEGIN();
            mbar_wait(acc2_full, tphase);
            tphase ^= 1;
            tc_fence_after();
            EPROF_END(e_wa2);
#pragma unroll 1
            for (int sl = 0; sl < 4; ++sl) {
                float* xp = p.x + (row0 + sub_row) * DM + slab_col(sl);
                uint32_t raw[32];
                tmem_ld_32x32(t_lane + TM_ACC2 + (sl >> 1) * 128 + ch * 64 + (sl & 1) * 32, raw);
                tmem_ld_wait();
                EPROF_END(r_tmem);
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    *reinterpret_cast<uint4*>(stg + lane * 128 + ((i ^ (lane & 7)) << 4)) =
                        make_uint4(raw[4 * i], raw[4 * i + 1], raw[4 * i + 2], raw[4 * i + 3]);
                __syncwarp();
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + sub_row;
                    v[i] = *reinterpret_cast<const float4*>(stg + r * 128 + ((chunk ^ (r & 7)) << 4));
                    v[i].x += b4.x + res[i].x; v[i].y += b4.y + res[i].y;
                    v[i].z += b4.z + res[i].z; v[i].w += b4.w + res[i].w;
                }
                EPROF_END(r_add);
                if (sl < 3) load_res(sl + 1);
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (4 * i < rows_valid && !(p.debug & 512)) stg128(xp + static_cast<long long>(4 * i) * DM, v[i]);
                EPROF_END(r_store);
            }
            EPROF_END(e_res);
            tc_fence_before();
            // x_done: the LayerNorm warps may re-read the new rows.  Every lane fences its global stores at CTA
            // scope before the warp converges; lane 0's mbarrier.arrive (release) then publishes them and the
            // LayerNorm warps acquire through mbarrier.try_wait.  (Measured: the fence costs nothing here.)
            if (p.h_next) __threadfence_block();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive_cluster(a2empty);
                if (p.h_next) mbar_arrive(x_done);
            }
        }
#ifdef OFX_FFN_EPROF
        if (eprof && lane == 0) {
            long long* o = p.prof + pair * 16 + 8;
            o[0] = r_tmem; o[1] = r_stage; o[2] = e_mish; o[3] = e_wa2; o[4] = e_res; o[5] = e_mish0; o[6] = r_add; o[7] = r_store;
        }
#endif
#undef EPROF_BEGIN
#undef EPROF_END
    } else if (warp >= LN_WARP0) {
        // ------------------------------------------------------------ LayerNorm warps
        // (1) prologue: LN2 of this tile's x rows -> H (16-bit, swizzled K-major operand layout);
        // (2) in the idle time that follows, LN1 of the NEXT layer on the PREVIOUS tile's freshly
        //     written x rows -> h_next (16-bit, row-major), re-read from L2: the separate LayerNorm
        //     kernel between two layers (one more read of x from HBM) disappears.
        const int lw = warp - LN_WARP0;
        const uint32_t hfull = mapa_shared(smem_u32(h_full), 0);
        uint32_t tphase = 0, xphase = 0;
        // two-pass LayerNorm of 4 rows held in registers (lane owns columns i*128 + lane*4 .. +3)
        // gamma / beta are fetched ONCE per tile, before the barrier wait that precedes the rows: with
        // ~224 KB of shared memory there is next to no L1, so loading them inside the row loop put an
        // extra L2 round trip behind every batch of rows.
        auto load_affine = [&](const float* gw, const float* gb, float4 (&g)[4], float4 (&be)[4]) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                g[i] = __ldg(reinterpret_cast<const float4*>(gw + i * 128 + lane * 4));
                be[i] = __ldg(reinterpret_cast<const float4*>(gb + i * 128 + lane * 4));
            }
        };
        auto norm4 = [&](float4 (&v)[4][4], const float4 (&gam)[4], const float4 (&bet)[4], auto&& emit) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i) s += v[u][i].x + v[u][i].y + v[u][i].z + v[u][i].w;
                const float mu = warp_sum(s) * (1.f / DM);
                float qq = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float a = v[u][i].x - mu, b = v[u][i].y - mu, c = v[u][i].z - mu, d = v[u][i].w - mu;
                    qq += a * a + b * b + c * c + d * d;
                }
                const float rstd = rsqrtf(warp_sum(qq) * (1.f / DM) + 1e-5f);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 g = gam[i], be = bet[i];
                    emit(u, i, (v[u][i].x - mu) * rstd * g.x + be.x, (v[u][i].y - mu) * rstd * g.y + be.y,
                         (v[u][i].z - mu) * rstd * g.z + be.z, (v[u][i].w - mu) * rstd * g.w + be.w);
                }
            }
        };
        auto ln_next = [&](int t) {      // LN1(next layer) of tile t's new rows -> h_next
            float4 gam[4], bet[4];
            load_affine(p.lnn_w, p.lnn_b, gam, bet);
            mbar_wait(x_done, xphase);   // this CTA's epilogue warps have stored them
            xphase ^= 1;
            const long long row0 = static_cast<long long>(t) * TILE + rank * ROWS + lw * 16;
#pragma unroll 1
            for (int rb = 0; rb < 16; rb += 4) {
                if (row0 + rb >= n_rows) break;
                float4 v[4][4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const long long row = row0 + rb + u;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        v[u][i] = row < n_rows ? ldg128(p.x + row * DM + i * 128 + lane * 4)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                norm4(v, gam, bet, [&](int u, int i, float y0, float y1, float y2, float y3) {
                    const long long row = row0 + rb + u;
                    if (row < n_rows)
                        *reinterpret_cast<uint2*>(static_cast<T*>(p.h_next) + row * DM + i * 128 + lane * 4) =
                            make_uint2(pack2_16<T>(y0, y1), pack2_16<T>(y2, y3));
                });
            }
        };
        // (A "staged" variant was built and measured: LN2 rows computed one tile ahead, parked as bf16 in the
        // tile's unused h_next rows and moved into H by TMA as soon as GEMM 1 released it.  It halves the
        // h_full wait, the kernel alone gets 2.5 % faster, the CP pass 1 % slower -- the stall moves to the
        // first mish chunk, see the residual epilogue -- so the simpler direct form stayed.)
        int prev = -1;
        for (int t = pair; t < n_tiles; t += n_pairs) {
            const long long row0 = static_cast<long long>(t) * TILE + rank * ROWS + lw * 16;
            // pull this warp's 16 rows (32 KB) towards L2 while the previous tile still owns H
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const long long off = (row0 * DM + (i * 32 + lane) * 32) ;   // 128-byte lines
                if (row0 + (i * 32 + lane) / 16 < n_rows)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(p.x + off));
            }
            float4 gam[4], bet[4];
            load_affine(p.ln_w, p.ln_b, gam, bet);
            float4 v[4][4];
            auto load4 = [&](int rb) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const long long row = row0 + rb + u;
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        v[u][i] = row < n_rows ? ldg128(p.x + row * DM + i * 128 + lane * 4)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            mbar_wait(h_empty, tphase ^ 1);     // GEMM 1 of the previous tile has consumed H
            tphase ^= 1;
#pragma unroll 1
            for (int rb = 0; rb < 16; rb += 4) {
                load4(rb);
                norm4(v, gam, bet, [&](int u, int i, float y0, float y1, float y2, float y3) {
                    const int r = lw * 16 + rb + u;      // row within this CTA's 64
                    if (row0 + rb + u >= n_rows) y0 = y1 = y2 = y3 = 0.f;
                    // element e = i*128 + lane*4: k-block e/64, 16-byte chunk (e%64)/8, 8-byte half
                    const int kb = i * 2 + (lane >> 4);
                    const int c16 = (lane & 15) >> 1;
                    uint8_t* dst = s_h + kb * KBLK_BYTES + (r >> 3) * 1024 + (r & 7) * 128 +
                                   ((c16 ^ (r & 7)) << 4) + (lane & 1) * 8;
                    *reinterpret_cast<uint2*>(dst) = make_uint2(pack2_16<T>(y0, y1), pack2_16<T>(y2, y3));
                });
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(hfull);
            if (p.h_next && prev >= 0) ln_next(prev);
            prev = t;
        }
        if (p.h_next && prev >= 0) ln_next(prev);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

}  // namespace ffnb

bool ffn_block_supported(int dm, int fp) { return dm == ffnb::DM && fp > 0 && fp % ffnb::CH == 0; }

// The kernel needs no scratch; the workspace the C ABI asks for (ofx_ffn_block_workspace_bytes) is a fixed 256 B.
size_t ffn_block_workspace_bytes() { return 256; }

template <class T>
static int ffn_block(const FfnBlockArgs& a, cudaStream_t stream) {
    using namespace ffnb;
    if (a.rows > 0 && ffn_block_supported(a.dm, a.fp) && (!a.workspace || a.workspace_bytes < ffn_block_workspace_bytes()))
        return fail(OFX_E_WORKSPACE, "ffn_block workspace %zu B < required %zu B", a.workspace_bytes, ffn_block_workspace_bytes());
    if (a.rows <= 0) return OFX_OK;
    if (a.dm != DM || a.fp <= 0 || a.fp % CH != 0)
        return fail(OFX_E_SHAPE, "ffn_block: needs d_model 512 and padded d_ffn %% 256 == 0 (got %d, %d)", a.dm, a.fp);
    CUtensorMap tm_w1, tm_w2;
    // OFX_FFN_DEBUG (timing experiments: bits 1 / 256 / 512 give WRONG results, bit 8 allocates and synchronises)
    // exists only in instrumented builds (-DOFX_DEBUG); the product library cannot be switched into either.
#ifdef OFX_DEBUG
    static int debug = -1;
    if (debug < 0) { const char* e = getenv("OFX_FFN_DEBUG"); debug = e ? atoi(e) : 0; }
#else
    constexpr int debug = 0;
#endif
    // the 2-byte tensor map moves fp16 weights unchanged (common.h)
    OFX_TRY(make_tmap_bf16(&tm_w1, a.w1, static_cast<uint64_t>(a.fp), DM, DM, 128));
    OFX_TRY(make_tmap_bf16(&tm_w2, a.w2, DM, static_cast<uint64_t>(a.fp), a.fp, 128));
    static DeviceOnce configured;
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(ffn_block_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    }
    const int n_tiles = (a.rows + TILE - 1) / TILE;
    const int max_pairs = sm_count() / 2;
    const int pairs = n_tiles < max_pairs ? n_tiles : max_pairs;
    if (a.h_next && (!a.lnn_w || !a.lnn_b)) return fail(OFX_E_ARG, "ffn_block: h_next needs the next layer's LayerNorm terms");
    Params p{a.x, a.rows, a.rows_dev, a.ln_w, a.ln_b, a.b1, a.b2, a.fp / CH, a.h_next, a.lnn_w, a.lnn_b, debug, nullptr};
    static long long* prof_dev = nullptr;
    if (debug & 8) {
        if (!prof_dev) OFX_CUDA(cudaMalloc(&prof_dev, 8 * 16 * 128));
        OFX_CUDA(cudaMemsetAsync(prof_dev, 0, 8 * 16 * 128, stream));
        p.prof = prof_dev;
    }
    ffn_block_kernel<T><<<pairs * 2, NTHREADS, SMEM_BYTES, stream>>>(tm_w1, tm_w2, p);
    OFX_LAUNCH_CHECK();
    if (debug & 8) {   // debug only: synchronous dump of the MMA warp's wait-cycle counters
        static int dumps = 0;
        long long h[16 * 128];
        OFX_CUDA(cudaStreamSynchronize(stream));
        OFX_CUDA(cudaMemcpy(h, prof_dev, sizeof(h), cudaMemcpyDeviceToHost));
        if (dumps++ < 2)
            for (int i = 0; i < pairs && i < 74; i += 18)
                fprintf(stderr, "ffn prof pair %d: total %lld  w_full %lld  u_full %lld (chunk 0: %lld, 1: %lld, last: %lld)  h_full %lld  acc2_empty %lld cycles\n",
                        i, h[i * 16], h[i * 16 + 1], h[i * 16 + 2], h[i * 16 + 5], h[i * 16 + 6], h[i * 16 + 7], h[i * 16 + 3], h[i * 16 + 4]),
                fprintf(stderr, "   epilogue warp (-DOFX_FFN_EPROF): mish %lld (chunk 0: %lld)  wait acc2_full %lld  residual: tmem %lld  stage %lld  add %lld  store %lld  tail %lld\n",
                        h[i * 16 + 10], h[i * 16 + 13], h[i * 16 + 11], h[i * 16 + 8], h[i * 16 + 9], h[i * 16 + 14], h[i * 16 + 15], h[i * 16 + 12]);
    }
    return OFX_OK;
}

int ffn_block_bf16(const FfnBlockArgs& a, cudaStream_t stream) { return ffn_block<__nv_bfloat16>(a, stream); }
int ffn_block_f16(const FfnBlockArgs& a, cudaStream_t stream) { return ffn_block<__half>(a, stream); }

}  // namespace ofx
