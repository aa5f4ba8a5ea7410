// Linear layers of the outfit encoder: C = A . W^T (+bias) (+mish) (+fp32 residual).
//   bf16 / fp16 mode: tcgen05 / TMEM / TMA pipeline (tc_pipeline.cuh) with the fused epilogue below
//   fp32 mode: the same pipeline on split-bf16 operands (gemm_f32_split, gemm.h)
// Replaces the cuBLAS calls behind torch.nn.functional.linear in the reference's
// nn.TransformerEncoderLayer (in_proj, out_proj, linear1+mish, linear2; SURVEY.md 2.1).
#include "gemm.h"

#include <stdlib.h>

#include "tc_pipeline.cuh"

namespace ofx {

// mish(x) = x * tanh(softplus(x)) = x * n / (n + 2),  n = e^x (e^x + 2)   (SURVEY.md H4);
// torch's softplus threshold (x > 20 -> x) is kept.
__device__ __forceinline__ float mish_fast(float x) {
    // n / (n + 2) with n = w (w + 2), w = e^x: two MUFU ops (ex2, rcp).  For x >= 20 the ratio
    // rounds to 1 (torch switches softplus to the identity there); the clamp keeps w^2 finite.
    float w, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(w) : "f"(fminf(x, 40.f) * 1.4426950408889634f));
    const float n = fmaf(w, w, w + w);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(n + 2.f));
    return x * n * r;
}

// -------------------------------------------------------------------------------------
// tcgen05 path
// -------------------------------------------------------------------------------------
struct SchedGemm {
    static constexpr bool kThrottle = false;
    __device__ void throttle() {}
    struct Params {
        int m;             // host-side row count (upper bound when m_dev != nullptr)
        const int* m_dev;  // optional device-side row count (token count after compaction)
        int n_tiles;       // N / BN
        int bn;
        int cl;            // cluster size: CL consecutive M tiles share one B (weight) tile
    };
    static constexpr bool kPrefetch = false;
    int m0, n0, m_actual, pf_n0;
    int tile, step, total, n_tiles, bn, cl, rank;
    __device__ SchedGemm(const Params& p, int cta, int n_cta) {
        m_actual = p.m_dev ? min(*p.m_dev, p.m) : p.m;
        n_tiles = p.n_tiles;
        bn = p.bn;
        cl = p.cl;
        rank = cta % cl;
        const int m_groups = ((m_actual + kBM - 1) / kBM + cl - 1) / cl;
        total = m_groups * n_tiles;
        step = n_cta / cl;
        tile = cta / cl - step;
        m0 = n0 = 0;
    }
    __device__ bool next() {
        tile += step;
        if (tile >= total) return false;
        // n fastest: clusters that run together share the same rows of A in L2.  A CTA whose
        // M tile lies beyond m_actual still runs the tile (TMA zero-fills, nothing is stored).
        m0 = ((tile / n_tiles) * cl + rank) * kBM;
        n0 = (tile % n_tiles) * bn;
        return true;
    }
};

// Epilogue of the linear layers.  8 warps: warp e serves accumulator rows 32*(e&3)..+31 and the
// column half (e>>2).  Per 32-column slab:
//   phase A  thread <-> row: tcgen05.ld gives each thread 32 consecutive fp32 columns of its row;
//            they go to a per-warp 32 x 128 B staging tile in shared memory (16-byte chunks
//            XOR-swizzled by row so both phases are bank-conflict free);
//   phase B  lane <-> (row % 4, 16-byte chunk): the warp re-reads the tile four rows at a time and
//            applies bias / mish / fp32 residual and stores -- every global access of the warp
//            is now 4 full 128-byte (fp32) or 64-byte (bf16) row segments instead of 32 scattered
//            16-byte pieces.
template <int BN>
struct EpiLinear {
    struct Params {
        const float* bias;
        const float* residual;
        long long ldr;
        void* out;
        long long ldo;
        int act_mish;
        int out_f32;
    };
    static constexpr int kWarps = 8;
    static constexpr int kSmemBytes = kWarps * 32 * 128;
    __device__ void begin(const Params&, const SchedGemm&, int, int, uint8_t*) {}
    __device__ void end(const Params&, int) {}
    __device__ void pre_tile(const Params&, const SchedGemm&, int, int, uint8_t*) {}
    __device__ void tile(const Params& p, const SchedGemm& s, uint32_t t_acc, int ewarp, int lane,
                         uint8_t* epi_smem) {
        const int quarter = ewarp & 3, half = ewarp >> 2;
        uint8_t* stage = epi_smem + ewarp * (32 * 128);
        const int sub_row = lane >> 3, chunk = lane & 7;
        const int row0 = s.m0 + quarter * 32;
        const int rows_valid = s.m_actual - row0 - sub_row;  // row 4 i + sub_row is live iff 4 i < rows_valid
        const int col0 = s.n0 + half * (BN / 2) + chunk * 4;
        const long long first = static_cast<long long>(row0 + sub_row);
        const float* resp = p.residual ? p.residual + first * p.ldr + col0 : nullptr;
        float* outf = static_cast<float*>(p.out) + first * p.ldo + col0;
        __nv_bfloat16* outh = static_cast<__nv_bfloat16*>(p.out) + first * p.ldo + col0;
        const long long ldr4 = 4 * p.ldr, ldo4 = 4 * p.ldo;
        constexpr int kSlabs = BN / 2 / 32;
        // the fp32 residual of a slab is fetched one slab ahead (before any store of this slab,
        // which may alias it), so its HBM latency hides behind the TMEM read and the staging
        float4 res[8];
        if (resp) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                res[i] = 4 * i < rows_valid ? *reinterpret_cast<const float4*>(resp + i * ldr4)
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int sl = 0; sl < kSlabs; ++sl) {
            const int c = half * (BN / 2) + sl * 32;
            uint32_t raw[32];
            tmem_ld_32x32(t_acc + c, raw);
            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + sl * 32));
            float4 nxt[8];
            if (resp && sl + 1 < kSlabs) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    nxt[i] = 4 * i < rows_valid
                                 ? *reinterpret_cast<const float4*>(resp + (sl + 1) * 32 + i * ldr4)
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            tmem_ld_wait();
            __syncwarp();  // previous slab's phase B has finished reading the staging tile
#pragma unroll
            for (int i = 0; i < 8; ++i)
                *reinterpret_cast<uint4*>(stage + lane * 128 + ((i ^ (lane & 7)) << 4)) =
                    make_uint4(raw[4 * i], raw[4 * i + 1], raw[4 * i + 2], raw[4 * i + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int r = 4 * i + sub_row;
                float4 v = *reinterpret_cast<const float4*>(stage + r * 128 + ((chunk ^ (r & 7)) << 4));
                if (4 * i < rows_valid) {
                    v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
                    if (p.act_mish) { v.x = mish_fast(v.x); v.y = mish_fast(v.y); v.z = mish_fast(v.z); v.w = mish_fast(v.w); }
                    if (resp) { v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w; }
                    if (p.out_f32 == 2) {
                        // fp32 mode: the result is the NEXT split GEMM's activation operand -- write its bf16 pieces
                        // [hi | lo | hi] (row pitch ldo = 3 N) instead of the fp32 value (gemm.h)
                        const float f[4] = {v.x, v.y, v.z, v.w};
                        __nv_bfloat16 hi[4], lo[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            hi[j] = __float2bfloat16_rn(f[j]);
                            lo[j] = __float2bfloat16_rn(f[j] - __bfloat162float(hi[j]));
                        }
                        __nv_bfloat16* o = outh + sl * 32 + i * ldo4;
                        const long long nn = p.ldo / 3;
                        const uint2 h2 = *reinterpret_cast<const uint2*>(hi), l2 = *reinterpret_cast<const uint2*>(lo);
                        *reinterpret_cast<uint2*>(o) = h2;
                        *reinterpret_cast<uint2*>(o + nn) = l2;
                        *reinterpret_cast<uint2*>(o + 2 * nn) = h2;
                    } else if (p.out_f32) {
                        *reinterpret_cast<float4*>(outf + sl * 32 + i * ldo4) = v;
                    } else {
                        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
                        uint2 u;
                        u.x = *reinterpret_cast<uint32_t*>(&lo);
                        u.y = *reinterpret_cast<uint32_t*>(&hi);
                        *reinterpret_cast<uint2*>(outh + sl * 32 + i * ldo4) = u;
                    }
                }
            }
            if (resp && sl + 1 < kSlabs) {
#pragma unroll
                for (int i = 0; i < 8; ++i) res[i] = nxt[i];
            }
        }
    }
};

// Epilogue of the 16-bit-output linear layers (QKV projection, linear1 + mish): TMEM -> registers
// (bias, mish, bf16 / fp16 pack: T is also the operand type) -> a per-warp 32-row x 128-byte staging
// tile in the 128B-swizzle layout
// -> ONE TMA store per 64 output columns.  No per-thread global addressing and no transposing
// read-back: ~2 instructions per output element instead of ~11, and a code footprint that fits
// the instruction cache (the unrolled version stalled on instruction fetch).  Rows beyond the
// tensor map's row count are clipped by the TMA unit; rows between the device-side row count
// and the host bound land in caller scratch that nobody reads.
struct alignas(64) EpiStoreParams {
    CUtensorMap tm_c;      // (M, N) 16-bit output, box = 64 columns x 32 rows, 128B swizzle
    const float* bias;
    int act_mish;
};
template <int BN, class T>
struct EpiStore16 {
    using Operand = T;
    using Params = EpiStoreParams;
    static constexpr int kWarps = 8;
    static constexpr int kSmemBytes = kWarps * 32 * 128;
    __device__ void begin(const Params&, const SchedGemm&, int, int, uint8_t*) {}
    __device__ void pre_tile(const Params&, const SchedGemm&, int, int, uint8_t*) {}
    __device__ void end(const Params&, int lane) {
        if (lane == 0) tma_store_wait_all();
        __syncwarp();
    }
    __device__ void tile(const Params& p, const SchedGemm& s, uint32_t t_acc, int ewarp, int lane,
                         uint8_t* epi_smem) {
        const int quarter = ewarp & 3, half = ewarp >> 2;
        uint8_t* stage = epi_smem + ewarp * (32 * 128);
        uint8_t* my_row = stage + lane * 128;
        const int sw = lane & 7;
#pragma unroll 1
        for (int sub = 0; sub < BN / 2 / 64; ++sub) {
            const int c = half * (BN / 2) + sub * 64;          // first tile column of this 64-wide piece
            uint32_t raw[2][32];
            tmem_ld_32x32(t_acc + c, raw[0]);
            tmem_ld_32x32(t_acc + c + 32, raw[1]);
            const float4* b4 = reinterpret_cast<const float4*>(p.bias + s.n0 + c);
            if (lane == 0) tma_store_wait_read();              // the previous store has drained the staging tile
            __syncwarp();
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; ++j) {                       // 16-byte chunk j = columns 8j .. 8j+7
                const uint32_t* r = &raw[j >> 2][(j & 3) * 8];
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(r[e]);
                if (p.bias) {
                    const float4 lo = __ldg(b4 + 2 * j), hi = __ldg(b4 + 2 * j + 1);
                    v[0] += lo.x; v[1] += lo.y; v[2] += lo.z; v[3] += lo.w;
                    v[4] += hi.x; v[5] += hi.y; v[6] += hi.z; v[7] += hi.w;
                }
                if (p.act_mish) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = mish_fast(v[e]);
                }
                const uint4 u = make_uint4(pack2_16<T>(v[0], v[1]), pack2_16<T>(v[2], v[3]),
                                           pack2_16<T>(v[4], v[5]), pack2_16<T>(v[6], v[7]));
                *reinterpret_cast<uint4*>(my_row + ((j ^ sw) << 4)) = u;
            }
            fence_proxy_async();       // staging writes -> visible to the TMA unit
            __syncwarp();
            if (lane == 0) {
                tma_store_2d(&p.tm_c, stage, s.n0 + c, s.m0 + quarter * 32);
                tma_store_commit();
            }
        }
    }
};

// Epilogue of the in-place residual update  x <- x + A . W^T + bias  (out-proj; fp32 residual stream).
// Per warp and 32-column slab: the residual slab (32 rows x 128 B) is TMA-loaded into a swizzled
// staging tile -- two tiles per warp, the next slab's load is in flight while this one is summed,
// and the first two of a tile are requested before the accumulator is even ready -- each thread
// adds its accumulator row (tcgen05.ld) and the bias in place, and ONE TMA store writes the slab
// back.  ~3 instructions per element instead of ~11, no per-thread global addressing.
template <int BN>
struct EpiResidualTma {
    struct alignas(64) Params {
        CUtensorMap tm_x;      // (M, N) fp32 residual stream, box = 32 columns x 32 rows, 128B swizzle
        const float* bias;
    };
    static constexpr int kWarps = 8;
    static constexpr int kSlabs = BN / 2 / 32;                      // per warp and tile
    static constexpr int kSmemBytes = kWarps * 2 * 4096 + 1024;      // staging tiles + mbarriers
    uint64_t* bar;          // [2] this warp's load barriers
    uint32_t ph0, ph1;      // their phases
    __device__ void begin(const Params&, const SchedGemm&, int ewarp, int lane, uint8_t* epi_smem) {
        bar = reinterpret_cast<uint64_t*>(epi_smem + kWarps * 2 * 4096) + ewarp * 2;
        ph0 = ph1 = 0;
        if (lane == 0) {
            mbar_init(&bar[0], 1);
            mbar_init(&bar[1], 1);
            fence_barrier_init();
        }
        __syncwarp();
    }
    __device__ void end(const Params&, int lane) {
        if (lane == 0) tma_store_wait_all();
        __syncwarp();
    }
    __device__ __forceinline__ void fetch(const Params& p, const SchedGemm& s, int ewarp, int lane, uint8_t* epi_smem,
                                          int sl) {
        if (lane == 0) {
            const int quarter = ewarp & 3, half = ewarp >> 2;
            uint8_t* buf = epi_smem + (ewarp * 2 + (sl & 1)) * 4096;
            tma_store_wait_read();                       // the store that last used this tile has drained it
            mbar_arrive_expect_tx(&bar[sl & 1], 4096);
            tma_load_2d(buf, &p.tm_x, &bar[sl & 1], s.n0 + half * (BN / 2) + sl * 32, s.m0 + quarter * 32);
        }
    }
    __device__ void pre_tile(const Params& p, const SchedGemm& s, int ewarp, int lane, uint8_t* epi_smem) {
        fetch(p, s, ewarp, lane, epi_smem, 0);
        fetch(p, s, ewarp, lane, epi_smem, 1);
    }
    __device__ void tile(const Params& p, const SchedGemm& s, uint32_t t_acc, int ewarp, int lane,
                         uint8_t* epi_smem) {
        const int half = ewarp >> 2, quarter = ewarp & 3;
        const int sw = lane & 7;
#pragma unroll 1
        for (int sl = 0; sl < kSlabs; ++sl) {
            const int c = half * (BN / 2) + sl * 32;
            const uint32_t buf = smem_u32(epi_smem + (ewarp * 2 + (sl & 1)) * 4096) + lane * 128;
            uint32_t raw[32];
            tmem_ld_32x32(t_acc + c, raw);
            const float4* b4 = reinterpret_cast<const float4*>(p.bias + s.n0 + c);
            if (sl & 1) { mbar_wait(&bar[1], ph1); ph1 ^= 1; }
            else        { mbar_wait(&bar[0], ph0); ph0 ^= 1; }
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t a = buf + ((j ^ sw) << 4);
                uint4 r = lds128(a);
                float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias) bb = __ldg(b4 + j);
                r.x = __float_as_uint(__uint_as_float(r.x) + __uint_as_float(raw[4 * j + 0]) + bb.x);
                r.y = __float_as_uint(__uint_as_float(r.y) + __uint_as_float(raw[4 * j + 1]) + bb.y);
                r.z = __float_as_uint(__uint_as_float(r.z) + __uint_as_float(raw[4 * j + 2]) + bb.z);
                r.w = __float_as_uint(__uint_as_float(r.w) + __uint_as_float(raw[4 * j + 3]) + bb.w);
                sts128(a, r);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                tma_store_2d(&p.tm_x, epi_smem + (ewarp * 2 + (sl & 1)) * 4096, s.n0 + c, s.m0 + quarter * 32);
                tma_store_commit();
            }
            if (sl + 2 < kSlabs) fetch(p, s, ewarp, lane, epi_smem, sl + 2);
        }
    }
};

// fp16 operands under an epilogue that only sees the fp32 accumulator and writes fp32
template <class Epi>
struct F16Operands : Epi {
    using Operand = __half;
};
template <class T, class Epi>
using WithOperands = std::conditional_t<std::is_same<T, __half>::value, F16Operands<Epi>, Epi>;

template <int BN>
static int make_epi_params(const GemmArgs& g, typename EpiLinear<BN>::Params* ep) {
    *ep = typename EpiLinear<BN>::Params{g.bias, g.residual, g.ldr, g.out, g.ldo, g.act_mish, g.out_f32};
    return OFX_OK;
}
template <int BN>
static int make_epi_params(const GemmArgs& g, EpiStoreParams* ep) {
    OFX_TRY(make_tmap_bf16(&ep->tm_c, g.out, static_cast<uint64_t>(g.m), g.n, g.ldo, 32));
    ep->bias = g.bias;
    ep->act_mish = g.act_mish;
    return OFX_OK;
}

template <int BN>
static int make_epi_params(const GemmArgs& g, typename EpiResidualTma<BN>::Params* ep) {
    OFX_TRY(make_tmap_f32(&ep->tm_x, g.out, static_cast<uint64_t>(g.m), g.n, g.ldo, 32));
    ep->bias = g.bias;
    return OFX_OK;
}

template <int BN, int CL, class Epi>
static int launch_tc(const GemmArgs& g, cudaStream_t stream) {
    CUtensorMap tm_a, tm_b;
    OFX_TRY(make_tmap_bf16(&tm_a, g.a, static_cast<uint64_t>(g.m), g.k, g.lda, kBM));
    OFX_TRY(make_tmap_bf16(&tm_b, g.w, static_cast<uint64_t>(g.n), g.k, g.ldw, BN / CL));   // each CTA fetches BN / CL rows
    SchedGemm::Params sp{g.m, g.m_dev, g.n / BN, BN, CL};
    typename Epi::Params ep;
    OFX_TRY(make_epi_params<BN>(g, &ep));
    // stage = 16 KB of A + (BN / CL) rows of B: 48 KB single-CTA, 32 KB per CTA of a pair at BN = 256
    constexpr bool kBigEpi = Epi::kSmemBytes > 40 * 1024;   // the residual epilogue keeps 64 KB of staging tiles
    constexpr int kStages = BN >= 256 ? (CL == 2 ? (kBigEpi ? 5 : 6) : (kBigEpi ? 3 : 4))
                                      : (CL == 2 ? (kBigEpi ? 6 : 7) : (kBigEpi ? 4 : 5));
    // CL = 2: the linear layers run as CTA pairs (QKV: 116 -> 102 us at 82k tokens)
    auto kern = tc_kernel<BN, kStages, CL, SchedGemm, Epi>;
    constexpr int smem = tc_smem_bytes<BN, kStages, Epi, CL>();
    static DeviceOnce configured;  // per instantiation
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    const int m_groups = ((g.m + kBM - 1) / kBM + CL - 1) / CL;
    const int tiles = m_groups * (g.n / BN);
    const int max_clusters = sm_count() / CL;
    const int clusters = tiles < max_clusters ? tiles : max_clusters;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(clusters * CL);
    cfg.blockDim = dim3(tc_threads<Epi>());
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    count_launch();
    // Role instrumentation (OFX_TC_PROF=1) allocates and synchronises, which the C ABI promises never to do:
    // it exists only in instrumented builds (python -m outfitx_b200.build --debug -> -DOFX_DEBUG, loaded
    // through OFX_LIB_PATH), never in the product library.
#ifdef OFX_DEBUG
    static int prof_on = -1;
    static long long* prof_dev = nullptr;
    if (prof_on < 0) { const char* e = getenv("OFX_TC_PROF"); prof_on = (e && e[0] == '1') ? 1 : 0; }
    if (prof_on) {   // debug only: synchronous dump of per-CTA wait counters
        if (!prof_dev) OFX_CUDA(cudaMalloc(&prof_dev, 8 * 8 * 256));
        OFX_CUDA(cudaMemsetAsync(prof_dev, 0, 8 * 8 * 256, stream));
        OFX_CUDA(cudaMemcpyToSymbolAsync(g_tc_prof, &prof_dev, sizeof(prof_dev), 0, cudaMemcpyHostToDevice, stream));
    }
#else
    constexpr int prof_on = 0;
    long long* const prof_dev = nullptr;
#endif
    OFX_CUDA(cudaLaunchKernelEx(&cfg, kern, tm_a, tm_b, sp, ep, g.k / kBK));
    if (prof_on) {
        long long h[8 * 256];
        OFX_CUDA(cudaStreamSynchronize(stream));
        OFX_CUDA(cudaMemcpy(h, prof_dev, sizeof(h), cudaMemcpyDeviceToHost));
        fprintf(stderr, "tc prof M=%d N=%d K=%d BN=%d CL=%d: cta0 mma total %lld wait_full %lld wait_tmem_empty %lld | epi total %lld wait_tmem_full %lld ; cta100 mma %lld %lld %lld | epi %lld %lld\n",
                g.m, g.n, g.k, BN, CL, h[0], h[1], h[2], h[4], h[5], h[800], h[801], h[802], h[804], h[805]);
    }
    return OFX_OK;
}

// T: the operand type, __nv_bfloat16 or __half (the caller has rejected 16-bit output with a residual for __half)
template <int BN, class T>
static int launch_tc_cl(const GemmArgs& g, cudaStream_t stream) {
    const long long m_tiles = (g.m + kBM - 1) / kBM;
    const int cl = m_tiles < 2 ? 1 : 2;  // CTA pairs; a single M tile: nothing to pair
    // 16-bit output without residual (QKV, linear1): TMA-store epilogue; otherwise the fp32 / residual one
    const bool store16 = !g.out_f32 && !g.residual;
    if (store16) {
        if (cl == 2) return launch_tc<BN, 2, EpiStore16<BN, T>>(g, stream);
        return launch_tc<BN, 1, EpiStore16<BN, T>>(g, stream);
    }
    // in-place fp32 residual update (out-proj, linear2): TMA load / add / TMA store epilogue
    const bool inplace = g.out_f32 && g.residual == g.out && g.ldr == g.ldo && !g.act_mish && g.ldo % 4 == 0;
    if (inplace) {
        if (cl == 2) return launch_tc<BN, 2, WithOperands<T, EpiResidualTma<BN>>>(g, stream);
        return launch_tc<BN, 1, WithOperands<T, EpiResidualTma<BN>>>(g, stream);
    }
    if (cl == 2) return launch_tc<BN, 2, WithOperands<T, EpiLinear<BN>>>(g, stream);
    return launch_tc<BN, 1, WithOperands<T, EpiLinear<BN>>>(g, stream);
}

template <class T>
static int gemm_16(const GemmArgs& g, cudaStream_t stream) {
    constexpr bool f16 = std::is_same<T, __half>::value;
    const char* name = f16 ? "gemm_f16" : "gemm_bf16";
    if (g.m <= 0) return OFX_OK;
    if (g.n % 128 != 0 || g.k % kBK != 0 || g.n <= 0 || g.k <= 0)
        return fail(OFX_E_SHAPE, "%s: need N %% 128 == 0 and K %% 64 == 0 (N=%d K=%d)", name, g.n, g.k);
    if ((reinterpret_cast<uintptr_t>(g.a) | reinterpret_cast<uintptr_t>(g.w) |
         reinterpret_cast<uintptr_t>(g.out)) & 15)
        return fail(OFX_E_ARG, "%s: operands must be 16-byte aligned", name);
    if ((g.lda % 8) || (g.ldw % 8) || (g.ldo % 8) || (g.residual && (g.ldr % 4)))
        return fail(OFX_E_ARG, "%s: pitches must keep rows 16-byte aligned", name);
    // the fp16 forms of the epilogues: fp16 output (TMA store, no residual) and fp32 output
    if (f16 && (g.out_f32 == 2 || (!g.out_f32 && g.residual)))
        return fail(OFX_E_ARG, "gemm_f16: a residual needs fp32 output (out_f32 = 1)");
    // BN = 256 halves the A re-reads; use 128 when 256 does not divide N or the grid would
    // leave most SMs idle.
    const long long tiles256 = static_cast<long long>((g.m + kBM - 1) / kBM) * (g.n / 256);
    if (g.n % 256 == 0 && tiles256 >= sm_count()) return launch_tc_cl<256, T>(g, stream);
    return launch_tc_cl<128, T>(g, stream);
}

int gemm_bf16(const GemmArgs& g, cudaStream_t stream) { return gemm_16<__nv_bfloat16>(g, stream); }
int gemm_f16(const GemmArgs& g, cudaStream_t stream) { return gemm_16<__half>(g, stream); }

// -------------------------------------------------------------------------------------
// fp32 operands as bf16 hi / lo pieces (gemm.h): one thread per 4 consecutive K elements
// -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
split3_kernel(const float* __restrict__ src, long long ld, int rows, const int* __restrict__ rows_dev, int k,
              __nv_bfloat16* __restrict__ dst, int order) {
    const int n = rows_dev ? min(*rows_dev, rows) : rows;
    const int k4 = k / 4;
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    if (i >= static_cast<long long>(n) * k4) return;
    const int r = static_cast<int>(i / k4), c = static_cast<int>(i - static_cast<long long>(r) * k4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(src + r * ld + c);
    const float f[4] = {v.x, v.y, v.z, v.w};
    __nv_bfloat16 hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        hi[j] = __float2bfloat16_rn(f[j]);
        lo[j] = __float2bfloat16_rn(f[j] - __bfloat162float(hi[j]));
    }
    __nv_bfloat16* o = dst + static_cast<long long>(r) * 3 * k + c;
    const uint2 h2 = *reinterpret_cast<const uint2*>(hi), l2 = *reinterpret_cast<const uint2*>(lo);
    *reinterpret_cast<uint2*>(o) = h2;
    *reinterpret_cast<uint2*>(o + k) = order == kSplitA ? l2 : h2;
    *reinterpret_cast<uint2*>(o + 2 * k) = order == kSplitA ? h2 : l2;
}

int split_bf16x3(const float* src, long long ld, int rows, const int* rows_dev, int k, void* dst, int order,
                 cudaStream_t stream) {
    if (rows <= 0) return OFX_OK;
    if (k % 4 || ld % 4 || (reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15)
        return fail(OFX_E_ARG, "split_bf16x3: K and the pitch must be multiples of 4, pointers 16-byte aligned");
    const long long n = static_cast<long long>(rows) * (k / 4);
    split3_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(src, ld, rows, rows_dev, k,
                                                                              static_cast<__nv_bfloat16*>(dst), order);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

int gemm_f32_split(const GemmArgs& g, cudaStream_t stream) {
    if (!g.out_f32) return fail(OFX_E_ARG, "gemm_f32_split: the output must be fp32 (1) or its bf16 pieces (2)");
    if (g.out_f32 == 2 && (g.residual || g.ldo != 3LL * g.n))
        return fail(OFX_E_ARG, "gemm_f32_split: piece output needs ldo == 3 N and no residual");
    GemmArgs t = g;
    t.k = 3 * g.k;
    return gemm_bf16(t, stream);
}

}  // namespace ofx
