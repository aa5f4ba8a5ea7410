// Non-GEMM pieces of the outfit encoder, fused per row / per outfit:
//   fuse / assemble (normalise + concat|mean + prefix token + drop padded slots),
//   LayerNorm, the masked attention over up to 65 tokens, CP head (+sigmoid), FITB distances.
// Reference arithmetic: SURVEY.md App. A, i.e. torch.nn.TransformerEncoderLayer's pre-LN
// slow path as driven by /root/reference/src/models/outfit_x.py:120-172.
//
// Token layout in HBM (all activations): rows [0, B) are the prefix tokens of the B outfits,
// rows [B + off[b], B + off[b+1]) are outfit b's valid items in slot order.  Padded slots are
// dropped: they are never attended to (key-padding mask = -inf) and only token 0 is read by
// the heads, so the result is unchanged (SURVEY.md App. A.4); the model has no positional
// encoding, so valid items may come from any slot.
#include "encoder_ops.h"
#include "ptx.cuh"

namespace ofx {

template <class T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<__half>(__half v) { return __half2float(v); }
template <class T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

// 8 consecutive elements (16-byte aligned for bf16 / fp16, 32-byte for fp32) <-> fp32 registers
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
    float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 u = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void load8(const __half* p, float (&v)[8]) {
    uint4 u = *reinterpret_cast<const uint4*>(p);
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = u;
}
__device__ __forceinline__ void store8(__half* p, const float (&v)[8]) {
    uint4 u;
    __half2* h = reinterpret_cast<__half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = u;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ offsets
// off[b] = number of valid items in outfits < b; off[B] = total items; n_tok = B + off[B].
__global__ void __launch_bounds__(1024)
scan_valid_kernel(const uint8_t* __restrict__ mask, int batch, int max_items, int* __restrict__ off,
                  int* __restrict__ n_tok) {
    __shared__ int warp_tot[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < batch; base += 1024) {
        const int b = base + threadIdx.x;
        int cnt = 0;
        if (b < batch)
            for (int j = 0; j < max_items; ++j) cnt += mask[b * max_items + j] == 0;
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int t = warp_tot[lane], s = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int u = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += u;
            }
            warp_tot[lane] = s - t;  // exclusive
        }
        __syncthreads();
        const int excl = carry + warp_tot[warp] + incl - cnt;
        if (b < batch) off[b] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + cnt;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        off[batch] = carry;
        *n_tok = batch + carry;
    }
}

// ------------------------------------------------------------------ fusion of one item row
// One warp produces one fused row in registers: lane l holds elements l*4 + 128*i (float4).
// concat: [img/|img| ; txt/|txt|]  (2*dpm)    mean: (img/|img| + txt/|txt|)/2  (dpm)
template <int DM>
__device__ __forceinline__ void load_fused_row(float4 (&v)[DM / 128], const float* img,
                                               const float* txt, int dpm, int mode, int normalize,
                                               int lane) {
    constexpr int NV = DM / 128;
    if (mode == OFX_FUSE_CONCAT) {
        // DM = 2*dpm: vectors [0, NV/2) come from img, the rest from txt
        float si = 0.f, st = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int e = i * 128 + lane * 4;
            const bool is_img = e < dpm;
            v[i] = *reinterpret_cast<const float4*>(is_img ? img + e : txt + (e - dpm));
            float s = v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
            if (is_img) si += s; else st += s;
        }
        if (normalize) {
            si = 1.f / fmaxf(sqrtf(warp_sum(si)), 1e-12f);
            st = 1.f / fmaxf(sqrtf(warp_sum(st)), 1e-12f);
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const float s = (i * 128 + lane * 4 < dpm) ? si : st;
                v[i].x *= s; v[i].y *= s; v[i].z *= s; v[i].w *= s;
            }
        }
    } else {
        float4 t[NV];
        float si = 0.f, st = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int e = i * 128 + lane * 4;
            v[i] = *reinterpret_cast<const float4*>(img + e);
            t[i] = *reinterpret_cast<const float4*>(txt + e);
            si += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
            st += t[i].x * t[i].x + t[i].y * t[i].y + t[i].z * t[i].z + t[i].w * t[i].w;
        }
        float ai = 0.5f, at = 0.5f;
        if (normalize) {
            ai = 0.5f / fmaxf(sqrtf(warp_sum(si)), 1e-12f);
            at = 0.5f / fmaxf(sqrtf(warp_sum(st)), 1e-12f);
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            v[i].x = v[i].x * ai + t[i].x * at; v[i].y = v[i].y * ai + t[i].y * at;
            v[i].z = v[i].z * ai + t[i].z * at; v[i].w = v[i].w * ai + t[i].w * at;
        }
    }
}

// standalone fusion (ofx_fuse): one warp per row
template <int DM>
__global__ void __launch_bounds__(256)
fuse_kernel(const float* __restrict__ img, const float* __restrict__ txt, long long rows, int dpm,
            int mode, int normalize, float* __restrict__ out) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    float4 v[DM / 128];
    load_fused_row<DM>(v, img + row * dpm, txt + row * dpm, dpm, mode, normalize, lane);
#pragma unroll
    for (int i = 0; i < DM / 128; ++i)
        *reinterpret_cast<float4*>(out + row * DM + i * 128 + lane * 4) = v[i];
}

int fuse_rows(const float* img, const float* txt, long long rows, int dpm, int mode, int normalize,
              float* out, cudaStream_t stream) {
    const int dm = mode == OFX_FUSE_CONCAT ? 2 * dpm : dpm;
    const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
    if (rows <= 0) return OFX_OK;
    switch (dm) {
        case 512: fuse_kernel<512><<<grid, 256, 0, stream>>>(img, txt, rows, dpm, mode, normalize, out); break;
        case 1024: fuse_kernel<1024><<<grid, 256, 0, stream>>>(img, txt, rows, dpm, mode, normalize, out); break;
        case 1536: fuse_kernel<1536><<<grid, 256, 0, stream>>>(img, txt, rows, dpm, mode, normalize, out); break;
        default: return fail(OFX_E_SHAPE, "ofx_fuse: fused width %d not in {512,1024,1536}", dm);
    }
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

// ------------------------------------------------------------------ LayerNorm of a row held
// in registers (two-pass in registers: mean, then biased variance), eps = 1e-5.
template <int DM, class T>
__device__ __forceinline__ void ln_store(const float4 (&v)[DM / 128], const float* __restrict__ gamma,
                                         const float* __restrict__ beta, T* __restrict__ out, int lane) {
    constexpr int NV = DM / 128;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) s += v[i].x + v[i].y + v[i].z + v[i].w;
    const float mu = warp_sum(s) * (1.f / DM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
        q += a * a + b * b + c * c + d * d;
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / DM) + 1e-5f);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int e = i * 128 + lane * 4;
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + e));
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta + e));
        float y0 = (v[i].x - mu) * rstd * g.x + b.x, y1 = (v[i].y - mu) * rstd * g.y + b.y;
        float y2 = (v[i].z - mu) * rstd * g.z + b.z, y3 = (v[i].w - mu) * rstd * g.w + b.w;
        if constexpr (sizeof(T) == 4) {
            *reinterpret_cast<float4*>(out + e) = make_float4(y0, y1, y2, y3);
        } else {
            *reinterpret_cast<uint2*>(out + e) = make_uint2(pack2_16<T>(y0, y1), pack2_16<T>(y2, y3));
        }
    }
}

// ------------------------------------------------------------------ assemble (+ LayerNorm 1 of layer 0)
// One warp per (outfit, slot): slot 0 = prefix token (outfit_token | [target_img ; text]),
// slot s>0 = item s-1.  Writes the fp32 residual stream x and h = LN1_0(x).
template <int DM, class T>
__global__ void __launch_bounds__(256)
assemble_kernel(AssembleArgs a, float* __restrict__ x, T* __restrict__ h) {
    const long long gw = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    const int slots = a.max_items + 1;
    const int b = static_cast<int>(gw / slots), s = static_cast<int>(gw % slots);
    if (b >= a.batch) return;
    const int lane = threadIdx.x & 31;
    constexpr int NV = DM / 128;
    float4 v[NV];
    long long row;
    if (s == 0) {
        row = b;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int e = i * 128 + lane * 4;
            if (a.task == OFX_TASK_CP) v[i] = __ldg(reinterpret_cast<const float4*>(a.outfit_token + e));
            else if (e < DM / 2) v[i] = __ldg(reinterpret_cast<const float4*>(a.target_img + e));
            else v[i] = *reinterpret_cast<const float4*>(a.text + static_cast<long long>(b) * (DM / 2) + (e - DM / 2));
        }
    } else {
        const uint8_t* m = a.mask + static_cast<long long>(b) * a.max_items;
        if (m[s - 1]) return;  // padded slot: dropped
        int rank = 0;
        for (int j = 0; j < s - 1; ++j) rank += m[j] == 0;
        row = a.batch + a.off[b] + rank;
        if (lane == 0) a.owner[row] = b;
        long long item = static_cast<long long>(b) * a.max_items + (s - 1);
        bool in_table = true;
        if (a.item_ids) {            // device-side collate: the slot names a row of the item tables
            item = a.item_ids[item];
            in_table = item >= 0 && item < a.n_table_rows;
            if (!in_table) item = 0;
        }
        if (a.emb) {
#pragma unroll
            for (int i = 0; i < NV; ++i)
                v[i] = *reinterpret_cast<const float4*>(a.emb + item * DM + i * 128 + lane * 4);
        } else {
            load_fused_row<DM>(v, a.img + item * a.dpm, a.txt + item * a.dpm, a.dpm, a.fuse_mode,
                               a.normalize, lane);
        }
        if (!in_table) {
#pragma unroll
            for (int i = 0; i < NV; ++i) v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) *reinterpret_cast<float4*>(x + row * DM + i * 128 + lane * 4) = v[i];
    ln_store<DM, T>(v, a.ln_w, a.ln_b, h + row * DM, lane);
}

template <class T>
int assemble(const AssembleArgs& a, int dm, float* x, T* h, cudaStream_t stream) {
    const long long warps = static_cast<long long>(a.batch) * (a.max_items + 1);
    const unsigned grid = static_cast<unsigned>((warps + 7) / 8);
    switch (dm) {
        case 512: assemble_kernel<512, T><<<grid, 256, 0, stream>>>(a, x, h); break;
        case 1024: assemble_kernel<1024, T><<<grid, 256, 0, stream>>>(a, x, h); break;
        case 1536: assemble_kernel<1536, T><<<grid, 256, 0, stream>>>(a, x, h); break;
        default: return fail(OFX_E_SHAPE, "d_model %d not in {512,1024,1536}", dm);
    }
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}
template int assemble<float>(const AssembleArgs&, int, float*, float*, cudaStream_t);
template int assemble<__nv_bfloat16>(const AssembleArgs&, int, float*, __nv_bfloat16*, cudaStream_t);
template int assemble<__half>(const AssembleArgs&, int, float*, __half*, cudaStream_t);

int scan_valid(const uint8_t* mask, int batch, int max_items, int* off, int* n_tok, cudaStream_t stream) {
    scan_valid_kernel<<<1, 1024, 0, stream>>>(mask, batch, max_items, off, n_tok);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

// ------------------------------------------------------------------ LayerNorm: one warp per row
template <int DM, class T>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, int rows, const int* __restrict__ rows_dev,
                 const float* __restrict__ gamma, const float* __restrict__ beta, T* __restrict__ out) {
    const int n = rows_dev ? min(*rows_dev, rows) : rows;
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    const int lane = threadIdx.x & 31;
    float4 v[DM / 128];
#pragma unroll
    for (int i = 0; i < DM / 128; ++i)
        v[i] = *reinterpret_cast<const float4*>(x + row * DM + i * 128 + lane * 4);
    ln_store<DM, T>(v, gamma, beta, out + row * DM, lane);
}

template <class T>
int layernorm(const float* x, int rows, const int* rows_dev, int dm, const float* gamma,
              const float* beta, T* out, cudaStream_t stream) {
    if (rows <= 0) return OFX_OK;
    const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
    switch (dm) {
        case 512: layernorm_kernel<512, T><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, out); break;
        case 1024: layernorm_kernel<1024, T><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, out); break;
        case 1536: layernorm_kernel<1536, T><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, out); break;
        default: return fail(OFX_E_SHAPE, "d_model %d not in {512,1024,1536}", dm);
    }
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}
// LayerNorm whose output is the activation operand of a split-bf16 GEMM (precision fp32 on the tensor cores, gemm.h):
// the normalised fp32 row is written as its bf16 pieces [hi | lo | hi], row pitch 3 DM -- same arithmetic as
// ln_store<DM, float> followed by split3_kernel, one pass instead of two.
template <int DM>
__global__ void __launch_bounds__(256)
layernorm_split3_kernel(const float* __restrict__ x, int rows, const int* __restrict__ rows_dev,
                        const float* __restrict__ gamma, const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
    constexpr int NV = DM / 128;
    const int n = rows_dev ? min(*rows_dev, rows) : rows;
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    const int lane = threadIdx.x & 31;
    float4 v[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(x + row * DM + i * 128 + lane * 4);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) s += v[i].x + v[i].y + v[i].z + v[i].w;
    const float mu = warp_sum(s) * (1.f / DM);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
        q += a * a + b * b + c * c + d * d;
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / DM) + 1e-5f);
    __nv_bfloat16* o = out + row * (3 * DM);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int e = i * 128 + lane * 4;
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + e));
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta + e));
        const float y[4] = {(v[i].x - mu) * rstd * g.x + b.x, (v[i].y - mu) * rstd * g.y + b.y,
                            (v[i].z - mu) * rstd * g.z + b.z, (v[i].w - mu) * rstd * g.w + b.w};
        __nv_bfloat16 hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            hi[j] = __float2bfloat16_rn(y[j]);
            lo[j] = __float2bfloat16_rn(y[j] - __bfloat162float(hi[j]));
        }
        const uint2 h2 = *reinterpret_cast<const uint2*>(hi), l2 = *reinterpret_cast<const uint2*>(lo);
        *reinterpret_cast<uint2*>(o + e) = h2;
        *reinterpret_cast<uint2*>(o + DM + e) = l2;
        *reinterpret_cast<uint2*>(o + 2 * DM + e) = h2;
    }
}

int layernorm_split3(const float* x, int rows, const int* rows_dev, int dm, const float* gamma, const float* beta,
                     void* out, cudaStream_t stream) {
    if (rows <= 0) return OFX_OK;
    const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
    __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
    switch (dm) {
        case 512: layernorm_split3_kernel<512><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, o); break;
        case 1024: layernorm_split3_kernel<1024><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, o); break;
        case 1536: layernorm_split3_kernel<1536><<<grid, 256, 0, stream>>>(x, rows, rows_dev, gamma, beta, o); break;
        default: return fail(OFX_E_SHAPE, "d_model %d not in {512,1024,1536}", dm);
    }
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

template int layernorm<float>(const float*, int, const int*, int, const float*, const float*, float*, cudaStream_t);
template int layernorm<__nv_bfloat16>(const float*, int, const int*, int, const float*, const float*, __nv_bfloat16*, cudaStream_t);
template int layernorm<__half>(const float*, int, const int*, int, const float*, const float*, __half*, cudaStream_t);

// ------------------------------------------------------------------ cast rows fp32 -> T
template <class T>
__global__ void cast_kernel(const float* __restrict__ in, long long n, T* __restrict__ out) {
    long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    float4 v = *reinterpret_cast<const float4*>(in + i);
    out[i] = from_f<T>(v.x); out[i + 1] = from_f<T>(v.y); out[i + 2] = from_f<T>(v.z); out[i + 3] = from_f<T>(v.w);
}
template <class T>
int cast_rows(const float* in, long long n, T* out, cudaStream_t stream) {
    if (n <= 0) return OFX_OK;
    cast_kernel<T><<<static_cast<unsigned>((n / 4 + 255) / 256), 256, 0, stream>>>(in, n, out);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}
template int cast_rows<float>(const float*, long long, float*, cudaStream_t);
template int cast_rows<__nv_bfloat16>(const float*, long long, __nv_bfloat16*, cudaStream_t);
template int cast_rows<__half>(const float*, long long, __half*, cudaStream_t);

// ------------------------------------------------------------------ attention, CUDA cores
// This lane's slice of the key (or value) rows j0 .. j0 + 3 of an outfit.  The four row loads are issued back to
// back, so every thread keeps several independent 16-byte loads in flight; rows past S are clamped to key 0 (a valid,
// cached address) and masked by the caller.
template <int NP, class T>
__device__ __forceinline__ void load_key_group(const T* src, long long ld, int b, int base, int S, int j0,
                                               float (&t)[4][NP][8]) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int j = j0 + u;
        const long long r = (j == 0 || j >= S) ? b : base + j - 1;
#pragma unroll
        for (int p = 0; p < NP; ++p) load8(src + r * ld + 32 * p, t[u][p]);
    }
}

// q . k over the head: each of the row's four lanes sums its 8 x NP dims, two xor-shuffles combine the partial sums
template <int NP>
__device__ __forceinline__ float dot_4lanes(const float (&q)[NP][8], const float (&k)[NP][8]) {
    float acc = 0.f;
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc = fmaf(q[p][e], k[p][e], acc);
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    return acc;
}

// One (token row, head) of an outfit with S > 17 tokens: one pass over groups of 4 keys with a running
// maximum and sum (online softmax); the output accumulator is rescaled whenever the maximum grows.
template <int HD, class T>
__device__ __forceinline__ void attention_row_online(const AttnArgs& a, int b, int base, int S, const T* qp,
                                                     const T* kp, const T* vp, T* op) {
    constexpr int NP = HD / 32;
    float q[NP][8];
#pragma unroll
    for (int p = 0; p < NP; ++p) load8(qp + 32 * p, q[p]);
    const float scale = rsqrtf(static_cast<float>(HD));
    float mx = -INFINITY, den = 0.f;
    float o[NP][8];
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 8; ++e) o[p][e] = 0.f;
#pragma unroll 1
    for (int j0 = 0; j0 < S; j0 += 4) {
        float t[4][NP][8];
        load_key_group<NP>(kp, a.ldk, b, base, S, j0, t);
        float sc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float acc = dot_4lanes<NP>(q, t[u]);
            sc[u] = j0 + u < S ? acc * scale : -INFINITY;
        }
        const float m_new = fmaxf(mx, fmaxf(fmaxf(sc[0], sc[1]), fmaxf(sc[2], sc[3])));   // finite: key 0 is valid
        const float corr = sizeof(T) == 4 ? expf(mx - m_new) : __expf(mx - m_new);      // exp(-inf) = 0 at j0 = 0
        mx = m_new;
        den *= corr;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            sc[u] = sizeof(T) == 4 ? expf(sc[u] - mx) : __expf(sc[u] - mx);
            den += sc[u];
        }
        load_key_group<NP>(vp, a.ldv, b, base, S, j0, t);
#pragma unroll
        for (int p = 0; p < NP; ++p)
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float acc = o[p][e] * corr;
#pragma unroll
                for (int u = 0; u < 4; ++u) acc = fmaf(sc[u], t[u][p][e], acc);
                o[p][e] = acc;
            }
    }
    const float inv = 1.f / den;
#pragma unroll
    for (int p = 0; p < NP; ++p) {
#pragma unroll
        for (int e = 0; e < 8; ++e) o[p][e] *= inv;
        store8(op + 32 * p, o[p]);
    }
}

// Four consecutive lanes serve one (token row, head): lane `sub` owns dims {32p + 8 sub .. +8}
// of the head for every 32-dim piece p, so each warp-wide 16-byte load covers contiguous 64-byte
// runs (8 heads x 4 lanes = 512 contiguous bytes of one token row at head_dim 32) -- fully
// coalesced q / K / V loads and output stores, no shared memory.  Partial q.k sums are combined
// with two xor-shuffles; the S <= 17 scores, the softmax and the output slice stay in registers.
// Softmax runs over the outfit's S = 1 + n valid tokens only: the dropped pads are exactly the
// -inf keys of the reference's float key-padding mask.
// row0_only: the pruned last layer (queries = the B prefix tokens, from a separate buffer).
// LONG = false: every outfit of the launch has S <= 17 tokens.  LONG = true (max_s > 17): rows of outfits with
// more tokens take the online softmax of attention_row_online; the others run the same two-pass code as with
// LONG = false.  All lanes of a row share S, so the branch is warp-uniform.
template <int HD, class T, bool LONG>
__global__ void __launch_bounds__(256)
attention_kernel(AttnArgs a) {
    constexpr int NP = HD / 32;  // 8-dim pieces per lane
    const int n_rows = a.row0_only ? a.batch : min(*a.n_tok, a.max_rows);
    const int row = blockIdx.x * 4 + (threadIdx.x >> 6);
    const int head = (threadIdx.x >> 2) & 15;
    const int sub = threadIdx.x & 3;
    if (row >= n_rows) return;  // whole 64-thread groups leave together (shuffles stay inside 4 lanes)
    const int b = row < a.batch ? row : a.owner[row];
    const int base = a.batch + a.off[b];
    const int S = 1 + (a.off[b + 1] - a.off[b]);
    const int col = head * HD + sub * 8;
    const T* kp = static_cast<const T*>(a.k) + col;
    const T* vp = static_cast<const T*>(a.v) + col;
    const T* qp = static_cast<const T*>(a.q) + static_cast<long long>(row) * a.ldq + col;
    T* op = static_cast<T*>(a.out) + static_cast<long long>(row) * a.ldo + col;
    if constexpr (LONG) {
        if (S > 17) {
            attention_row_online<HD, T>(a, b, base, S, qp, kp, vp, op);
            return;
        }
    }

    float q[NP][8];
#pragma unroll
    for (int p = 0; p < NP; ++p) load8(qp + 32 * p, q[p]);
    // keys are taken four at a time (load_key_group)
    constexpr int kGroups = 5;  // 5 x 4 >= 17
    float sc[kGroups * 4];
    const float scale = rsqrtf(static_cast<float>(HD));
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
#pragma unroll
        for (int u = 0; u < 4; ++u) sc[4 * g + u] = -INFINITY;
        if (4 * g < S) {
            float t[4][NP][8];
            load_key_group<NP>(kp, a.ldk, b, base, S, 4 * g, t);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float acc = dot_4lanes<NP>(q, t[u]);
                if (4 * g + u < S) sc[4 * g + u] = acc * scale;
            }
        }
    }
    float mx = sc[0];
#pragma unroll
    for (int j = 1; j < kGroups * 4; ++j) mx = fmaxf(mx, sc[j]);
    float den = 0.f;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        if (4 * g < S) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float e = sizeof(T) == 4 ? expf(sc[4 * g + u] - mx) : __expf(sc[4 * g + u] - mx);
                sc[4 * g + u] = e;  // exp(-inf) = 0 for the masked tail of the group
                den += e;
            }
        }
    }
    const float inv = 1.f / den;
    float o[NP][8];
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int e = 0; e < 8; ++e) o[p][e] = 0.f;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        if (4 * g < S) {
            float t[4][NP][8];
            load_key_group<NP>(vp, a.ldv, b, base, S, 4 * g, t);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float pj = sc[4 * g + u];
#pragma unroll
                for (int p = 0; p < NP; ++p)
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[p][e] = fmaf(pj, t[u][p][e], o[p][e]);
            }
        }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) {
#pragma unroll
        for (int e = 0; e < 8; ++e) o[p][e] *= inv;
        store8(op + 32 * p, o[p]);
    }
}

// ------------------------------------------------------------------ attention, bf16 / fp16 path
// One CTA (4 warps) per outfit.  The outfit's q / K / V rows (S <= 65 tokens x d_model) are
// gathered into shared memory once with 16-byte cp.async (row stride d_model + 8 elements, so
// the ldmatrix row addresses of a fragment fall into distinct banks); every warp then serves 4
// of the 16 heads with warp-level tensor-core MMAs (mma.sync m16n8k16, bf16 or fp16 in / fp32 out):
// scores = q.K^T over 16-key tiles, masked warp-shuffle softmax in registers, out = P.V with V
// read through ldmatrix.trans.  The S x S problem is far below a tcgen05 tile (SURVEY.md H1);
// what matters is that each q / K / V element is read from global memory exactly once and that
// the instruction count per (outfit, head) is ~100 instead of ~1400 for the CUDA-core version.
// Rows >= S of a 16-row tile are redirected to a zero row, so padded keys contribute
// exp(-inf) * 0 = 0 exactly -- the reference's -inf key-padding mask.
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
template <class T>
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    if constexpr (std::is_same<T, __half>::value)
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
            "{%0, %1, %2, %3};"
            : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    else
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
            "{%0, %1, %2, %3};"
            : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
            : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

constexpr int kAttnMaxS = 17;       // tokens at up to 16 item slots
constexpr int kAttnLongMaxS = 65;   // tokens at up to 64 item slots

// The kernel picks the body per CTA from the outfit's item count, so the common cases run straight-line code
// without per-tile predicates:
//   SMALL (MT = KT = 1): S <= 8 tokens (40 % of the outfits at n ~ U{2..16}): only query rows 0..7 (h = 0) and the
//     first 8-key n-tile exist, so the second score MMA, half of the softmax and half of the output stores are skipped.
//   MT = KT = 1: S <= 16 tokens (one 16-row query tile, one 16-key tile) -- 14 of 15 outfits when n ~ U{2..16}.
//   MT = KT = 2: adds the second tiles for S = 17.
//   PASSES (MT = 1, KT = 5): S <= 65 tokens.  Each warp walks the up to five 16-row query tiles of its heads one
//     pass at a time; per pass it scores all 16-key tiles in use into registers (10 n8-tiles) and runs the
//     softmax over the whole row.  Under row0_only only query tile 0 exists.
//
// NSPLIT > 1 splits the 16 heads over NSPLIT CTAs (grid.y): each gathers only its DM / NSPLIT columns
// (still >= 512 contiguous bytes per row), so a CTA needs 1 / NSPLIT of the shared memory and twice
// as many CTAs are resident per SM -- the kernel is latency-bound (gather -> compute -> store with no
// overlap inside a CTA), so residency is what hides the gather.
// T: the 16-bit type of q / K / V, P and the output (__nv_bfloat16 or __half)
// MT, KT: 16-row query tiles per pass, 16-key tiles
// cap: rows reserved for each of q, K and V in shared memory (kAttnMaxS, or max_s when max_s > 17)
template <int HD, int NSPLIT, class T, int MT, int KT, bool SMALL, bool PASSES>
__device__ __forceinline__ void attention_mma_body(const AttnArgs& a, uint8_t* sm, int cap) {
    static_assert(PASSES ? MT == 1 : MT <= 2 && KT <= 2, "a pass is one query tile; without passes, two at most");
    static_assert(!SMALL || (MT == 1 && KT == 1), "SMALL is one tile");
    constexpr int NH = SMALL ? 1 : 2;            // row halves (g, g + 8) in use
    constexpr int NNT = SMALL ? 1 : 2 * KT;      // 8-key n-tiles in use
    constexpr int DM = 16 * HD / NSPLIT;     // columns this CTA serves
    constexpr int HPW = 4 / NSPLIT;          // heads per warp
    constexpr int CPR = DM / 8;              // 16-byte chunks per row
    constexpr int STRIDE = (DM + 8) * 2;     // bytes per shared-memory row
    constexpr int KS = HD / 16;              // k-steps over the head dimension
    uint8_t* s_q = sm;
    uint8_t* s_k = sm + cap * STRIDE;
    uint8_t* s_v = s_k + cap * STRIDE;
    uint8_t* s_z = s_v + cap * STRIDE;   // one zero row
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int base = a.batch + a.off[b];
    const int S = min(1 + (a.off[b + 1] - a.off[b]), PASSES ? cap : kAttnMaxS);
    const int n_q = a.row0_only ? 1 : S;
    const int gcol = NSPLIT > 1 ? static_cast<int>(blockIdx.y) * DM : 0;     // first global column of this CTA
    const T* gq = static_cast<const T*>(a.q) + gcol;
    const T* gk = static_cast<const T*>(a.k) + gcol;
    const T* gv = static_cast<const T*>(a.v) + gcol;

    for (int i = tid; i < STRIDE / 16; i += 128) reinterpret_cast<uint4*>(s_z)[i] = make_uint4(0, 0, 0, 0);
    // gather: 16-byte cp.async chunks, (row, chunk) advanced incrementally (no per-chunk division)
    auto load_rows = [&](const T* g, long long ld, uint8_t* dst, int n_rows) {
        int j = tid / CPR, cc = tid - j * CPR;
        while (j < n_rows) {
            const long long row = j == 0 ? b : base + j - 1;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(
                             __cvta_generic_to_shared(dst + j * STRIDE + cc * 16))),
                         "l"(g + row * ld + cc * 8)
                         : "memory");
            cc += 128;
            while (cc >= CPR) { cc -= CPR; ++j; }
        }
    };
    load_rows(gk, a.ldk, s_k, S);
    load_rows(gv, a.ldv, s_v, S);
    load_rows(gq, a.ldq, s_q, n_q);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    const uint32_t q_s = static_cast<uint32_t>(__cvta_generic_to_shared(s_q));
    const uint32_t k_s = static_cast<uint32_t>(__cvta_generic_to_shared(s_k));
    const uint32_t v_s = static_cast<uint32_t>(__cvta_generic_to_shared(s_v));
    const uint32_t z_s = static_cast<uint32_t>(__cvta_generic_to_shared(s_z));
    const int n_pass = PASSES ? (n_q + 15) / 16 : 1;
    const int n_mt = MT > 1 && n_q > 16 ? 2 : 1;                              // 16-row query tiles in use per pass
    const int n_kt = PASSES ? (S + 15) / 16 : KT > 1 && S > 16 ? 2 : 1;      // 16-key tiles in use
    const int g = lane >> 2, t4 = lane & 3;
    // ldmatrix row / column roles of this lane
    const int a_row = (lane & 7) + 8 * ((lane >> 3) & 1), a_col = 8 * (lane >> 4);     // A operand (q) and V^T
    const int b_row = (lane & 7) + 8 * (lane >> 4), b_col = 8 * ((lane >> 3) & 1);     // B operand (K)
    const float sl2 = rsqrtf(static_cast<float>(HD)) * 1.4426950408889634f;           // scale * log2(e)
    uint32_t kvalid = 0;      // bit nt*2+e: key nt*8 + 2*t4 + e exists
#pragma unroll
    for (int nt = 0; nt < 2 * KT; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) kvalid |= (nt * 8 + 2 * t4 + e < S ? 1u : 0u) << (nt * 2 + e);

#pragma unroll 1
    for (int hh = 0; hh < HPW; ++hh) {
        const int col0 = (warp * HPW + hh) * HD;   // first (CTA-local) column of this head
#pragma unroll 1
        for (int pass = 0; pass < n_pass; ++pass) {
            const int row0 = pass * 16 * MT;           // first query row of this pass
            float sc[MT][2 * KT][4];                          // [query tile][8-key tile][fragment]
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < 2 * KT; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) sc[mt][nt][e] = 0.f;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                uint32_t qa[MT][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    if (mt < n_mt) {
                        const int r = row0 + mt * 16 + a_row;
                        ldsm_x4(qa[mt], (r < n_q ? q_s + r * STRIDE : z_s) + (col0 + ks * 16 + a_col) * 2);
                    }
                }
#pragma unroll
                for (int kt = 0; kt < KT; ++kt) {
                    if (kt < n_kt) {
                        uint32_t kb[4];
                        const int r = kt * 16 + b_row;
                        ldsm_x4(kb, (r < S ? k_s + r * STRIDE : z_s) + (col0 + ks * 16 + b_col) * 2);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            if (mt < n_mt) {
                                mma_16816<T>(sc[mt][2 * kt], qa[mt], kb[0], kb[1]);
                                if constexpr (!SMALL) mma_16816<T>(sc[mt][2 * kt + 1], qa[mt], kb[2], kb[3]);
                            }
                        }
                    }
                }
            }
            // masked softmax over the keys of each query row (rows g and g + 8 of every tile)
            uint32_t pa[MT][KT][4];      // P as the A operand of P.V: [query tile][16-key tile]
            float inv[MT][2];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                if (mt < n_mt) {
#pragma unroll
                    for (int h = 0; h < NH; ++h) {      // h = 0: row g, h = 1: row g + 8
                        float mx = -INFINITY;
#pragma unroll
                        for (int nt = 0; nt < NNT; ++nt)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                float v = (kvalid >> (nt * 2 + e)) & 1u ? sc[mt][nt][2 * h + e] * sl2 : -INFINITY;
                                sc[mt][nt][2 * h + e] = v;
                                mx = fmaxf(mx, v);
                            }
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
                        float sum = 0.f;
#pragma unroll
                        for (int nt = 0; nt < NNT; ++nt)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const float pz = ex2_fast(sc[mt][nt][2 * h + e] - mx);   // key 0 is always valid: mx finite
                                sc[mt][nt][2 * h + e] = pz;
                                sum += pz;
                            }
                        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                        inv[mt][h] = 1.f / sum;
                    }
#pragma unroll
                    for (int kt = 0; kt < KT; ++kt) {
                        pa[mt][kt][0] = pack2_16<T>(sc[mt][2 * kt][0], sc[mt][2 * kt][1]);
                        if constexpr (SMALL) {     // rows 8..15 and keys 8..15 do not exist
                            pa[mt][kt][1] = pa[mt][kt][2] = pa[mt][kt][3] = 0u;
                        } else {
                            pa[mt][kt][1] = pack2_16<T>(sc[mt][2 * kt][2], sc[mt][2 * kt][3]);
                            pa[mt][kt][2] = pack2_16<T>(sc[mt][2 * kt + 1][0], sc[mt][2 * kt + 1][1]);
                            pa[mt][kt][3] = pack2_16<T>(sc[mt][2 * kt + 1][2], sc[mt][2 * kt + 1][3]);
                        }
                    }
                }
            }
            // out = P . V, 16 head dims at a time
#pragma unroll
            for (int dp = 0; dp < KS; ++dp) {
                float o[MT][2][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int x = 0; x < 2; ++x)
#pragma unroll
                        for (int e = 0; e < 4; ++e) o[mt][x][e] = 0.f;
#pragma unroll
                for (int kt = 0; kt < KT; ++kt) {
                    if (kt < n_kt) {
                        uint32_t vb[4];
                        const int r = kt * 16 + a_row;
                        ldsm_x4_trans(vb, (r < S ? v_s + r * STRIDE : z_s) + (col0 + dp * 16 + a_col) * 2);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            if (mt < n_mt) {
                                mma_16816<T>(o[mt][0], pa[mt][kt], vb[0], vb[1]);
                                mma_16816<T>(o[mt][1], pa[mt][kt], vb[2], vb[3]);
                            }
                        }
                    }
                }
                // the head's slice of the pass's q rows is dead (fragments are in registers): reuse it for the output
                __syncwarp();
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    if (mt < n_mt) {
#pragma unroll
                        for (int h = 0; h < NH; ++h) {
                            const int r = row0 + mt * 16 + g + 8 * h;
                            if (r < n_q) {
#pragma unroll
                                for (int x = 0; x < 2; ++x)
                                    *reinterpret_cast<uint32_t*>(s_q + r * STRIDE + (col0 + dp * 16 + x * 8 + 2 * t4) * 2) =
                                        pack2_16<T>(o[mt][x][2 * h] * inv[mt][h], o[mt][x][2 * h + 1] * inv[mt][h]);
                            }
                        }
                    }
                }
            }
        }
    }
    __syncthreads();
    T* go = static_cast<T*>(a.out) + gcol;
    for (int c = tid; c < n_q * CPR; c += 128) {
        const int r = c / CPR, cc = c - r * CPR;
        const long long row = r == 0 ? b : base + r - 1;
        *reinterpret_cast<uint4*>(go + row * a.ldo + cc * 8) = *reinterpret_cast<const uint4*>(s_q + r * STRIDE + cc * 16);
    }
}

// LONG (max_s > 17): shared-memory rows are max_s apart, and outfits of more than 16 items take the PASSES body
template <int HD, int NSPLIT, class T, bool LONG>
__global__ void __launch_bounds__(128)
attention_mma_kernel(const AttnArgs a) {
    extern __shared__ __align__(16) uint8_t attn_sm[];
    const int cap = LONG ? a.max_s : kAttnMaxS;
    const int b = blockIdx.x;
    const int n_items = a.off[b + 1] - a.off[b];
    if (n_items < 8) attention_mma_body<HD, NSPLIT, T, 1, 1, true, false>(a, attn_sm, cap);            // S = 1 + n <= 8
    else if (n_items < 16) attention_mma_body<HD, NSPLIT, T, 1, 1, false, false>(a, attn_sm, cap);     // S <= 16
    else if (!LONG || n_items == 16) attention_mma_body<HD, NSPLIT, T, 2, 2, false, false>(a, attn_sm, cap);
    else attention_mma_body<HD, NSPLIT, T, 1, (kAttnLongMaxS + 15) / 16, false, true>(a, attn_sm, cap);
}

// Shared memory is (3 cap + 1) rows of (16 HD / NSPLIT + 8) x 2 bytes.  The 16 heads of an outfit split over NSPLIT
// CTAs: 2 with max_s <= 17; at max_s = 65 the split that keeps two CTAs per SM is 2 at head_dim 32 (103 KB) and 4 at
// 64 (103 KB); at 96 a split of 4 (154 KB) is the least that fits at all (2 needs 304 KB).
template <int HD> constexpr int attn_long_split() { return HD == 32 ? 2 : 4; }
template <int HD, int NSPLIT> constexpr int attn_mma_smem(int cap) { return (3 * cap + 1) * (16 * HD / NSPLIT + 8) * 2; }

template <int HD, class T, bool LONG>
static int launch_attention_mma(const AttnArgs& a, cudaStream_t stream) {
    constexpr int kSplit = LONG ? attn_long_split<HD>() : 2;
    constexpr int kMaxCap = LONG ? kAttnLongMaxS : kAttnMaxS;
    const int cap = LONG ? a.max_s : kAttnMaxS;
    static DeviceOnce configured;
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(attention_mma_kernel<HD, kSplit, T, LONG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      attn_mma_smem<HD, kSplit>(kMaxCap)));
    }
    attention_mma_kernel<HD, kSplit, T, LONG><<<dim3(a.batch, kSplit), 128, attn_mma_smem<HD, kSplit>(cap), stream>>>(a);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

template <int HD, class T>
static int launch_attention(const AttnArgs& a, cudaStream_t stream) {
    const bool long_s = a.max_s > kAttnMaxS;     // some outfit may hold more than 16 items
    if constexpr (sizeof(T) == 2) {
        return long_s ? launch_attention_mma<HD, T, true>(a, stream) : launch_attention_mma<HD, T, false>(a, stream);
    } else {
        const int rows = a.row0_only ? a.batch : a.max_rows;
        const unsigned grid = static_cast<unsigned>((rows + 3) / 4);
        if (long_s) attention_kernel<HD, T, true><<<grid, 256, 0, stream>>>(a);
        else attention_kernel<HD, T, false><<<grid, 256, 0, stream>>>(a);
        OFX_LAUNCH_CHECK();
        return OFX_OK;
    }
}

template <class T>
int attention(const AttnArgs& a, int head_dim, cudaStream_t stream) {
    if (a.batch <= 0) return OFX_OK;
    if (a.n_head != 16) return fail(OFX_E_SHAPE, "attention: n_head %d != 16", a.n_head);
    if (a.max_s < 2 || a.max_s > kAttnLongMaxS) return fail(OFX_E_SHAPE, "attention: max_s %d not in [2,%d]", a.max_s, kAttnLongMaxS);
    // the mma kernels move 16-byte chunks of 8 elements: every row must start 16-byte aligned
    if (sizeof(T) == 2 && ((a.ldq % 8) || (a.ldk % 8) || (a.ldv % 8) || (a.ldo % 8)))
        return fail(OFX_E_ARG, "attention: 16-bit pitches must be multiples of 8 (q %lld, k %lld, v %lld, out %lld)",
                    a.ldq, a.ldk, a.ldv, a.ldo);
    switch (head_dim) {
        case 32: return launch_attention<32, T>(a, stream);
        case 64: return launch_attention<64, T>(a, stream);
        case 96: return launch_attention<96, T>(a, stream);
        default: return fail(OFX_E_SHAPE, "head_dim %d not in {32,64,96}", head_dim);
    }
}
template int attention<float>(const AttnArgs&, int, cudaStream_t);
template int attention<__nv_bfloat16>(const AttnArgs&, int, cudaStream_t);
template int attention<__half>(const AttnArgs&, int, cudaStream_t);

// ------------------------------------------------------------------ CP head: warp per outfit
__global__ void __launch_bounds__(256)
cp_head_kernel(const float* __restrict__ x0, int batch, int dm, const float* __restrict__ w,
               const float* __restrict__ bias, float* __restrict__ logits, float* __restrict__ probs) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= batch) return;
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int e = lane * 4; e < dm; e += 128) {
        float4 xv = *reinterpret_cast<const float4*>(x0 + static_cast<long long>(b) * dm + e);
        float4 wv = __ldg(reinterpret_cast<const float4*>(w + e));
        s += xv.x * wv.x + xv.y * wv.y + xv.z * wv.z + xv.w * wv.w;
    }
    s = warp_sum(s);
    if (lane == 0) {
        const float z = s + bias[0];
        logits[b] = z;
        if (probs) probs[b] = 1.f / (1.f + expf(-z));
    }
}
int cp_head(const float* x0, int batch, int dm, const float* w, const float* bias, float* logits,
            float* probs, cudaStream_t stream) {
    if (batch <= 0) return OFX_OK;
    cp_head_kernel<<<(batch + 7) / 8, 256, 0, stream>>>(x0, batch, dm, w, bias, logits, probs);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

// ------------------------------------------------------------------ FITB: warp per outfit
// d_j = || q - c_j ||_2 (direct differences, like torch.cdist for small inputs), argmin = first minimum
__global__ void __launch_bounds__(256)
fitb_kernel(const float* __restrict__ query, const float* __restrict__ cand, const int* __restrict__ cand_ids,
            long long n_cand_rows, int batch, int n_cand, int de, float* __restrict__ dist,
            long long* __restrict__ argmin) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= batch) return;
    const int lane = threadIdx.x & 31;
    float best = INFINITY;
    int best_j = 0;
    for (int j = 0; j < n_cand; ++j) {
        long long crow = static_cast<long long>(b) * n_cand + j;
        bool in_table = true;
        if (cand_ids) {
            crow = cand_ids[crow];
            in_table = crow >= 0 && crow < n_cand_rows;
            if (!in_table) crow = 0;
        }
        const float* c = cand + crow * de;
        float s = 0.f;
        for (int e = lane * 4; e < de; e += 128) {
            float4 qv = *reinterpret_cast<const float4*>(query + static_cast<long long>(b) * de + e);
            float4 cv = in_table ? *reinterpret_cast<const float4*>(c + e) : make_float4(0.f, 0.f, 0.f, 0.f);
            float d0 = qv.x - cv.x, d1 = qv.y - cv.y, d2 = qv.z - cv.z, d3 = qv.w - cv.w;
            s += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        }
        const float d = sqrtf(warp_sum(s));
        if (lane == 0 && dist) dist[static_cast<long long>(b) * n_cand + j] = d;
        if (d < best) { best = d; best_j = j; }
    }
    if (lane == 0 && argmin) argmin[b] = best_j;
}
int fitb(const float* query, const float* cand, const int* cand_ids, long long n_cand_rows, int batch,
         int n_cand, int de, float* dist, long long* argmin, cudaStream_t stream) {
    if (batch <= 0) return OFX_OK;
    fitb_kernel<<<(batch + 7) / 8, 256, 0, stream>>>(query, cand, cand_ids, n_cand_rows, batch, n_cand, de, dist,
                                                     argmin);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

// ------------------------------------------------------------------ weight packing
template <class T>
__global__ void pack_matrix_kernel(const float* __restrict__ src, int rows, int cols, T* __restrict__ dst,
                                   int prow, int pcol) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(prow) * pcol) return;
    const int r = static_cast<int>(i / pcol), c = static_cast<int>(i % pcol);
    dst[i] = from_f<T>((r < rows && c < cols) ? src[static_cast<long long>(r) * cols + c] : 0.f);
}
template <class T>
int pack_matrix(const float* src, int rows, int cols, T* dst, int prow, int pcol, cudaStream_t stream) {
    const long long n = static_cast<long long>(prow) * pcol;
    pack_matrix_kernel<T><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(src, rows, cols, dst, prow, pcol);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}
template int pack_matrix<float>(const float*, int, int, float*, int, int, cudaStream_t);
template int pack_matrix<__nv_bfloat16>(const float*, int, int, __nv_bfloat16*, int, int, cudaStream_t);
template int pack_matrix<__half>(const float*, int, int, __half*, int, int, cudaStream_t);

}  // namespace ofx
