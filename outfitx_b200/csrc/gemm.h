#pragma once
#include "common.h"

namespace ofx {

// C[m,n] = A[m,k] . W[n,k]^T  (+bias[n]) (mish) (+residual[m,n] fp32)
struct GemmArgs {
    const void* a;         // bf16 or fp16, row pitch lda elements
    long long lda;
    const void* w;         // same element type as a, row pitch ldw
    long long ldw;
    int m;                 // rows (host upper bound)
    const int* m_dev;      // optional device-side row count, <= m
    int n, k;
    const float* bias;
    int act_mish;
    const float* residual; // fp32, may alias out when out_f32
    long long ldr;
    void* out;             // 16-bit (the operand type) or fp32: out_f32 selects
    long long ldo;
    int out_f32;
};

int gemm_bf16(const GemmArgs& g, cudaStream_t stream);
// the same with fp16 a / w; a 16-bit output (out_f32 = 0) is fp16 and takes no residual
int gemm_f16(const GemmArgs& g, cudaStream_t stream);

// fp32 operands on the tensor cores: every fp32 value v is carried as two bf16 pieces hi = bf16(v), lo = bf16(v - hi)
// (16 mantissa bits), laid out along K as three blocks so that an ordinary bf16 GEMM with K' = 3K evaluates
//     A.W^T ~= A_hi.W_hi^T + A_lo.W_hi^T + A_hi.W_lo^T          (error ~2^-16 |a||w| per product, fp32 accumulation)
// activations: [hi | lo | hi] (kSplitA), weights: [hi | hi | lo] (kSplitW).  rows_dev: optional device-side row count.
constexpr int kSplitA = 0, kSplitW = 1;
int split_bf16x3(const float* src, long long ld, int rows, const int* rows_dev, int k, void* dst, int order,
                 cudaStream_t stream);
// g.a / g.w are the SPLIT operands (bf16, pitches 3K); g.k = K (unsplit); out_f32 = 1: fp32 output;
// out_f32 = 2: the output is written as the [hi | lo | hi] pieces of the next split GEMM's activation operand
// (bf16, ldo = 3 N, no residual)
int gemm_f32_split(const GemmArgs& g, cudaStream_t stream);

}  // namespace ofx
