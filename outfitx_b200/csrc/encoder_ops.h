#pragma once
#include "common.h"

namespace ofx {

struct AssembleArgs {
    int task, batch, max_items;
    const float* emb;      // (B,max_items,Dm) fused, or null
    const float* img;      // (B,max_items,dpm)
    const float* txt;
    int dpm, fuse_mode, normalize;
    const uint8_t* mask;   // (B,max_items) non-zero = pad
    const int* off;        // (B+1) exclusive prefix of valid counts
    const float* outfit_token;  // (Dm)
    const float* target_img;    // (Dm/2)
    const float* text;          // (B, Dm/2)
    const float* ln_w;          // LayerNorm 1 of layer 0 (fused here)
    const float* ln_b;
    int* owner;                 // out: (B + total items) token row -> outfit (item rows only)
    const int* item_ids;        // optional (B, max_items): img / txt are tables, slot -> table row
    long long n_table_rows;
};

struct AttnArgs {
    int batch, n_head, row0_only;
    int max_s;             // upper bound of tokens per outfit (1 + max_items, <= 65)
    int max_rows;          // host upper bound of token rows
    const int* n_tok;      // device token-row count
    const int* owner;      // token row -> outfit (rows >= batch)
    const int* off;
    const void* q; long long ldq;   // element pitches
    const void* k; long long ldk;
    const void* v; long long ldv;
    void* out; long long ldo;
};

// fused LN2 -> linear1 -> mish -> linear2 -> +residual on the fp32 residual stream (ffn_block.cu)
struct FfnBlockArgs {
    float* x;              // (rows, dm) fp32, updated in place
    int rows;              // host upper bound
    const int* rows_dev;   // optional device-side row count
    int dm, fp;            // d_model, padded d_ffn
    const float* ln_w;     // norm2
    const float* ln_b;
    const void* w1;        // (fp, dm) bf16 / fp16 (ffn_block_bf16 / ffn_block_f16)
    const float* b1;       // (fp)
    const void* w2;        // (dm, fp), the same type
    const float* b2;       // (dm)
    void* h_next = nullptr;        // optional (rows, dm), the same type: LayerNorm (lnn_w, lnn_b) of the updated x,
    const float* lnn_w = nullptr;  // i.e. norm1 of the next layer, emitted by the same kernel
    const float* lnn_b = nullptr;
    void* workspace = nullptr;     // at least ffn_block_workspace_bytes() (unused by the kernel)
    size_t workspace_bytes = 0;
};
bool ffn_block_supported(int dm, int fp);
size_t ffn_block_workspace_bytes();
int ffn_block_bf16(const FfnBlockArgs& a, cudaStream_t stream);
int ffn_block_f16(const FfnBlockArgs& a, cudaStream_t stream);

int scan_valid(const uint8_t* mask, int batch, int max_items, int* off, int* n_tok, cudaStream_t stream);
int fuse_rows(const float* img, const float* txt, long long rows, int dpm, int mode, int normalize,
              float* out, cudaStream_t stream);
template <class T> int assemble(const AssembleArgs& a, int dm, float* x, T* h, cudaStream_t stream);
template <class T> int layernorm(const float* x, int rows, const int* rows_dev, int dm, const float* gamma,
                                 const float* beta, T* out, cudaStream_t stream);
// LayerNorm written as the bf16 pieces [hi | lo | hi] (row pitch 3 dm) of a split-bf16 GEMM's activation operand
int layernorm_split3(const float* x, int rows, const int* rows_dev, int dm, const float* gamma, const float* beta,
                     void* out, cudaStream_t stream);
template <class T> int cast_rows(const float* in, long long n, T* out, cudaStream_t stream);
template <class T> int attention(const AttnArgs& a, int head_dim, cudaStream_t stream);
int cp_head(const float* x0, int batch, int dm, const float* w, const float* bias, float* logits,
            float* probs, cudaStream_t stream);
int fitb(const float* query, const float* cand, const int* cand_ids, long long n_cand_rows, int batch,
         int n_cand, int de, float* dist, long long* argmin, cudaStream_t stream);
template <class T> int pack_matrix(const float* src, int rows, int cols, T* dst, int prow, int pcol,
                                   cudaStream_t stream);

}  // namespace ofx
