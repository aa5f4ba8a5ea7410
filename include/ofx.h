/* libofx.so -- C ABI of the B200-native OutfitX outfit-scoring hot path (sm_100a).
 *
 * Every entry point below replaces a piece of the reference's Python path
 * (/root/reference, cited as file:line).  The reference has no FFI of its own: its "plugin
 * interface" for this path is the nn.Module API of src/models/outfit_x.py plus three caller
 * idioms in the trainers / demo.  outfitx_b200/model.py mirrors that Python API and binds
 * this library with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - plain pointers + sizes, no C++ / torch types; all data pointers are DEVICE pointers
 *    unless the name says host; tensors are dense row-major.
 *  - every call returns int: OFX_OK or a negative OFX_E_*; ofx_last_error() gives the
 *    thread-local message.  No exceptions, no exit().
 *  - all work is enqueued on the caller's CUDA stream (passed as void* = cudaStream_t);
 *    no hidden synchronisation, no allocation: scratch memory is a caller-provided
 *    workspace whose size is queried first.
 *  - there is no CPU fallback: without an sm_100 device every compute call fails with
 *    OFX_E_ARCH.
 */
#ifndef OFX_H_
#define OFX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFX_VERSION 100

#if defined(__GNUC__)
#define OFX_API __attribute__((visibility("default")))
#else
#define OFX_API
#endif

enum {
    OFX_OK = 0,
    OFX_E_SHAPE = -1,   /* unsupported / inconsistent shape                    */
    OFX_E_ARG = -2,     /* null or misaligned pointer, bad enum value          */
    OFX_E_ARCH = -3,    /* no CUDA device of compute capability 10.x            */
    OFX_E_CUDA = -4,    /* a CUDA runtime / driver call failed                  */
    OFX_E_WORKSPACE = -5 /* workspace too small                                 */
};

/* arithmetic of the hot GEMMs */
enum {
    OFX_PREC_BF16 = 0, /* bf16 operands on tcgen05 tensor cores, fp32 accumulate (TMEM)   */
    OFX_PREC_FP32 = 1, /* fp32 (split-bf16 tensor-core GEMMs): the <=1e-3-relative parity mode */
    OFX_PREC_FP16 = 2  /* fp16 operands, fp32 accumulate: the arithmetic of the reference's
                        * evaluation under torch.autocast(float16).  The residual stream,
                        * LayerNorm / softmax statistics and the heads stay fp32 as in bf16 mode;
                        * an operand outside the fp16 range (|v| > 65504) overflows to inf, as it
                        * does under autocast -- nothing is clamped.  Packed weights and workspace
                        * have the bf16 sizes. */
};

enum { OFX_TASK_CP = 0, OFX_TASK_CIR = 1 }; /* FITB uses the CIR task (outfit_x.py:86-87) */
enum { OFX_FUSE_CONCAT = 0, OFX_FUSE_MEAN = 1 };
enum { OFX_METRIC_DOT = 0, OFX_METRIC_L2 = 1 };

/* Model dimensions: OutfitXConfig / TransformerConfig
 * (src/models/configs/outfit_x_config.py:8-30, transformer_config.py:7-23). */
typedef struct ofx_shape {
    int32_t d_model;   /* 512 (clip+mean), 1024 (clip+concat) or 1536 (slip+concat)         */
    int32_t d_embed;   /* cir_ffn output = 2*dim_per_modality (outfit_x_config.py:23)        */
    int32_t n_head;    /* 16                                                                */
    int32_t n_layers;  /* 6                                                                 */
    int32_t d_ffn;     /* 2024 (zero-padded to a multiple of 64 inside the packed weights)  */
    int32_t max_items; /* item slots per outfit, 1..64; the reference default is 16         */
                       /* (max_length, outfit_x_config.py:13)                               */
    int32_t precision; /* OFX_PREC_*                                                        */
} ofx_shape;

/* Order of the fp32 parameter pointers handed to ofx_pack_weights: per layer
 * OFX_W_PER_LAYER tensors in this order, then the OFX_W_GLOBAL model-level ones
 * (state_dict keys of src/models/outfit_x.py:32-71; SURVEY.md App. C). */
enum {
    OFX_W_IN_PROJ_W = 0, /* self_attn.in_proj_weight (3Dm, Dm) */
    OFX_W_IN_PROJ_B,     /* self_attn.in_proj_bias   (3Dm)     */
    OFX_W_OUT_PROJ_W,    /* self_attn.out_proj.weight (Dm, Dm) */
    OFX_W_OUT_PROJ_B,    /* self_attn.out_proj.bias  (Dm)      */
    OFX_W_LINEAR1_W,     /* linear1.weight (F, Dm)             */
    OFX_W_LINEAR1_B,     /* linear1.bias   (F)                 */
    OFX_W_LINEAR2_W,     /* linear2.weight (Dm, F)             */
    OFX_W_LINEAR2_B,     /* linear2.bias   (Dm)                */
    OFX_W_NORM1_W,
    OFX_W_NORM1_B,
    OFX_W_NORM2_W,
    OFX_W_NORM2_B,
    OFX_W_PER_LAYER
};
enum {
    OFX_G_OUTFIT_TOKEN = 0, /* outfit_token (Dm)             outfit_x.py:53-55 */
    OFX_G_TARGET_IMG,       /* target_item_image_emb (Dm/2)  outfit_x.py:69-71 */
    OFX_G_CP_W,             /* cp_ffn.1.weight (1, Dm)       outfit_x.py:57-61 */
    OFX_G_CP_B,             /* cp_ffn.1.bias (1)                               */
    OFX_G_CIR_W,            /* cir_ffn.0.weight (De, Dm)     outfit_x.py:65-67 */
    OFX_W_GLOBAL
};

OFX_API int ofx_version(void);
OFX_API const char* ofx_last_error(void);
/* number of CUDA kernels this library has launched in this process (all threads) */
OFX_API int64_t ofx_launch_count(void);
/* 0 when cuda device `device` has compute capability 10.x, else OFX_E_ARCH */
OFX_API int ofx_device_ok(int device);

/* ---- weights: replaces nn.Module parameter storage + load_state_dict (demo/app.py:102-103) */
OFX_API size_t ofx_packed_weights_bytes(const ofx_shape* shape);
/* params: HOST array of n_layers*OFX_W_PER_LAYER + OFX_W_GLOBAL DEVICE fp32 pointers */
OFX_API int ofx_pack_weights(const ofx_shape* shape, const float* const* params, void* packed,
                     void* stream);

/* ---- fusion: F.normalize per modality + aggregate_embeddings
 * (src/models/encoders/image/base_image_encoder.py:46-47, text/base_text_encoder.py:37-38,
 *  src/utils/model_utils.py:26-45).  img, txt: (rows, dpm) fp32 -> out (rows, 2*dpm | dpm). */
OFX_API int ofx_fuse(const float* img, const float* txt, int64_t rows, int32_t dpm, int32_t mode,
             int32_t normalize, float* out, void* stream);

/* ---- encoder forward: OutfitX._cp_forward / _cir_forward (outfit_x.py:120-172) plus the
 * caller idioms sigmoid (compatibility_prediction_trainer.py:408) and FITB cdist->argmin
 * (fill_in_the_blank_trainer.py:50-53).
 *
 * Inputs: either `emb` (B, max_items, Dm) fused fp32 embeddings (the reference's outfit_embedding),
 * or raw modalities img/txt (B, max_items, dpm) fused on the fly (fuse_mode, normalize) with
 * emb == NULL.  mask (B, max_items) bytes, non-zero = padding (outfit_mask, True = pad).  Valid
 * items may sit in any slot; padded slots are never read. */
typedef struct ofx_forward_args {
    int32_t task;          /* OFX_TASK_*                                              */
    int32_t batch;         /* B outfits                                               */
    const float* emb;      /* (B, max_items, Dm) or NULL                              */
    const float* img;      /* (B, max_items, dpm) or NULL                             */
    const float* txt;      /* (B, max_items, dpm) or NULL                             */
    int32_t fuse_mode;     /* OFX_FUSE_* (used with img/txt)                          */
    int32_t normalize;     /* L2-normalise each modality first (reference: yes)       */
    const uint8_t* mask;   /* (B, max_items)                                          */
    const float* text;     /* CIR: target_item_text_embedding (B, Dm/2)               */
    float* logits;         /* CP out: (B) logits  (== reference (B,1))                */
    float* probs;          /* CP out: (B) sigmoid(logit), may be NULL                 */
    float* query;          /* CIR out: (B, De) query embeddings                       */
    const float* cand;     /* FITB: (B, n_cand, De) candidates or NULL                */
    int32_t n_cand;        /* 4 in the reference                                      */
    float* fitb_dist;      /* FITB out: (B, n_cand) L2 distances, may be NULL         */
    int64_t* fitb_argmin;  /* FITB out: (B) first-minimum index                       */
    /* Device-side collate (replaces the per-batch gather + pad of the reference's processors,
     * src/models/processor/outfit_x/outfit_x_base_processor.py:20-81): when item_ids != NULL,
     * img / txt are TABLES (n_table_rows, dpm) resident in HBM and slot (b, s) reads row
     * item_ids[b * max_items + s]; ids of padded slots are ignored, ids outside the table read
     * as zero rows.  Likewise cand is a table (n_cand_rows, De) when cand_ids != NULL.        */
    const int32_t* item_ids;   /* (B, max_items) or NULL                              */
    int64_t n_table_rows;
    const int32_t* cand_ids;   /* (B, n_cand) or NULL                                 */
    int64_t n_cand_rows;
} ofx_forward_args;

OFX_API size_t ofx_encoder_workspace_bytes(const ofx_shape* shape, int32_t batch);
OFX_API int ofx_encoder_forward(const ofx_shape* shape, const void* packed_weights,
                        const ofx_forward_args* args, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- CIR search: torch.cdist -> torch.topk(largest=False)
 * (complementary_item_retrieval_trainer.py:240-242, demo/app.py:189-190), restated as the
 * arg-max of  q.g - 0.5|g|^2  (OFX_METRIC_L2, same ranking as ascending L2 distance) or of
 * q.g (OFX_METRIC_DOT); ties are broken by the lowest gallery index. */
OFX_API size_t ofx_gallery_packed_bytes(int64_t n_rows, int32_t dim);
/* gallery (n_rows, dim) fp32 -> packed bf16 rows of dim + 64 columns (the extra k-block carries
 * -0.5|g|^2 as bf16 hi + lo, so the L2 bias is part of the contraction) + fp32 0.5|g|^2 per row + its
 * maximum over the shard (used by the exactness certificate) */
OFX_API int ofx_gallery_pack(const float* gallery, int64_t n_rows, int32_t dim, void* packed,
                     void* stream);
OFX_API size_t ofx_search_workspace_bytes(int64_t n_rows, int32_t dim, int32_t n_query, int32_t k);
/* Exact top-k (k <= 64) of every query over this shard's rows.  Candidates come from a bf16 tcgen05
 * pass with a fused per-row top-k' selection (the score matrix never reaches HBM); they are
 * re-scored in fp64 from the fp32 gallery and ranked by (-score, index).  out_idx carries
 * GLOBAL ids (id_offset + local row); slots beyond n_rows get idx -1 / score -inf.
 * out_certified (n_query bytes, may be NULL): 1 = PROVEN equal to the exhaustive fp64 result -- the k-th
 * best exact score clears every score the bf16 pass may have dropped by a rigorous bound on the bf16
 * error (|q| max|g| (2^-8 + ...)); candidates inside that band are re-scored as well.  0 = not proven
 * (gallery rows closer to each other than bf16 resolves, more of them than the lists hold): run
 * ofx_exact_search on those queries.  Always 0 when gallery_f32 == NULL (bf16 ranking requested). */
OFX_API int ofx_topk_search(const void* packed, const float* gallery_f32, int64_t n_rows, int32_t dim,
                    int64_t id_offset, const float* queries, int32_t n_query, int32_t k,
                    int32_t metric, double* out_score, int64_t* out_idx, uint8_t* out_certified,
                    void* workspace, size_t workspace_bytes, void* stream);
/* Exhaustive fp64 search of the n_sel queries listed in sel (device int32 query indices): the fallback for
 * uncertified queries.  Rows sel[i] of out_score / out_idx (n_query, k) are overwritten (and out_certified[sel[i]]
 * set to 1 when given); cost is one pass over the fp32 gallery per 8 selected queries. */
OFX_API size_t ofx_exact_search_workspace_bytes(int64_t n_rows, int32_t n_sel, int32_t k);
OFX_API int ofx_exact_search(const float* gallery_f32, int64_t n_rows, int32_t dim, int64_t id_offset,
                     const float* queries, const int32_t* sel, int32_t n_sel, int32_t k, int32_t metric,
                     double* out_score, int64_t* out_idx, uint8_t* out_certified, void* workspace,
                     size_t workspace_bytes, void* stream);
/* Merge R per-shard lists (R, nq, k) by (-score, idx) into (nq, k): the step after the NCCL
 * all-gather of the gallery-sharded search (no reference counterpart: its inference is
 * single-GPU, complementary_item_retrieval_trainer.py:350-351). */
OFX_API int ofx_topk_merge(const double* scores, const int64_t* idx, int32_t n_lists, int32_t n_query,
                   int32_t k, double* out_score, int64_t* out_idx, void* stream);

/* ---- category-restricted search over a whole gallery shard: the reference ranks a CIR query only against
 * the items of its target category (compute_recall_metrics, complementary_item_retrieval_trainer.py:192-249;
 * demo/app.py:182-190).  Same arithmetic, ranking, exactness certificate and sharding as ofx_topk_search, but
 * the exact top-k of each query is taken over the shard's rows of the query's category only.
 *
 * Packing: categories (n_rows) int32 ids in [0, n_categories), n_categories <= 65536 (empty categories are
 * fine; a row with an id outside the range belongs to no category and is never returned).  The shard is sorted
 * stably by category: packed row p holds gallery row perm[p], category c is packed rows
 * [seg_off[c], seg_off[c+1]), so within a category packed order is the original order.  Outputs: packed
 * (ofx_category_gallery_packed_bytes: the bf16 rows of ofx_gallery_pack in packed order, then scratch of the
 * sort), perm (n_rows) int32, seg_off (n_categories + 1) int64, cat_max_half_sqnorm (n_categories) fp32 =
 * max 0.5|g|^2 of each category, for the certificate.  The fp32 rows stay in the caller's order: the re-rank
 * and the fallback read them through perm. */
OFX_API size_t ofx_category_gallery_packed_bytes(int64_t n_rows, int32_t dim, int32_t n_categories);
OFX_API int ofx_category_gallery_pack(const float* gallery, const int32_t* categories, int64_t n_rows, int32_t dim,
                              int32_t n_categories, void* packed, int32_t* perm, int64_t* seg_off,
                              float* cat_max_half_sqnorm, void* stream);
/* workspace for any distribution of the n_query query categories */
OFX_API size_t ofx_category_search_workspace_bytes(int32_t dim, int32_t n_categories, int32_t n_query, int32_t k);
/* Exact top-k of every query over this shard's rows of category query_category[q] (n_query int32, device).
 * Outputs as ofx_topk_search: GLOBAL ids id_offset + perm[p], ties to the lowest id, idx -1 / score -inf past
 * the category's rows; a query whose category has no row here, or is out of range, gets padding only (and
 * out_certified 1).  out_certified 0: run ofx_category_exact_search on those queries.  The work list is built
 * on the device: no synchronisation, capturable in a CUDA graph. */
OFX_API int ofx_category_search(const void* packed, const int32_t* perm, const int64_t* seg_off,
                        const float* cat_max_half_sqnorm, int32_t n_categories, const float* gallery_f32,
                        int64_t n_rows, int32_t dim, int64_t id_offset, const float* queries,
                        const int32_t* query_category, int32_t n_query, int32_t k, int32_t metric,
                        double* out_score, int64_t* out_idx, uint8_t* out_certified, void* workspace,
                        size_t workspace_bytes, void* stream);
/* ofx_exact_search restricted to each selected query's category segment (cost proportional to the segment);
 * workspace: ofx_exact_search_workspace_bytes(n_rows, n_sel, k). */
OFX_API int ofx_category_exact_search(const float* gallery_f32, const int32_t* perm, const int64_t* seg_off,
                              int32_t n_categories, int64_t n_rows, int32_t dim, int64_t id_offset,
                              const float* queries, const int32_t* query_category, const int32_t* sel,
                              int32_t n_sel, int32_t k, int32_t metric, double* out_score, int64_t* out_idx,
                              uint8_t* out_certified, void* workspace, size_t workspace_bytes, void* stream);

/* ---- per-category candidate pools (SURVEY.md N1): the retrieval evaluation of
 * complementary_item_retrieval_trainer.py:192-249 ranks every query against the pool of its target
 * category only (<= 3000 items, polyvore_complementary_item_retrieval_dataset.py:111-153) with
 * cdist -> topk(50, largest=False).  pools: all pools concatenated, (total_rows, dim) fp32;
 * pool_offsets (n_pools + 1) row offsets (device); query_pool (n_query) pool index of each query
 * (device).  Exact fp64 scores, ties to the lowest index; out_idx (n_query, k) are POOL-LOCAL row
 * indices (-1 past the pool size), k <= 64, pools of at most 4096 rows. */
OFX_API int ofx_pool_search(const float* pools, const int64_t* pool_offsets, int32_t n_pools,
                    int32_t max_pool_rows, const float* queries, const int32_t* query_pool,
                    int32_t n_query, int32_t dim, int32_t k, int32_t metric, double* out_score,
                    int64_t* out_idx, void* stream);

/* ---- evaluation-side scoring (SURVEY.md N4), forward only.  Scalars come back in fp64 device
 * memory; reductions are two-stage in a fixed order (deterministic). */
OFX_API size_t ofx_loss_workspace_bytes(int64_t batch);
/* FocalLoss.forward (src/losses/focal_loss.py:23-41): logits, labels (n) fp32 (labels as floats, as
 * the trainer passes them).  per_elem (n) receives the reduction='none' tensor (may be NULL);
 * out[0] = sum, out[1] = mean.  alpha < 0 skips the alpha_t weighting (focal_loss.py:31). */
OFX_API int ofx_focal_loss(const float* logits, const float* labels, int64_t n, float gamma, float alpha,
                   float* per_elem, double* out, void* workspace, size_t workspace_bytes,
                   void* stream);
/* SetWiseRankingLoss.forward (src/losses/set_wise_ranking_loss.py:14-37): y, y_hat (B, dim);
 * negatives (B, n_neg, dim); negative_mask (B, n_neg) bytes, non-zero = padding.
 * out[0] = L_all + L_hard, out[1] = L_all, out[2] = L_hard. */
OFX_API int ofx_set_wise_ranking_loss(const float* y, const float* y_hat, const float* negatives,
                              const uint8_t* negative_mask, int32_t batch, int32_t n_neg,
                              int32_t dim, float margin, double* out, void* workspace,
                              size_t workspace_bytes, void* stream);
/* compute_cp_metrics (src/trains/trainers/compatibility_prediction_trainer.py:406-436):
 * probs (n) <- sigmoid(logits); counts[0..5] = TP, FP, FN, #correct, #positive, #negative at the
 * 0.5 threshold; counts[6] = 2 #{pos i, neg j: p_j < p_i} + #{p_j == p_i}, so that
 * AUC = counts[6] / (2 counts[4] counts[5]) is sklearn's roc_auc_score (ties count 1/2). n <= 2^22. */
OFX_API int ofx_cp_metrics(const float* logits, const float* labels, int64_t n, float* probs,
                   int64_t* counts, void* stream);

/* ---- building block exported for tests / profiling: C = A . W^T (+bias)(+mish)(+residual)
 * A (M,K) bf16 pitch lda, W (N,K) bf16 pitch ldw on the tcgen05 pipeline.  out is bf16 or
 * fp32 (out_f32), pitch ldo; residual fp32 pitch ldr or NULL.  N % 128 == 0, K % 64 == 0. */
OFX_API int ofx_gemm_bf16(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t m, int32_t n,
                  int32_t k, const float* bias, int32_t act_mish, const float* residual,
                  int64_t ldr, void* out, int64_t ldo, int32_t out_f32, void* stream);
/* The same with fp16 A and W (the linear layers of precision OFX_PREC_FP16).  out_f32 = 0 writes fp16 and takes no
 * residual (OFX_E_ARG); out_f32 = 1 writes fp32 with or without the fp32 residual.  Results outside the fp16 range
 * overflow to inf, as under the reference's autocast; nothing is clamped. */
OFX_API int ofx_gemm_f16(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t m, int32_t n,
                 int32_t k, const float* bias, int32_t act_mish, const float* residual,
                 int64_t ldr, void* out, int64_t ldo, int32_t out_f32, void* stream);

/* ---- the fp32 mode's linear layer (the nn.Linear / F.linear calls inside the nn.TransformerEncoderLayer stack of
 * src/models/outfit_x.py:32-45 and the CIR head :62-66 when the model runs without autocast) on the tensor cores:
 * fp32 A (M,K) and W (N,K) are cut into bf16 hi / lo pieces
 * (16 mantissa bits) and  A.W^T ~= A_hi.W_hi^T + A_lo.W_hi^T + A_hi.W_lo^T  runs as ONE bf16 tcgen05 GEMM with K' = 3K
 * and fp32 accumulation (relative error ~2^-16 instead of bf16's 2^-8); out fp32.  What precision="fp32" of
 * ofx_encoder_forward uses for every nn.Linear (weights are split once by ofx_pack_weights).  K % 64 == 0,
 * N % 128 == 0.  workspace: ofx_gemm_f32_tc_workspace_bytes(m, n, k) bytes, 256-byte aligned. */
OFX_API size_t ofx_gemm_f32_tc_workspace_bytes(int32_t m, int32_t n, int32_t k);
OFX_API int ofx_gemm_f32_tc(const float* a, int64_t lda, const float* w, int64_t ldw, int32_t m, int32_t n, int32_t k,
                    const float* bias, int32_t act_mish, const float* residual, int64_t ldr, float* out,
                    int64_t ldo, void* workspace, size_t workspace_bytes, void* stream);

/* ---- building block exported for tests / profiling: the fused feed-forward block of one
 * encoder layer,  x <- x + W2 . mish(W1 . LayerNorm(x) + b1) + b2  in place on the fp32 rows
 * (torch TransformerEncoderLayer._ff_block as configured at outfit_x.py:32-45).
 * x (rows, d_model) fp32; w1 (d_ffn_padded, d_model) bf16; w2 (d_model, d_ffn_padded) bf16;
 * b1 (d_ffn_padded), b2 / ln_w / ln_b (d_model) fp32.  d_model == 512, d_ffn_padded % 256 == 0. */
OFX_API size_t ofx_ffn_block_workspace_bytes(int32_t rows, int32_t d_model, int32_t d_ffn_padded);
OFX_API int ofx_ffn_block_bf16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded,
                       const float* ln_w, const float* ln_b, const void* w1, const float* b1,
                       const void* w2, const float* b2, void* workspace, size_t workspace_bytes,
                       void* stream);

/* Same block, and in the same kernel h_next (rows, d_model) bf16 <- LayerNorm(x_new; next_ln_w,
 * next_ln_b): norm1 of the FOLLOWING encoder layer (transformer.py:944-947), computed by otherwise idle
 * warps from the rows the block has just written, so the inter-layer LayerNorm kernel disappears.
 * workspace: at least ofx_ffn_block_workspace_bytes bytes, required by both entries (a smaller one fails with
 * OFX_E_WORKSPACE); the kernel keeps nothing in it. */
OFX_API int ofx_ffn_block_ln_bf16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded,
                          const float* ln_w, const float* ln_b, const void* w1, const float* b1,
                          const void* w2, const float* b2, void* h_next, const float* next_ln_w,
                          const float* next_ln_b, void* workspace, size_t workspace_bytes, void* stream);

/* The fp16 form of both (precision OFX_PREC_FP16): w1 / w2 fp16, LayerNorm output, hidden activation and h_next
 * rounded to fp16, fp32 accumulation and residual stream.  h_next (rows, d_model) fp16 may be NULL: the plain block
 * (next_ln_w / next_ln_b are then ignored).  Same shapes and workspace rule as ofx_ffn_block_bf16.  Values outside
 * the fp16 range overflow to inf, as under the reference's autocast; nothing is clamped. */
OFX_API int ofx_ffn_block_f16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded,
                      const float* ln_w, const float* ln_b, const void* w1, const float* b1,
                      const void* w2, const float* b2, void* h_next, const float* next_ln_w,
                      const float* next_ln_b, void* workspace, size_t workspace_bytes, void* stream);

/* ---- building block exported for tests / profiling: the masked multi-head self-attention of one encoder layer
 * (softmax(q.K^T / sqrt(head_dim)) . V per outfit and head, padded slots dropped), launched exactly as
 * ofx_encoder_forward launches it.
 * Packed token layout: row b < batch is outfit b's prefix token; its items are rows batch + off[b] ..
 * batch + off[b+1] - 1, and owner[r] is the outfit of item row r; *n_tok == batch + off[batch].  off (batch + 1),
 * owner (at least *n_tok) and n_tok are int32 device arrays supplied by the caller.  An outfit attends over its
 * S = 1 + off[b+1] - off[b] tokens.
 * Elements are bf16, fp16 or fp32 after `precision` (OFX_PREC_*); 16 heads of d_model / 16 consecutive columns.
 * q, k, v and out hold rows of pitch ldq, ldk, ldv, ldo elements; out receives every token row, or with
 * row0_only = 1 (the pruned last layer) only rows 0 .. batch - 1, whose queries are then rows 0 .. batch - 1
 * of q.  Nothing else of out is written.
 * Refused before anything is launched: precision not an OFX_PREC_* (OFX_E_ARG); d_model not 512 / 1024 / 1536,
 * max_items not in 1..64, batch < 0 or above the encoder's bound 2^26 / (max_items + 1) (OFX_E_SHAPE); a null or
 * not 16-byte aligned pointer, row0_only not 0 / 1, a pitch below d_model or not a multiple of 8 elements for
 * bf16 / fp16 or of 4 for fp32 (OFX_E_ARG). */
OFX_API int ofx_attention(int32_t precision, int32_t d_model, int32_t batch, int32_t max_items,
                          const int32_t* off, const int32_t* owner, const int32_t* n_tok, int32_t row0_only,
                          const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                          void* out, int64_t ldo, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OFX_H_ */
