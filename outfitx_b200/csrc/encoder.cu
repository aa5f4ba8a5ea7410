// Encoder forward of the outfit-scoring path behind the C ABI:
//   ofx_pack_weights / ofx_encoder_forward / ofx_fuse / ofx_gemm_bf16 / ofx_gemm_f16 / ofx_attention.
// Mirrors OutfitX._cp_forward / _cir_forward (/root/reference/src/models/outfit_x.py:120-172)
// with the exact simplifications of SURVEY.md App. A.4: padded tokens dropped, last layer
// evaluated for the prefix-token query row only.

#include "encoder_ops.h"
#include "gemm.h"

namespace ofx {

static int round_up(int x, int a) { return (x + a - 1) / a * a; }

struct WLayout {
    int dm, de, f, fp, nl;
    size_t esz;
    size_t w_qkv, w_o, w_1, w_2, b_qkv, b_o, b_1, b_2, ln1w, ln1b, ln2w, ln2b, layer_bytes;
    size_t g_token, g_timg, g_cpw, g_cpb, g_cir, total;
    // fp32 precision only: the GEMM weights once more as bf16 hi / lo pieces [hi | hi | lo] along K (gemm.h), so that
    // the fp32 mode's linear layers run on the tensor cores (0 = absent)
    size_t s_qkv, s_o, s_1, s_2, s_cir;
};

static int check_shape(const ofx_shape* s) {
    if (!s) return fail(OFX_E_ARG, "shape is null");
    if (s->d_model != 512 && s->d_model != 1024 && s->d_model != 1536)
        return fail(OFX_E_SHAPE, "d_model %d not in {512,1024,1536}", s->d_model);
    if (s->n_head != 16) return fail(OFX_E_SHAPE, "n_head %d != 16", s->n_head);
    if (s->n_layers < 1 || s->n_layers > 64) return fail(OFX_E_SHAPE, "n_layers %d", s->n_layers);
    if (s->d_ffn < 1 || s->d_ffn > 16384) return fail(OFX_E_SHAPE, "d_ffn %d", s->d_ffn);
    if (s->d_embed < 128 || s->d_embed % 128) return fail(OFX_E_SHAPE, "d_embed %d must be a multiple of 128", s->d_embed);
    if (s->max_items < 1 || s->max_items > 64) return fail(OFX_E_SHAPE, "max_items %d not in [1,64]", s->max_items);
    if (s->precision != OFX_PREC_BF16 && s->precision != OFX_PREC_FP32 && s->precision != OFX_PREC_FP16)
        return fail(OFX_E_ARG, "precision %d not in {0 (bf16), 1 (fp32), 2 (fp16)}", s->precision);
    return OFX_OK;
}

static WLayout make_layout(const ofx_shape* s) {
    WLayout L{};
    L.dm = s->d_model; L.de = s->d_embed; L.f = s->d_ffn; L.fp = round_up(s->d_ffn, 128); L.nl = s->n_layers;
    L.esz = s->precision == OFX_PREC_FP32 ? 4 : 2;     // bf16 and fp16: 2-byte matrices
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    const size_t dm = L.dm, fp = L.fp;
    L.w_qkv = take(3 * dm * dm * L.esz);
    L.w_o = take(dm * dm * L.esz);
    L.w_1 = take(fp * dm * L.esz);
    L.w_2 = take(dm * fp * L.esz);
    L.b_qkv = take(3 * dm * 4);
    L.b_o = take(dm * 4);
    L.b_1 = take(fp * 4);
    L.b_2 = take(dm * 4);
    L.ln1w = take(dm * 4); L.ln1b = take(dm * 4); L.ln2w = take(dm * 4); L.ln2b = take(dm * 4);
    if (s->precision == OFX_PREC_FP32) {
        L.s_qkv = take(3 * dm * 3 * dm * 2);
        L.s_o = take(dm * 3 * dm * 2);
        L.s_1 = take(fp * 3 * dm * 2);
        L.s_2 = take(dm * 3 * fp * 2);
    }
    L.layer_bytes = o;
    o = L.layer_bytes * L.nl;
    L.g_token = take(dm * 4);
    L.g_timg = take(dm / 2 * 4);
    L.g_cpw = take(dm * 4);
    L.g_cpb = take(256);
    L.g_cir = take(static_cast<size_t>(L.de) * dm * L.esz);
    if (s->precision == OFX_PREC_FP32) L.s_cir = take(static_cast<size_t>(L.de) * 3 * dm * 2);
    L.total = o;
    return L;
}

template <class T>
static int pack_all(const WLayout& L, const float* const* p, uint8_t* dst, cudaStream_t st) {
    for (int l = 0; l < L.nl; ++l) {
        const float* const* q = p + l * OFX_W_PER_LAYER;
        uint8_t* base = dst + L.layer_bytes * l;
        for (int i = 0; i < OFX_W_PER_LAYER; ++i)
            if (!q[i]) return fail(OFX_E_ARG, "ofx_pack_weights: layer %d tensor %d is null", l, i);
        OFX_TRY(pack_matrix<T>(q[OFX_W_IN_PROJ_W], 3 * L.dm, L.dm, reinterpret_cast<T*>(base + L.w_qkv), 3 * L.dm, L.dm, st));
        OFX_TRY(pack_matrix<T>(q[OFX_W_OUT_PROJ_W], L.dm, L.dm, reinterpret_cast<T*>(base + L.w_o), L.dm, L.dm, st));
        // d_ffn 2024 -> 2048: zero rows of W1 / zero bias give mish(0) = 0, zero columns of W2
        OFX_TRY(pack_matrix<T>(q[OFX_W_LINEAR1_W], L.f, L.dm, reinterpret_cast<T*>(base + L.w_1), L.fp, L.dm, st));
        OFX_TRY(pack_matrix<T>(q[OFX_W_LINEAR2_W], L.dm, L.f, reinterpret_cast<T*>(base + L.w_2), L.dm, L.fp, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_IN_PROJ_B], 1, 3 * L.dm, reinterpret_cast<float*>(base + L.b_qkv), 1, 3 * L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_OUT_PROJ_B], 1, L.dm, reinterpret_cast<float*>(base + L.b_o), 1, L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_LINEAR1_B], 1, L.f, reinterpret_cast<float*>(base + L.b_1), 1, L.fp, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_LINEAR2_B], 1, L.dm, reinterpret_cast<float*>(base + L.b_2), 1, L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_NORM1_W], 1, L.dm, reinterpret_cast<float*>(base + L.ln1w), 1, L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_NORM1_B], 1, L.dm, reinterpret_cast<float*>(base + L.ln1b), 1, L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_NORM2_W], 1, L.dm, reinterpret_cast<float*>(base + L.ln2w), 1, L.dm, st));
        OFX_TRY(pack_matrix<float>(q[OFX_W_NORM2_B], 1, L.dm, reinterpret_cast<float*>(base + L.ln2b), 1, L.dm, st));
        if (sizeof(T) == 4 && L.s_qkv) {     // the packed (padded) fp32 matrices -> bf16 hi / lo pieces
            auto f = [&](size_t o) { return reinterpret_cast<const float*>(base + o); };
            OFX_TRY(split_bf16x3(f(L.w_qkv), L.dm, 3 * L.dm, nullptr, L.dm, base + L.s_qkv, kSplitW, st));
            OFX_TRY(split_bf16x3(f(L.w_o), L.dm, L.dm, nullptr, L.dm, base + L.s_o, kSplitW, st));
            OFX_TRY(split_bf16x3(f(L.w_1), L.dm, L.fp, nullptr, L.dm, base + L.s_1, kSplitW, st));
            OFX_TRY(split_bf16x3(f(L.w_2), L.fp, L.dm, nullptr, L.fp, base + L.s_2, kSplitW, st));
        }
    }
    const float* const* g = p + L.nl * OFX_W_PER_LAYER;
    for (int i = 0; i < OFX_W_GLOBAL; ++i)
        if (!g[i]) return fail(OFX_E_ARG, "ofx_pack_weights: model-level tensor %d is null", i);
    OFX_TRY(pack_matrix<float>(g[OFX_G_OUTFIT_TOKEN], 1, L.dm, reinterpret_cast<float*>(dst + L.g_token), 1, L.dm, st));
    OFX_TRY(pack_matrix<float>(g[OFX_G_TARGET_IMG], 1, L.dm / 2, reinterpret_cast<float*>(dst + L.g_timg), 1, L.dm / 2, st));
    OFX_TRY(pack_matrix<float>(g[OFX_G_CP_W], 1, L.dm, reinterpret_cast<float*>(dst + L.g_cpw), 1, L.dm, st));
    OFX_TRY(pack_matrix<float>(g[OFX_G_CP_B], 1, 1, reinterpret_cast<float*>(dst + L.g_cpb), 1, 1, st));
    OFX_TRY(pack_matrix<T>(g[OFX_G_CIR_W], L.de, L.dm, reinterpret_cast<T*>(dst + L.g_cir), L.de, L.dm, st));
    if (sizeof(T) == 4 && L.s_cir)
        OFX_TRY(split_bf16x3(reinterpret_cast<const float*>(dst + L.g_cir), L.dm, L.de, nullptr, L.dm, dst + L.s_cir, kSplitW, st));
    return OFX_OK;
}

// workspace carve-up (all 256-byte aligned)
struct WsLayout {
    size_t off, n_tok, owner, x, h, big, q0, a0, u0, ffn, ffn_bytes, split, total;
    int t_max, big_ld;
};
static WsLayout make_ws(const ofx_shape* s, int batch) {
    WsLayout W{};
    const size_t esz = s->precision == OFX_PREC_FP32 ? 4 : 2;
    const size_t dm = s->d_model, fp = round_up(s->d_ffn, 128);
    W.t_max = batch * (s->max_items + 1);
    W.big_ld = static_cast<int>(3 * dm > fp ? 3 * dm : fp);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    const size_t t = static_cast<size_t>(W.t_max);
    W.off = take((static_cast<size_t>(batch) + 1) * 4);
    W.n_tok = take(4);
    W.owner = take(t * 4);
    W.x = take(t * dm * 4);
    W.h = take(t * dm * esz);
    // fp32 precision: `big` / `u0` also hold the hidden activation as bf16 pieces (3 x fp bf16 per row, gemm.h)
    const size_t big_row = s->precision == OFX_PREC_FP32 ? (W.big_ld * esz > 6 * fp ? W.big_ld * esz : 6 * fp) : W.big_ld * esz;
    W.big = take(t * big_row);
    W.q0 = take(static_cast<size_t>(batch) * dm * esz);
    W.a0 = take(static_cast<size_t>(batch) * dm * esz);
    W.u0 = take(static_cast<size_t>(batch) * fp * (s->precision == OFX_PREC_FP32 ? 6 : esz));
    // the fused FFN block's workspace (bf16 / fp16 path, d_model 512; the kernel itself uses none of it)
    W.ffn_bytes = (s->precision != OFX_PREC_FP32 && ffn_block_supported(s->d_model, static_cast<int>(fp))) ? ffn_block_workspace_bytes() : 0;
    W.ffn = take(W.ffn_bytes);
    // fp32 precision: bf16 hi / lo pieces of the current GEMM's activation operand (3 x K bf16 per token row)
    W.split = take(s->precision == OFX_PREC_FP32 ? t * 3 * (dm > fp ? dm : fp) * 2 : 0);
    W.total = o;
    return W;
}

// the 16-bit building blocks for operand type T (__nv_bfloat16 or __half)
template <class T>
static int gemm_16(const GemmArgs& g, cudaStream_t st) {
    return std::is_same<T, __half>::value ? gemm_f16(g, st) : gemm_bf16(g, st);
}
template <class T>
static int ffn_block_16(const FfnBlockArgs& a, cudaStream_t st) {
    return std::is_same<T, __half>::value ? ffn_block_f16(a, st) : ffn_block_bf16(a, st);
}

template <class T>
static int forward(const ofx_shape* s, const uint8_t* wts, const ofx_forward_args* a, uint8_t* ws,
                   cudaStream_t st) {
    const WLayout L = make_layout(s);
    const WsLayout W = make_ws(s, a->batch);
    const int B = a->batch, dm = L.dm, fp = L.fp, hd = dm / s->n_head;
    int* off = reinterpret_cast<int*>(ws + W.off);
    int* n_tok = reinterpret_cast<int*>(ws + W.n_tok);
    int* owner = reinterpret_cast<int*>(ws + W.owner);
    float* x = reinterpret_cast<float*>(ws + W.x);
    T* h = reinterpret_cast<T*>(ws + W.h);
    T* big = reinterpret_cast<T*>(ws + W.big);
    T* q0 = reinterpret_cast<T*>(ws + W.q0);
    T* a0 = reinterpret_cast<T*>(ws + W.a0);
    T* u0 = reinterpret_cast<T*>(ws + W.u0);
    auto lw = [&](int l, size_t o) { return wts + L.layer_bytes * l + o; };
    auto lf = [&](int l, size_t o) { return reinterpret_cast<const float*>(lw(l, o)); };
    // linear layer: bf16 / fp16 mode -> tcgen05 GEMM on the 16-bit operands; fp32 mode -> the activation operand is cut into
    // bf16 hi / lo pieces and multiplied with the pre-split weights on the same tensor-core pipeline (gemm.h)
    uint8_t* split_a = ws + W.split;
    constexpr bool f32 = sizeof(T) == 4;
    // a_pre: the activation operand already lies somewhere as pieces (layernorm_split3 / a piece-output GEMM wrote it);
    // piece_out: write the result as the pieces of the NEXT GEMM's operand instead of fp32
    auto mm = [&](const GemmArgs& g, const uint8_t* w_split, const void* a_pre = nullptr, void* piece_out = nullptr) -> int {
        if constexpr (sizeof(T) == 4) {
            if (!a_pre) {
                OFX_TRY(split_bf16x3(static_cast<const float*>(g.a), g.lda, g.m, g.m_dev, g.k, split_a, kSplitA, st));
                a_pre = split_a;
            }
            GemmArgs t = g;
            t.a = a_pre; t.lda = 3LL * g.k; t.w = w_split; t.ldw = 3LL * g.k; t.out_f32 = 1;
            if (piece_out) { t.out = piece_out; t.ldo = 3LL * g.n; t.out_f32 = 2; }
            return gemm_f32_split(t, st);
        } else {
            (void)w_split; (void)a_pre; (void)piece_out;
            return gemm_16<T>(g, st);
        }
    };
    // LayerNorm in front of a linear layer: h = LN(x); in fp32 mode the pieces of the GEMM operand are
    // written straight into split_a instead (*pre = where they are)
    auto ln_mm = [&](int rows, const int* rows_dev, const float* w, const float* b, const void** pre) -> int {
        *pre = nullptr;
        if constexpr (sizeof(T) == 4) {
            *pre = split_a;
            return layernorm_split3(x, rows, rows_dev, dm, w, b, split_a, st);
        }
        return layernorm<T>(x, rows, rows_dev, dm, w, b, h, st);
    };
    const bool fused_ffn = sizeof(T) == 2 && ffn_block_supported(dm, fp);

    OFX_TRY(scan_valid(a->mask, B, s->max_items, off, n_tok, st));
    AssembleArgs as{};
    as.task = a->task; as.batch = B; as.max_items = s->max_items;
    as.emb = a->emb; as.img = a->img; as.txt = a->txt;
    as.dpm = a->fuse_mode == OFX_FUSE_CONCAT ? dm / 2 : dm;
    as.fuse_mode = a->fuse_mode; as.normalize = a->normalize;
    as.mask = a->mask; as.off = off;
    as.outfit_token = reinterpret_cast<const float*>(wts + L.g_token);
    as.target_img = reinterpret_cast<const float*>(wts + L.g_timg);
    as.text = a->text;
    as.ln_w = lf(0, L.ln1w); as.ln_b = lf(0, L.ln1b);
    as.owner = owner;
    as.item_ids = a->item_ids; as.n_table_rows = a->n_table_rows;
    OFX_TRY(assemble<T>(as, dm, x, h, st));

    for (int l = 0; l < L.nl; ++l) {
        const bool last = l == L.nl - 1;
        // with the fused FFN block the previous layer has already emitted h = norm1_l(x)
        const void* pre1 = nullptr;      // pieces of norm1's output, when the LayerNorm wrote them itself
        if (l > 0 && !fused_ffn)
            OFX_TRY(ln_mm(W.t_max, n_tok, lf(l, L.ln1w), lf(l, L.ln1b), &pre1));
        AttnArgs at{};
        at.batch = B; at.n_head = s->n_head; at.off = off; at.max_s = s->max_items + 1;
        at.max_rows = W.t_max; at.n_tok = n_tok; at.owner = owner;
        if (!last) {
            // dense layer over every valid token
            GemmArgs g{h, dm, lw(l, L.w_qkv), dm, W.t_max, n_tok, 3 * dm, dm, lf(l, L.b_qkv), 0, nullptr, 0, big, 3 * dm, 0};
            OFX_TRY(mm(g, lw(l, L.s_qkv), pre1));
            at.row0_only = 0;
            at.q = big; at.k = big + dm; at.v = big + 2 * dm; at.ldq = at.ldk = at.ldv = 3 * dm;
            at.out = h; at.ldo = dm;
            OFX_TRY(attention<T>(at, hd, st));
            GemmArgs go{h, dm, lw(l, L.w_o), dm, W.t_max, n_tok, dm, dm, lf(l, L.b_o), 0, x, dm, x, dm, 1};
            OFX_TRY(mm(go, lw(l, L.s_o)));
            if (fused_ffn) {
                FfnBlockArgs fa{x, W.t_max, n_tok, dm, fp, lf(l, L.ln2w), lf(l, L.ln2b), lw(l, L.w_1),
                                lf(l, L.b_1), lw(l, L.w_2), lf(l, L.b_2)};
                fa.h_next = h; fa.lnn_w = lf(l + 1, L.ln1w); fa.lnn_b = lf(l + 1, L.ln1b);
                fa.workspace = ws + W.ffn; fa.workspace_bytes = W.ffn_bytes;
                OFX_TRY(ffn_block_16<T>(fa, st));
            } else {
                const void* pre2 = nullptr;
                OFX_TRY(ln_mm(W.t_max, n_tok, lf(l, L.ln2w), lf(l, L.ln2b), &pre2));
                GemmArgs g1{h, dm, lw(l, L.w_1), dm, W.t_max, n_tok, fp, dm, lf(l, L.b_1), 1, nullptr, 0, big, fp, 0};
                OFX_TRY(mm(g1, lw(l, L.s_1), pre2, f32 ? big : nullptr));          // fp32: hidden as pieces
                GemmArgs g2{big, fp, lw(l, L.w_2), fp, W.t_max, n_tok, dm, fp, lf(l, L.b_2), 0, x, dm, x, dm, 1};
                OFX_TRY(mm(g2, lw(l, L.s_2), f32 ? big : nullptr));
            }
        } else {
            // last layer: K,V for every token, everything else for the prefix row only
            const T* w_in = reinterpret_cast<const T*>(lw(l, L.w_qkv));
            GemmArgs gkv{h, dm, w_in + static_cast<size_t>(dm) * dm, dm, W.t_max, n_tok, 2 * dm, dm,
                         lf(l, L.b_qkv) + dm, 0, nullptr, 0, big, 2 * dm, 0};
            OFX_TRY(mm(gkv, lw(l, L.s_qkv) + static_cast<size_t>(dm) * 3 * dm * 2, pre1));     // rows dm.. of the split W_qkv
            GemmArgs gq{h, dm, w_in, dm, B, nullptr, dm, dm, lf(l, L.b_qkv), 0, nullptr, 0, q0, dm, 0};
            // without pre1 (single-layer model) the K/V GEMM above has just split all of h into split_a: rows [0, B) of it
            OFX_TRY(mm(gq, lw(l, L.s_qkv), f32 ? static_cast<const void*>(split_a) : nullptr));
            at.row0_only = 1;
            at.q = q0; at.ldq = dm; at.k = big; at.v = big + dm; at.ldk = at.ldv = 2 * dm;
            at.out = a0; at.ldo = dm;
            OFX_TRY(attention<T>(at, hd, st));
            GemmArgs go{a0, dm, lw(l, L.w_o), dm, B, nullptr, dm, dm, lf(l, L.b_o), 0, x, dm, x, dm, 1};
            OFX_TRY(mm(go, lw(l, L.s_o)));
            if (fused_ffn) {
                FfnBlockArgs fa{x, B, nullptr, dm, fp, lf(l, L.ln2w), lf(l, L.ln2b), lw(l, L.w_1),
                                lf(l, L.b_1), lw(l, L.w_2), lf(l, L.b_2)};
                fa.workspace = ws + W.ffn; fa.workspace_bytes = W.ffn_bytes;
                OFX_TRY(ffn_block_16<T>(fa, st));
            } else {
                const void* pre2 = nullptr;
                OFX_TRY(ln_mm(B, nullptr, lf(l, L.ln2w), lf(l, L.ln2b), &pre2));
                GemmArgs g1{h, dm, lw(l, L.w_1), dm, B, nullptr, fp, dm, lf(l, L.b_1), 1, nullptr, 0, u0, fp, 0};
                OFX_TRY(mm(g1, lw(l, L.s_1), pre2, f32 ? u0 : nullptr));
                GemmArgs g2{u0, fp, lw(l, L.w_2), fp, B, nullptr, dm, fp, lf(l, L.b_2), 0, x, dm, x, dm, 1};
                OFX_TRY(mm(g2, lw(l, L.s_2), f32 ? u0 : nullptr));
            }
        }
    }
    if (a->task == OFX_TASK_CP) {
        OFX_TRY(cp_head(x, B, dm, reinterpret_cast<const float*>(wts + L.g_cpw),
                        reinterpret_cast<const float*>(wts + L.g_cpb), a->logits, a->probs, st));
    } else {
        OFX_TRY(cast_rows<T>(x, static_cast<long long>(B) * dm, q0, st));
        GemmArgs gc{q0, dm, wts + L.g_cir, dm, B, nullptr, L.de, dm, nullptr, 0, nullptr, 0, a->query, L.de, 1};
        OFX_TRY(mm(gc, wts + L.s_cir));
        if (a->cand)
            OFX_TRY(fitb(a->query, a->cand, a->cand_ids, a->n_cand_rows, B, a->n_cand, L.de, a->fitb_dist,
                         reinterpret_cast<long long*>(a->fitb_argmin), st));
    }
    return OFX_OK;
}

}  // namespace ofx

using namespace ofx;

extern "C" {

size_t ofx_packed_weights_bytes(const ofx_shape* shape) {
    if (check_shape(shape) != OFX_OK) return 0;
    return make_layout(shape).total;
}

int ofx_pack_weights(const ofx_shape* shape, const float* const* params, void* packed, void* stream) {
    OFX_TRY(check_shape(shape));
    if (!params || !packed) return fail(OFX_E_ARG, "ofx_pack_weights: null argument");
    OFX_TRY(require_sm100());
    const WLayout L = make_layout(shape);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    OFX_CUDA(cudaMemsetAsync(packed, 0, L.total, st));
    if (shape->precision == OFX_PREC_BF16)
        return pack_all<__nv_bfloat16>(L, params, static_cast<uint8_t*>(packed), st);
    if (shape->precision == OFX_PREC_FP16)
        return pack_all<__half>(L, params, static_cast<uint8_t*>(packed), st);
    return pack_all<float>(L, params, static_cast<uint8_t*>(packed), st);
}

size_t ofx_encoder_workspace_bytes(const ofx_shape* shape, int32_t batch) {
    if (check_shape(shape) != OFX_OK || batch < 0) return 0;
    return make_ws(shape, batch).total;
}

int ofx_encoder_forward(const ofx_shape* shape, const void* packed_weights, const ofx_forward_args* a,
                        void* workspace, size_t workspace_bytes, void* stream) {
    OFX_TRY(check_shape(shape));
    if (!packed_weights || !a) return fail(OFX_E_ARG, "ofx_encoder_forward: null argument");
    if (a->batch < 0 || a->batch > (1 << 26) / (shape->max_items + 1))
        return fail(OFX_E_SHAPE, "batch %d out of range", a->batch);
    if (a->batch == 0) return OFX_OK;
    if (a->task != OFX_TASK_CP && a->task != OFX_TASK_CIR) return fail(OFX_E_ARG, "task %d", a->task);
    if (!a->mask) return fail(OFX_E_ARG, "outfit_mask is null");
    if (!a->emb && !(a->img && a->txt)) return fail(OFX_E_ARG, "need outfit_embedding or img+txt");
    if (!a->emb && a->fuse_mode != OFX_FUSE_CONCAT && a->fuse_mode != OFX_FUSE_MEAN)
        return fail(OFX_E_ARG, "Unsupported aggregation method %d. Use concat or mean.", a->fuse_mode);
    if (a->task == OFX_TASK_CP && !a->logits) return fail(OFX_E_ARG, "logits is null");
    if (a->task == OFX_TASK_CIR && (!a->text || !a->query))
        return fail(OFX_E_ARG, "CIR needs target_item_text_embedding and a query output");
    if (a->cand && (a->n_cand < 1 || (!a->fitb_dist && !a->fitb_argmin)))
        return fail(OFX_E_ARG, "FITB needs n_cand >= 1 and an output");
    if (a->item_ids && (a->emb || !a->img || !a->txt || a->n_table_rows < 1))
        return fail(OFX_E_ARG, "item_ids needs img / txt tables with n_table_rows >= 1 (and no outfit_embedding)");
    if (a->cand_ids && (!a->cand || a->n_cand_rows < 1))
        return fail(OFX_E_ARG, "cand_ids needs a candidate table with n_cand_rows >= 1");
    if (reinterpret_cast<uintptr_t>(a->emb) % 16 || reinterpret_cast<uintptr_t>(a->img) % 16 ||
        reinterpret_cast<uintptr_t>(a->txt) % 16 || reinterpret_cast<uintptr_t>(a->text) % 16 ||
        reinterpret_cast<uintptr_t>(a->cand) % 16 || reinterpret_cast<uintptr_t>(a->query) % 16 ||
        reinterpret_cast<uintptr_t>(workspace) % 256 || reinterpret_cast<uintptr_t>(packed_weights) % 256)
        return fail(OFX_E_ARG, "misaligned pointer (tensors 16 B, workspace / weights 256 B)");
    const size_t need = make_ws(shape, a->batch).total;
    if (!workspace || workspace_bytes < need)
        return fail(OFX_E_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, need);
    OFX_TRY(require_sm100());
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (shape->precision == OFX_PREC_BF16)
        return forward<__nv_bfloat16>(shape, static_cast<const uint8_t*>(packed_weights), a,
                                      static_cast<uint8_t*>(workspace), st);
    if (shape->precision == OFX_PREC_FP16)
        return forward<__half>(shape, static_cast<const uint8_t*>(packed_weights), a,
                               static_cast<uint8_t*>(workspace), st);
    return forward<float>(shape, static_cast<const uint8_t*>(packed_weights), a,
                          static_cast<uint8_t*>(workspace), st);
}

int ofx_fuse(const float* img, const float* txt, int64_t rows, int32_t dpm, int32_t mode,
             int32_t normalize, float* out, void* stream) {
    if (!img || !txt || !out) return fail(OFX_E_ARG, "ofx_fuse: At least image and text embeddings must be provided");
    if (mode != OFX_FUSE_CONCAT && mode != OFX_FUSE_MEAN)
        return fail(OFX_E_ARG, "Unsupported aggregation method %d. Use concat or mean.", mode);
    if (rows < 0) return fail(OFX_E_SHAPE, "rows %lld", (long long)rows);
    OFX_TRY(require_sm100());
    return fuse_rows(img, txt, rows, dpm, mode, normalize, out, static_cast<cudaStream_t>(stream));
}

int ofx_gemm_bf16(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t m, int32_t n, int32_t k,
                  const float* bias, int32_t act_mish, const float* residual, int64_t ldr, void* out,
                  int64_t ldo, int32_t out_f32, void* stream) {
    if (!a || !w || !out) return fail(OFX_E_ARG, "ofx_gemm_bf16: null operand");
    OFX_TRY(require_sm100());
    GemmArgs g{a, lda, w, ldw, m, nullptr, n, k, bias, act_mish, residual, ldr, out, ldo, out_f32};
    return gemm_bf16(g, static_cast<cudaStream_t>(stream));
}

int ofx_gemm_f16(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t m, int32_t n, int32_t k,
                 const float* bias, int32_t act_mish, const float* residual, int64_t ldr, void* out,
                 int64_t ldo, int32_t out_f32, void* stream) {
    if (!a || !w || !out) return fail(OFX_E_ARG, "ofx_gemm_f16: null operand");
    OFX_TRY(require_sm100());
    GemmArgs g{a, lda, w, ldw, m, nullptr, n, k, bias, act_mish, residual, ldr, out, ldo, out_f32};
    return gemm_f16(g, static_cast<cudaStream_t>(stream));
}

size_t ofx_gemm_f32_tc_workspace_bytes(int32_t m, int32_t n, int32_t k) {
    if (m < 0 || n <= 0 || k <= 0) return 0;
    return align_up(static_cast<size_t>(m) * 3 * k * 2, 256) + align_up(static_cast<size_t>(n) * 3 * k * 2, 256);
}

int ofx_gemm_f32_tc(const float* a, int64_t lda, const float* w, int64_t ldw, int32_t m, int32_t n, int32_t k,
                    const float* bias, int32_t act_mish, const float* residual, int64_t ldr, float* out,
                    int64_t ldo, void* workspace, size_t workspace_bytes, void* stream) {
    if (!a || !w || !out) return fail(OFX_E_ARG, "ofx_gemm_f32_tc: null operand");
    if (m < 0 || n <= 0 || k <= 0) return fail(OFX_E_SHAPE, "ofx_gemm_f32_tc: M=%d N=%d K=%d", m, n, k);
    const size_t need = ofx_gemm_f32_tc_workspace_bytes(m, n, k);
    if (!workspace || workspace_bytes < need || reinterpret_cast<uintptr_t>(workspace) % 256)
        return fail(OFX_E_WORKSPACE, "ofx_gemm_f32_tc: workspace %zu B < required %zu B (256-byte aligned)", workspace_bytes, need);
    OFX_TRY(require_sm100());
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* sa = static_cast<uint8_t*>(workspace);
    uint8_t* sw = sa + align_up(static_cast<size_t>(m) * 3 * k * 2, 256);
    OFX_TRY(split_bf16x3(a, lda, m, nullptr, k, sa, kSplitA, st));
    OFX_TRY(split_bf16x3(w, ldw, n, nullptr, k, sw, kSplitW, st));
    GemmArgs g{sa, 3LL * k, sw, 3LL * k, m, nullptr, n, k, bias, act_mish, residual, ldr, out, ldo, 1};
    return gemm_f32_split(g, st);
}

size_t ofx_ffn_block_workspace_bytes(int32_t rows, int32_t d_model, int32_t d_ffn_padded) {
    if (rows < 0 || !ffn_block_supported(d_model, d_ffn_padded)) return 0;
    return ffn_block_workspace_bytes();
}

int ofx_ffn_block_bf16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded, const float* ln_w,
                       const float* ln_b, const void* w1, const float* b1, const void* w2, const float* b2,
                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !ln_w || !ln_b || !w1 || !b1 || !w2 || !b2) return fail(OFX_E_ARG, "ofx_ffn_block_bf16: null argument");
    if (rows < 0) return fail(OFX_E_SHAPE, "ofx_ffn_block_bf16: rows %d", rows);
    if (!ffn_block_supported(d_model, d_ffn_padded))
        return fail(OFX_E_SHAPE, "ofx_ffn_block_bf16: needs d_model 512 and d_ffn_padded %% 256 == 0");
    OFX_TRY(require_sm100());
    FfnBlockArgs fa{x, rows, nullptr, d_model, d_ffn_padded, ln_w, ln_b, w1, b1, w2, b2};
    fa.workspace = workspace; fa.workspace_bytes = workspace_bytes;
    return ffn_block_bf16(fa, static_cast<cudaStream_t>(stream));
}

int ofx_ffn_block_ln_bf16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded, const float* ln_w,
                          const float* ln_b, const void* w1, const float* b1, const void* w2, const float* b2,
                          void* h_next, const float* next_ln_w, const float* next_ln_b, void* workspace,
                          size_t workspace_bytes, void* stream) {
    if (!x || !ln_w || !ln_b || !w1 || !b1 || !w2 || !b2 || !h_next || !next_ln_w || !next_ln_b)
        return fail(OFX_E_ARG, "ofx_ffn_block_ln_bf16: null argument");
    if (rows < 0) return fail(OFX_E_SHAPE, "ofx_ffn_block_ln_bf16: rows %d", rows);
    if (!ffn_block_supported(d_model, d_ffn_padded))
        return fail(OFX_E_SHAPE, "ofx_ffn_block_ln_bf16: needs d_model 512 and d_ffn_padded %% 256 == 0");
    if (reinterpret_cast<uintptr_t>(h_next) % 16) return fail(OFX_E_ARG, "ofx_ffn_block_ln_bf16: misaligned h_next");
    OFX_TRY(require_sm100());
    FfnBlockArgs fa{x, rows, nullptr, d_model, d_ffn_padded, ln_w, ln_b, w1, b1, w2, b2};
    fa.h_next = h_next; fa.lnn_w = next_ln_w; fa.lnn_b = next_ln_b;
    fa.workspace = workspace; fa.workspace_bytes = workspace_bytes;
    return ffn_block_bf16(fa, static_cast<cudaStream_t>(stream));
}

int ofx_ffn_block_f16(float* x, int32_t rows, int32_t d_model, int32_t d_ffn_padded, const float* ln_w,
                      const float* ln_b, const void* w1, const float* b1, const void* w2, const float* b2,
                      void* h_next, const float* next_ln_w, const float* next_ln_b, void* workspace,
                      size_t workspace_bytes, void* stream) {
    if (!x || !ln_w || !ln_b || !w1 || !b1 || !w2 || !b2 || (h_next && (!next_ln_w || !next_ln_b)))
        return fail(OFX_E_ARG, "ofx_ffn_block_f16: null argument");
    if (rows < 0) return fail(OFX_E_SHAPE, "ofx_ffn_block_f16: rows %d", rows);
    if (!ffn_block_supported(d_model, d_ffn_padded))
        return fail(OFX_E_SHAPE, "ofx_ffn_block_f16: needs d_model 512 and d_ffn_padded %% 256 == 0");
    if (reinterpret_cast<uintptr_t>(h_next) % 16) return fail(OFX_E_ARG, "ofx_ffn_block_f16: misaligned h_next");
    OFX_TRY(require_sm100());
    FfnBlockArgs fa{x, rows, nullptr, d_model, d_ffn_padded, ln_w, ln_b, w1, b1, w2, b2};
    fa.h_next = h_next; fa.lnn_w = next_ln_w; fa.lnn_b = next_ln_b;
    fa.workspace = workspace; fa.workspace_bytes = workspace_bytes;
    return ffn_block_f16(fa, static_cast<cudaStream_t>(stream));
}

int ofx_attention(int32_t precision, int32_t d_model, int32_t batch, int32_t max_items, const int32_t* off,
                  const int32_t* owner, const int32_t* n_tok, int32_t row0_only, const void* q, int64_t ldq,
                  const void* k, int64_t ldk, const void* v, int64_t ldv, void* out, int64_t ldo, void* stream) {
    if (precision != OFX_PREC_BF16 && precision != OFX_PREC_FP32 && precision != OFX_PREC_FP16)
        return fail(OFX_E_ARG, "ofx_attention: precision %d not in {0 (bf16), 1 (fp32), 2 (fp16)}", precision);
    if (d_model != 512 && d_model != 1024 && d_model != 1536)
        return fail(OFX_E_SHAPE, "ofx_attention: d_model %d not in {512,1024,1536}", d_model);
    if (max_items < 1 || max_items > 64) return fail(OFX_E_SHAPE, "ofx_attention: max_items %d not in [1,64]", max_items);
    if (batch < 0 || batch > (1 << 26) / (max_items + 1)) return fail(OFX_E_SHAPE, "ofx_attention: batch %d out of range", batch);
    if (row0_only != 0 && row0_only != 1) return fail(OFX_E_ARG, "ofx_attention: row0_only %d not 0 / 1", row0_only);
    const void* ptrs[] = {off, owner, n_tok, q, k, v, out};
    for (const void* p : ptrs)
        if (!p || reinterpret_cast<uintptr_t>(p) % 16)
            return fail(OFX_E_ARG, "ofx_attention: null or not 16-byte aligned pointer");
    // 16-byte rows: 8 elements of bf16 / fp16, 4 of fp32
    const int64_t unit = precision == OFX_PREC_FP32 ? 4 : 8;
    const int64_t lds[] = {ldq, ldk, ldv, ldo};
    for (int64_t ld : lds)
        if (ld < d_model || ld % unit)
            return fail(OFX_E_ARG, "ofx_attention: pitch %lld below d_model %d or not a multiple of %lld", (long long)ld,
                        d_model, (long long)unit);
    OFX_TRY(require_sm100());
    AttnArgs at{};
    at.batch = batch; at.n_head = 16; at.row0_only = row0_only;
    at.max_s = max_items + 1; at.max_rows = batch * (max_items + 1);
    at.n_tok = n_tok; at.owner = owner; at.off = off;
    at.q = q; at.ldq = ldq; at.k = k; at.ldk = ldk; at.v = v; at.ldv = ldv; at.out = out; at.ldo = ldo;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int hd = d_model / 16;
    if (precision == OFX_PREC_BF16) return attention<__nv_bfloat16>(at, hd, st);
    if (precision == OFX_PREC_FP16) return attention<__half>(at, hd, st);
    return attention<float>(at, hd, st);
}
}
