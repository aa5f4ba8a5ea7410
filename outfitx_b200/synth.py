"""Deterministic synthetic weights and inputs for the outfit-scoring path.

Pretrained CLIP weights and the Polyvore data are not available offline, so every test,
fixture and benchmark draws its weights and embeddings from here.  Everything is generated
with numpy's ``Generator(PCG64(seed))`` (bit-stable across numpy versions and hosts), never
with torch's RNG, so the GPU box, this container and the golden fixtures all see the same
bytes without shipping 200 MB of parameters.

Shapes and state_dict key names follow the reference model
(``src/models/outfit_x.py:25-90``; SURVEY.md App. C).  The input contract (zero pad rows,
mask True = pad, valid items left-aligned) follows the reference collate
(``src/models/processor/outfit_x/outfit_x_base_processor.py:20-43``), and the per-modality
L2 normalisation follows ``src/models/encoders/image/base_image_encoder.py:46-47`` /
``text/base_text_encoder.py:37-38``.
"""
from __future__ import annotations

import numpy as np

N_LAYERS = 6
N_HEAD = 16
D_FFN = 2024
MAX_ITEMS = 16


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64(seed))


def make_state_dict(d_model: int, d_embed: int = 1024, seed: int = 0,
                    n_layers: int = N_LAYERS, d_ffn: int = D_FFN) -> dict[str, np.ndarray]:
    """Random-init parameters with the reference's key names (fp32 numpy arrays).

    Magnitudes mimic torch's default init (uniform(+-1/sqrt(fan_in)) Linear weights,
    xavier-uniform in_proj) but biases and LayerNorm affine terms are made non-trivial so
    that every term of the arithmetic is exercised.
    """
    g = _rng(seed)
    sd: dict[str, np.ndarray] = {}

    def uni(shape, bound):
        return g.uniform(-bound, bound, size=shape).astype(np.float32)

    sd["outfit_token"] = (g.standard_normal(d_model) * 0.02).astype(np.float32)
    sd["target_item_image_emb"] = (g.standard_normal(d_model // 2) * 0.02).astype(np.float32)
    for l in range(n_layers):
        p = f"transformer_encoder.layers.{l}."
        xav = float(np.sqrt(6.0 / (d_model + 3 * d_model)))
        sd[p + "self_attn.in_proj_weight"] = uni((3 * d_model, d_model), xav)
        sd[p + "self_attn.in_proj_bias"] = uni((3 * d_model,), 0.02)
        b = 1.0 / np.sqrt(d_model)
        sd[p + "self_attn.out_proj.weight"] = uni((d_model, d_model), b)
        sd[p + "self_attn.out_proj.bias"] = uni((d_model,), 0.02)
        sd[p + "linear1.weight"] = uni((d_ffn, d_model), b)
        sd[p + "linear1.bias"] = uni((d_ffn,), b)
        b2 = 1.0 / np.sqrt(d_ffn)
        sd[p + "linear2.weight"] = uni((d_model, d_ffn), b2)
        sd[p + "linear2.bias"] = uni((d_model,), b2)
        for n in ("norm1", "norm2"):
            sd[p + n + ".weight"] = (1.0 + 0.1 * g.standard_normal(d_model)).astype(np.float32)
            sd[p + n + ".bias"] = (0.05 * g.standard_normal(d_model)).astype(np.float32)
    b = 1.0 / np.sqrt(d_model)
    sd["cp_ffn.1.weight"] = uni((1, d_model), b)
    sd["cp_ffn.1.bias"] = uni((1,), b)
    sd["cir_ffn.0.weight"] = uni((d_embed, d_model), b)
    return sd


def _normalize(x: np.ndarray) -> np.ndarray:
    n = np.sqrt((x.astype(np.float64) ** 2).sum(-1, keepdims=True))
    return (x / np.maximum(n, 1e-12)).astype(np.float32)


def make_modalities(batch: int, dim_per_modality: int = 512, seed: int = 1,
                    normalized: bool = False, max_items: int = MAX_ITEMS) -> tuple[np.ndarray, np.ndarray]:
    """Raw (un-normalised unless asked) image / text item embeddings, (B,max_items,dpm) fp32 each."""
    g = _rng(seed)
    img = g.standard_normal((batch, max_items, dim_per_modality), dtype=np.float32)
    txt = g.standard_normal((batch, max_items, dim_per_modality), dtype=np.float32)
    if normalized:
        img, txt = _normalize(img), _normalize(txt)
    return img, txt


def make_lengths(batch: int, seed: int = 2, lo: int = 2, hi: int = MAX_ITEMS) -> np.ndarray:
    """Valid item count per outfit, n ~ Uniform{lo..hi} (SURVEY.md section 8d)."""
    return _rng(seed).integers(lo, hi + 1, size=batch).astype(np.int32)


def make_mask(lengths: np.ndarray, max_items: int = MAX_ITEMS) -> np.ndarray:
    """(B,max_items) bool, True = pad; valid items left-aligned (reference collate contract)."""
    return np.arange(max_items)[None, :] >= np.asarray(lengths)[:, None]


def fuse(img: np.ndarray, txt: np.ndarray, method: str) -> np.ndarray:
    """Reference fusion contract: normalise each modality then concat / mean (App. A.0).

    This is only used to *build inputs* for API calls that take an already fused
    ``outfit_embedding``; the product's own fusion runs on the GPU (``ofx_fuse``).
    """
    i, t = _normalize(img), _normalize(txt)
    if method == "concat":
        return np.concatenate([i, t], axis=-1)
    if method == "mean":
        return ((i + t) * np.float32(0.5)).astype(np.float32)
    raise ValueError(f"Unsupported aggregation method: {method}. Use 'concat' or 'mean'.")


def make_outfits(batch: int, method: str = "concat", dim_per_modality: int = 512,
                 seed: int = 1, fixed_len: int | None = None, max_items: int = MAX_ITEMS):
    """Fused outfit embeddings + mask as the reference processors would emit them, padded to
    ``max_items`` slots with n ~ Uniform{2..max_items} valid items unless ``fixed_len`` is given."""
    img, txt = make_modalities(batch, dim_per_modality, seed, max_items=max_items)
    lengths = (np.full(batch, fixed_len, np.int32) if fixed_len is not None
               else make_lengths(batch, seed + 1, hi=max_items))
    mask = make_mask(lengths, max_items)
    emb = fuse(img, txt, method)
    emb[mask] = 0.0  # reference pad rows are zeros
    return emb, mask, lengths


def make_text_prefix(batch: int, dim: int, seed: int = 3) -> np.ndarray:
    """CIR / FITB target-item text embedding, (B, d_model/2), L2-normalised."""
    return _normalize(_rng(seed).standard_normal((batch, dim), dtype=np.float32))


def make_items(n: int, dim_per_modality: int = 512, seed: int = 5, dup: int = 0) -> np.ndarray:
    """Gallery / candidate items: (n, 2*dpm) with each modality half normalised (|g|^2 = 2).

    ``dup`` rows at the end are exact copies of randomly chosen earlier rows, to exercise
    the lowest-index tie-break of the exact search.
    """
    g = _rng(seed)
    a = _normalize(g.standard_normal((n, dim_per_modality), dtype=np.float32))
    b = _normalize(g.standard_normal((n, dim_per_modality), dtype=np.float32))
    items = np.concatenate([a, b], axis=-1)
    if dup:
        src = g.integers(0, n - dup, size=dup)
        items[n - dup:] = items[src]
    return items


def make_queries(nq: int, dim: int = 1024, seed: int = 6) -> np.ndarray:
    return _rng(seed).standard_normal((nq, dim), dtype=np.float32)
