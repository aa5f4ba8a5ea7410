"""fp64 reference of the encoder's masked multi-head self-attention over the packed token layout of
``ofx_attention`` (include/ofx.h), its error bound, and the argument cases ``ofx_attention`` refuses.
Shared by test_attention_host.py (CPU) and test_gpu_attention.py."""
import numpy as np
import torch

N_HEAD = 16
PREC = {"bf16": 0, "fp32": 1, "fp16": 2}                               # OFX_PREC_*
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}
# unit of the output / P rounding in the error bound (test_gpu_attention.py derives it)
U = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11, "fp32": 2.0 ** -21}
E_SHAPE, E_ARG, E_ARCH = -1, -2, -3


def packed_layout(lengths):
    """off (B + 1) and owner (n_tok) as int32, and n_tok, of outfits holding `lengths` items.  owner of a prefix
    row is its own outfit (the kernels read owner for item rows only)."""
    lengths = np.asarray(lengths, dtype=np.int64)
    B = len(lengths)
    off = np.zeros(B + 1, np.int64)
    off[1:] = np.cumsum(lengths)
    owner = np.concatenate([np.arange(B), np.repeat(np.arange(B), lengths)]).astype(np.int32)
    return off.astype(np.int32), owner, B + int(off[-1])


def token_rows(lengths):
    """(B, S_max) packed row of token j of outfit b (j = 0: the prefix row b; 0 where j >= S_b) and the validity
    mask j < S_b = 1 + lengths[b]."""
    lengths = np.asarray(lengths, dtype=np.int64)
    B = len(lengths)
    S = lengths + 1
    off = np.concatenate([[0], np.cumsum(lengths)])
    j = np.arange(int(S.max()))[None, :]
    rows = np.where(j == 0, np.arange(B)[:, None], B + off[:-1, None] + j - 1)
    valid = j < S[:, None]
    return np.where(valid, rows, 0), valid


def attention_ref(q, k, v, lengths, row0_only):
    """Plain fp64 attention of every outfit and head over its S = 1 + n tokens.

    q: the query rows -- (n_tok, d), or (B, d) prefix rows with row0_only; k, v: (n_tok, d).  Returns, for the
    output rows (0..n_tok-1, or 0..B-1 with row0_only), in fp64 and broadcast to (rows, d):
    ref = sum_j P_j v_j, M = sum_j P_j |v_j|, A = max_j sum_d |q_d k_jd| / sqrt(hd) of the column's head, S, and
    W = sum_j |v_j| / sum_j exp(s_j - max_i s_i) (the weight of an absolute error in the unnormalised P)."""
    q, k, v = q.double(), k.double(), v.double()
    dev, d = k.device, k.shape[1]
    hd = d // N_HEAD
    rows, valid = token_rows(lengths)
    B, smax = rows.shape
    rows_t = torch.from_numpy(rows).to(dev)
    valid_t = torch.from_numpy(valid).to(dev)
    heads = lambda x: x.reshape(B, -1, N_HEAD, hd).transpose(1, 2)          # (B, H, tokens, hd)
    K, V = heads(k[rows_t]), heads(v[rows_t])
    Q = heads(q[:B]) if row0_only else heads(q[rows_t])
    scale = 1.0 / np.sqrt(hd)
    key_ok = valid_t[:, None, None, :]
    s = (Q @ K.transpose(-1, -2) * scale).masked_fill(~key_ok, float("-inf"))
    e = torch.exp(s - s.amax(-1, keepdim=True))
    den = e.sum(-1, keepdim=True)
    P = e / den
    ref, M = P @ V, P @ V.abs()
    W = (V.abs() * key_ok.transpose(-1, -2)).sum(-2, keepdim=True) / den
    A = (Q.abs() @ K.abs().transpose(-1, -2) * scale).masked_fill(~key_ok, 0.0).amax(-1, keepdim=True)
    A = A.expand(-1, -1, -1, hd)
    flat = lambda x: x.transpose(1, 2).reshape(B, -1, d)                    # (B, tokens, d)
    S = torch.from_numpy(valid.sum(1)).to(dev, torch.float64)
    if row0_only:
        return flat(ref)[:, 0], flat(M)[:, 0], flat(A)[:, 0], S[:, None].expand(B, d), flat(W)[:, 0]
    n_tok = int(rows[valid].max()) + 1
    out = [torch.empty(n_tok, d, dtype=torch.float64, device=dev) for _ in range(5)]
    for o, x in zip(out, (flat(ref), flat(M), flat(A), S[:, None, None].expand(B, smax, d), flat(W))):
        o[rows_t[valid_t]] = x[valid_t]
    return tuple(out)


def error_bound(precision, ref, M, A, S, W):
    """|got - ref| <= u (M + |ref|) + (2 gamma max_j A_j + S 2^-23 + 2^-21) M  [+ 2^-24 W for fp16],
    gamma = hd 2^-23."""
    hd = ref.shape[1] // N_HEAD
    gamma = hd * 2.0 ** -23
    bound = U[precision] * (M + ref.abs()) + (2 * gamma * A + S * 2.0 ** -23 + 2.0 ** -21) * M
    return bound + 2.0 ** -24 * W if precision == "fp16" else bound


def refusal_cases(precision, d_model, ptrs):
    """(what, arguments, expected code) of calls ofx_attention must refuse: each differs from valid_args() in one
    argument (or in the three input pitches)."""
    base = valid_args(precision, d_model, ptrs)
    unit = 4 if precision == "fp32" else 8
    esz = 4 if precision == "fp32" else 2
    cases = [("precision 3", dict(precision=3), E_ARG), ("precision -1", dict(precision=-1), E_ARG),
             ("d_model 768", dict(d_model=768), E_SHAPE), ("d_model 256", dict(d_model=256), E_SHAPE),
             ("max_items 0", dict(max_items=0), E_SHAPE), ("max_items 65", dict(max_items=65), E_SHAPE),
             ("batch -1", dict(batch=-1), E_SHAPE),
             ("batch above 2^26 / 65", dict(batch=(1 << 26) // 65 + 1), E_SHAPE),
             ("row0_only 2", dict(row0_only=2), E_ARG)]
    for name in ("off", "owner", "n_tok", "q", "k", "v", "out"):
        cases.append((f"{name} null", {name: None}, E_ARG))
        cases.append((f"{name} misaligned", {name: base[name] + (4 if name in ("off", "owner", "n_tok") else esz)},
                      E_ARG))
    for ld in ("ldq", "ldk", "ldv", "ldo"):
        cases.append((f"{ld} below d_model", {ld: d_model - unit}, E_ARG))
        cases.append((f"{ld} not a multiple of {unit}", {ld: base[ld] + unit // 2}, E_ARG))
    if precision != "fp32":
        cases.append(("16-bit pitch 3 d_model + 4", dict(ldq=3 * d_model + 4, ldk=3 * d_model + 4,
                                                         ldv=3 * d_model + 4), E_ARG))
    return [(what, {**base, **over}, code) for what, over, code in cases]


ARG_ORDER = ("precision", "d_model", "batch", "max_items", "off", "owner", "n_tok", "row0_only",
             "q", "ldq", "k", "ldk", "v", "ldv", "out", "ldo")


def valid_args(precision, d_model, ptrs, batch=4, max_items=64):
    """A valid call in the encoder's interleaved layout: q | k | v at pitch 3 d_model, out at pitch d_model.  `ptrs`
    maps off, owner, n_tok, q (the q | k | v buffer) and out to 256-byte aligned addresses of large enough buffers."""
    esz = 4 if precision == "fp32" else 2
    return dict(precision=PREC[precision], d_model=d_model, batch=batch, max_items=max_items, off=ptrs["off"],
                owner=ptrs["owner"], n_tok=ptrs["n_tok"], row0_only=0, q=ptrs["q"], ldq=3 * d_model,
                k=ptrs["q"] + d_model * esz, ldk=3 * d_model, v=ptrs["q"] + 2 * d_model * esz, ldv=3 * d_model,
                out=ptrs["out"], ldo=d_model)


def call(lib, args, stream=None):
    return lib.ofx_attention(*(args[n] for n in ARG_ORDER), stream)
