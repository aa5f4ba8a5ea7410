"""GPU: the encoder's attention kernels (ofx_attention) against a plain fp64 reference (tests/attention_ref.py) at
every precision, head size (d_model 512 / 1024 / 1536 = head_dim 32 / 64 / 96), outfit length, query set (all tokens,
or the prefix rows of the pruned last layer) and both encoder layouts.  bf16 / fp16 run attention_mma_kernel
(with LONG = true when max_items > 16); fp32 runs the CUDA-core attention_kernel.

Exact routing tests hold a kernel to the bit (or one unit in the last place), so a wrong row, head, tile or key mask
fails however small its effect on the result:
  * q = 0: every P_j = exp(0) = 1 exactly, so the output is the mean of the outfit's S value rows; small-integer V
    keeps the fp32 sum exact.  One key too many or too few moves the mean by about 1 / S.
  * one-hot selection: keys carry their slot j = 8a + b as two one-hot digits in each head's columns, and each
    (query row, head) asks for one slot j* with a score gap of 512 / sqrt(hd) >= 52 over every other key, so
    exp(-gap) vanishes against one ulp and the output is V[j*] bit for bit.  V carries (outfit, slot, head) as small
    integers; j* sweeps key 0, the last key and the tile edges 15 / 16 / 31 / 32 / 47 / 48 / 63 / 64 and changes
    with the head and the query tile.

Bounded-error tests use random q / K / V (unit scores; peaked scores, entries x4, where most exp() underflow; for
fp16, q and V of magnitude up to 2^12 with K scaled down so the scores stay unit-sized).  With s_j the fp64
scores, P_j the fp64 softmax, ref = sum_j P_j v_j, M = sum_j P_j |v_j| and A_j = sum_d |q_d k_jd| / sqrt(hd), every
output element satisfies

    |got - ref| <= u (M + |ref|) + (2 gamma max_j A_j + S 2^-23 + 2^-21) M  [+ 2^-24 W for fp16],

gamma = hd 2^-23, W = sum_j |v_j| / sum_j exp(s_j - max_i s_i), u = 2^-8 (bf16), 2^-11 (fp16), 2^-21 (fp32).
Derivation, with eps = 2^-24 the fp32 unit roundoff:
  * Scores.  The hd-term dot product accumulated in fp32 (fmaf chain, or the mma.sync accumulator) is off by at most
    hd eps sum_d |q_d k_jd| (2 eps per step bounds a truncating accumulator); the scale, log2(e) and max-subtraction
    roundings add a few eps |s_j| <= a few eps A_j.  So |delta_j| <= gamma A_j.
  * Softmax.  exp(s_j + delta_j) / sum_i exp(s_i + delta_i) = P_j exp(delta_j - delta_bar) with |delta_j - delta_bar|
    <= 2 max_j |delta_j|: to first order the output moves by at most 2 gamma max_j A_j sum_j P_j |v_j|.  exp itself
    (expf, __expf or ex2.approx) adds a relative error of a few eps per term.
  * Sums.  The S-term denominator and the S-term P.V sum in fp32 (tensor-core or fmaf, and the online softmax's
    rescales, one per group of 4 keys) are relatively off by at most about S eps of sum_j P_j |v_j|; the reciprocal
    and the final scaling add a few eps more: S 2^-23 + 2^-21 covers them with room.
  * Rounding to the operand type.  The mma kernels round the unnormalised P to bf16 / fp16 (relative u / 2 each,
    weighted by |v_j|: u M / 2) while the denominator keeps the unrounded sum, and every path rounds the output
    (u |ref| / 2, plus the error terms above).  fp32 stores fp32: u = 2^-21 covers the exp and reciprocal errors.
  * fp16 subnormals.  fp16 has no normal number below 2^-14, so an unnormalised P_j = exp(s_j - max) < 2^-14 is
    rounded with an absolute error of up to 2^-25 (half the least subnormal), not a relative one.  Over all keys
    that adds at most 2^-25 sum_j |v_j| to the numerator, divided by the denominator sum_j exp(s_j - max) >= 1:
    2^-25 W, doubled for the same room.  Peaked scores make it visible where the dominant key's v_j is near 0.
The first-order terms leave at least a factor 2 of room, so the bound holds for every input, not on average.  Each
test prints its worst err / bound ratio; a module summary prints the worst per precision, kernel and regime."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/attention_ref.py
from attention_ref import (DTYPES, PREC, attention_ref, call, error_bound, packed_layout,  # noqa: E402
                           token_rows, valid_args)

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHORT = (1, 7, 8, 15, 16)                            # the 16-slot launch
LONG = (17, 24, 31, 32, 33, 48, 63, 64)              # the long launch (outfits <= 16 items: its short bodies)
LAYOUTS = ("qkv", "last")
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _summary():
    yield
    print("\nworst err / bound per precision, kernel and regime:")
    for key in sorted(WORST):
        print("  %-36s %.4f" % (" ".join(key), WORST[key]))


def _kernel(precision, max_items):
    if precision == "fp32":
        return "cuda-core"
    return "mma" if max_items <= 16 else "mma-long"


def _lengths(max_items, seed, extra=7):
    """Every length 0..max_items once plus `extra` random ones, shuffled."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lengths = np.concatenate([np.arange(max_items + 1), rng.integers(0, max_items + 1, extra)])
    return rng.permutation(lengths)


def _bits(x):
    return x.view(torch.int32 if x.dtype == torch.float32 else torch.int16)


def _run(precision, d_model, max_items, lengths, row0_only, layout, q, k, v, pad=0):
    """ofx_attention on q (n_tok rows, or the B prefix rows with row0_only), k, v (n_tok rows) placed in an encoder
    layout: 'qkv' = q | k | v interleaved at pitch 3 d_model with out at pitch d_model (layers 0..L-2), 'last' = a
    separate q at pitch d_model and k | v at pitch 2 d_model (the last layer).  `pad` widens every pitch.  Rows up to
    the host bound B (max_items + 1) are allocated; everything the call must not read is NaN and everything it must
    not write is checked unchanged.  Returns the contracted output rows as fp32."""
    dt = DTYPES[precision]
    B = len(lengths)
    off, owner, n_tok = packed_layout(lengths)
    T = B * (max_items + 1)
    assert n_tok <= T and k.shape[0] == v.shape[0] == n_tok
    n_q = B if row0_only else n_tok
    assert q.shape[0] == n_q
    dm = d_model
    nan = float("nan")
    if layout == "qkv":
        big = torch.full((T, 3 * dm + pad), nan, dtype=dt, device=DEV)
        big[:n_q, :dm] = q.to(dt)
        big[:n_tok, dm:2 * dm] = k.to(dt)
        big[:n_tok, 2 * dm:3 * dm] = v.to(dt)
        qp, kp, vp = big, big[:, dm:], big[:, 2 * dm:]
        ldq = ldk = ldv = 3 * dm + pad
    else:
        qp = torch.full((n_q, dm + pad), nan, dtype=dt, device=DEV)
        qp[:, :dm] = q.to(dt)
        kv = torch.full((T, 2 * dm + pad), nan, dtype=dt, device=DEV)
        kv[:n_tok, :dm] = k.to(dt)
        kv[:n_tok, dm:2 * dm] = v.to(dt)
        kp, vp = kv, kv[:, dm:]
        ldq, ldk, ldv = dm + pad, 2 * dm + pad, 2 * dm + pad
    ldo = dm + pad
    out = torch.full((T + 4, ldo), nan, dtype=dt, device=DEV)
    before = _bits(out).clone()
    t_off = torch.from_numpy(off).to(DEV)
    t_owner = torch.from_numpy(owner).to(DEV)
    t_ntok = torch.tensor([n_tok], dtype=torch.int32, device=DEV)
    args = dict(precision=PREC[precision], d_model=dm, batch=B, max_items=max_items, off=t_off.data_ptr(),
                owner=t_owner.data_ptr(), n_tok=t_ntok.data_ptr(), row0_only=row0_only, q=qp.data_ptr(), ldq=ldq,
                k=kp.data_ptr(), ldk=ldk, v=vp.data_ptr(), ldv=ldv, out=out.data_ptr(), ldo=ldo)
    from outfitx_b200 import _lib
    _lib.check(call(_lib.lib(), args, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    changed = _bits(out) != before
    changed[:n_q, :dm] = False
    assert not bool(changed.any()), "ofx_attention wrote outside rows [0, %d) x columns [0, %d)" % (n_q, dm)
    return out[:n_q, :dm].float()


def _rounded(x, precision):
    return x.to(DTYPES[precision]).float()


def _cases():
    for precision in ("bf16", "fp16", "fp32"):
        for d_model in (512, 1024, 1536):
            for max_items in SHORT + LONG:
                yield precision, d_model, max_items


CASES = list(_cases())
VARIANTS = [(r, lay) for r in (0, 1) for lay in LAYOUTS]


# ------------------------------------------------------------------------------------------------ exact routing
@pytest.mark.parametrize("precision,d_model,max_items", CASES)
def test_zero_queries_give_the_mean_of_the_value_rows(precision, d_model, max_items):
    lengths = _lengths(max_items, seed=d_model + max_items)
    _, _, n_tok = packed_layout(lengths)
    g = torch.Generator(device=DEV).manual_seed(max_items)
    for row0_only, layout in VARIANTS:
        B = len(lengths)
        q = torch.zeros(B if row0_only else n_tok, d_model, device=DEV)
        k = _rounded(torch.randn(n_tok, d_model, device=DEV, generator=g), precision)
        v = torch.randint(1, 17, (n_tok, d_model), device=DEV, generator=g).float()
        got = _run(precision, d_model, max_items, lengths, row0_only, layout, q, k, v)
        want = attention_ref(q, k, v, lengths, row0_only)[0].to(DTYPES[precision])
        ulps = (_bits(got.to(DTYPES[precision])).long() - _bits(want).long()).abs()
        worst = int(ulps.max())
        # positive values: bit patterns are monotone.  fp32 has two roundings (1 / S, the product) at its own ulp
        assert worst <= (2 if precision == "fp32" else 1), (row0_only, layout, worst)


def _one_hot_inputs(lengths, d_model, row0_only, L=512.0):
    """q, k, v of the one-hot selection test, and the (output row -> key row) choice per head."""
    hd = d_model // 16
    B = len(lengths)
    off, owner, n_tok = packed_layout(lengths)
    S = np.asarray(lengths) + 1
    r = np.arange(n_tok)
    outfit = owner
    slot = np.where(r < B, 0, r - B - off[owner] + 1)                   # token index within the outfit
    heads = np.arange(16)
    k = np.zeros((n_tok, 16, hd), np.float32)
    k[r[:, None], heads[None, :], (slot // 8)[:, None]] = 1.0
    k[r[:, None], heads[None, :], (9 + slot % 8)[:, None]] = 1.0
    c = np.arange(hd)
    v = 1 + (outfit[:, None, None] * 31 + slot[:, None, None] * 7 + heads[None, :, None] * 3 + c * 5) % 200
    v[:, :, 0] = slot[:, None] + 1
    v[:, :, 1] = outfit[:, None] % 200 + 1
    v[:, :, 2] = heads[None, :] + 1
    n_q = B if row0_only else n_tok
    qr = r[:n_q]
    edges = np.array([0, -1, 15, 16, 31, 32, 47, 48, 63, 64])         # -1: the last key
    s_q = S[outfit[qr]]
    cand = np.where(edges[None, :] < 0, s_q[:, None] - 1, edges[None, :] % s_q[:, None])     # (n_q, 10), < S
    pick = (heads[None, :] + slot[qr, None] + 3 * (slot[qr, None] // 16) + outfit[qr, None]) % len(edges)
    jstar = np.take_along_axis(cand, pick, 1)                          # (n_q, 16) chosen slot per head
    q = np.zeros((n_q, 16, hd), np.float32)
    q[qr[:, None], heads[None, :], jstar // 8] = L
    q[qr[:, None], heads[None, :], 9 + jstar % 8] = L
    key_row = np.where(jstar == 0, outfit[qr, None], B + off[outfit[qr]][:, None] + jstar - 1)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x.reshape(x.shape[0], -1), dtype=np.float32)).to(DEV)
    return t(q), t(k), t(v), key_row, jstar


@pytest.mark.parametrize("precision,d_model,max_items", CASES)
def test_one_hot_selection_is_exact(precision, d_model, max_items):
    lengths = _lengths(max_items, seed=7 * d_model + max_items)
    hd = d_model // 16
    hit = set()
    for row0_only, layout in VARIANTS:
        q, k, v, key_row, jstar = _one_hot_inputs(lengths, d_model, row0_only)
        got = _run(precision, d_model, max_items, lengths, row0_only, layout, q, k, v)
        want = v.view(-1, 16, hd)[torch.from_numpy(key_row).to(DEV), torch.arange(16, device=DEV)[None, :]]
        bad = (got.view(-1, 16, hd) != want).any(-1)
        if bool(bad.any()):
            row, head = (int(x) for x in bad.nonzero()[0])
            raise AssertionError(f"row0_only {row0_only} {layout}: row {row} head {head} wanted key slot "
                                 f"{jstar[row, head]} (id {want[row, head, :3].tolist()}), got "
                                 f"{got.view(-1, 16, hd)[row, head, :3].tolist()}; {int(bad.sum())} (row, head) wrong")
        hit |= set(int(j) for j in np.unique(jstar))
    assert {0, max_items} <= hit and {15, 16, 31, 32, 47, 48, 63, 64} & set(range(max_items + 1)) <= hit


# ------------------------------------------------------------------------------------------------ bounded error
def _regimes(precision):
    out = [("unit", 1.0, 1.0, 1.0), ("peaked", 4.0, 4.0, 1.0)]
    if precision == "fp16":
        out.append(("large", 2.0 ** 10, 2.0 ** -10, 2.0 ** 10))
    return out


def _random(n, d_model, scale, g, precision):
    x = torch.randn(n, d_model, device=DEV, generator=g) * scale
    return _rounded(x.clamp(-2.0 ** 12, 2.0 ** 12) if scale > 1 else x, precision)


def _check_bound(precision, got, q, k, v, lengths, row0_only):
    ref, M, A, S, W = attention_ref(q, k, v, lengths, row0_only)
    bound = error_bound(precision, ref, M, A, S, W)
    assert bool(torch.isfinite(got).all())
    return ((got.double() - ref).abs() / bound).max().item()


@pytest.mark.parametrize("precision,d_model,max_items", CASES)
def test_random_inputs_within_the_error_bound(precision, d_model, max_items):
    lengths = _lengths(max_items, seed=11 * d_model + max_items)
    _, _, n_tok = packed_layout(lengths)
    B = len(lengths)
    g = torch.Generator(device=DEV).manual_seed(3 * d_model + max_items)
    line = []
    for regime, sq, sk, sv in _regimes(precision):
        worst = 0.0
        for row0_only, layout in VARIANTS:
            q = _random(B if row0_only else n_tok, d_model, sq, g, precision)
            k = _random(n_tok, d_model, sk, g, precision)
            v = _random(n_tok, d_model, sv, g, precision)
            got = _run(precision, d_model, max_items, lengths, row0_only, layout, q, k, v)
            ratio = _check_bound(precision, got, q, k, v, lengths, row0_only)
            assert ratio <= 1.0, (regime, row0_only, layout, ratio)
            worst = max(worst, ratio)
        key = (precision, _kernel(precision, max_items), regime)
        WORST[key] = max(WORST.get(key, 0.0), worst)
        line.append(f"{regime} {worst:.4f}")
    print(f"{precision} d_model {d_model} max_items {max_items}: worst err / bound " + ", ".join(line))


# ------------------------------------------------------------------------------------------------ containment
@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_writes_stay_inside_the_contracted_rows_and_columns(precision, d_model):
    """Pitches wider than the rows (the padding columns are NaN on input and must stay untouched on output), and
    *n_tok below the host row bound: _run checks every other element of out is unchanged."""
    g = torch.Generator(device=DEV).manual_seed(d_model)
    for max_items in (16, 64):
        lengths = _lengths(max_items, seed=max_items, extra=3)
        _, _, n_tok = packed_layout(lengths)
        B = len(lengths)
        for row0_only, layout in VARIANTS:
            q = _random(B if row0_only else n_tok, d_model, 1.0, g, precision)
            k = _random(n_tok, d_model, 1.0, g, precision)
            v = _random(n_tok, d_model, 1.0, g, precision)
            got = _run(precision, d_model, max_items, lengths, row0_only, layout, q, k, v, pad=24)
            assert _check_bound(precision, got, q, k, v, lengths, row0_only) <= 1.0


# ------------------------------------------------------------------------------------------------ batch independence
@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_an_outfit_alone_equals_it_inside_a_large_mixed_batch(precision, d_model):
    B, W = 4096, 64
    rng = np.random.Generator(np.random.PCG64(d_model))
    lengths = rng.integers(0, W + 1, B)
    targets = {0: 64, 5: 0, 1000: 17, 2047: 16, 3000: 1, 4094: 33, 4095: 8}
    for b, n in targets.items():
        lengths[b] = n
    _, _, n_tok = packed_layout(lengths)
    g = torch.Generator(device=DEV).manual_seed(d_model + 1)
    q = _random(n_tok, d_model, 1.0, g, precision)
    k = _random(n_tok, d_model, 1.0, g, precision)
    v = _random(n_tok, d_model, 1.0, g, precision)
    rows, valid = token_rows(lengths)
    for row0_only in (0, 1):
        qb = q[:B] if row0_only else q
        big = _run(precision, d_model, W, lengths, row0_only, "qkv", qb, k, v)
        for b, n in targets.items():
            r = torch.from_numpy(rows[b, valid[b]]).to(DEV)           # the outfit's token rows, prefix first
            alone = _run(precision, d_model, W, [n], row0_only, "qkv", q[r[:1]] if row0_only else q[r], k[r], v[r])
            want = big[r[:1]] if row0_only else big[r]
            assert torch.equal(_bits(alone.to(DTYPES[precision])), _bits(want.to(DTYPES[precision]))), (b, n, row0_only)


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_unaligned_16bit_pitch_is_refused_on_device_buffers(precision):
    """A 16-bit pitch that is not a multiple of 8 has no kernel (its odd rows would not be 16-byte aligned): refused
    without a launch, while the same call at pitch 3 d_model launches one kernel."""
    from outfitx_b200 import _lib
    L = _lib.lib()
    dm, B = 512, 4
    lengths = [3, 0, 64, 1]
    off, owner, n_tok = packed_layout(lengths)
    bufs = {"off": torch.from_numpy(off).to(DEV), "owner": torch.from_numpy(owner).to(DEV),
            "n_tok": torch.tensor([n_tok], dtype=torch.int32, device=DEV),
            "q": torch.zeros(B * 65, 3 * dm + 8, dtype=DTYPES[precision], device=DEV),
            "out": torch.zeros(B * 65, dm, dtype=DTYPES[precision], device=DEV)}
    args = valid_args(precision, dm, {n: t.data_ptr() for n, t in bufs.items()}, batch=B)
    stream = torch.cuda.current_stream().cuda_stream
    n0 = L.ofx_launch_count()
    bad = {**args, "ldq": 3 * dm + 4, "ldk": 3 * dm + 4, "ldv": 3 * dm + 4}
    assert call(L, bad, stream) == -2 and b"multiple of 8" in L.ofx_last_error()
    assert L.ofx_launch_count() == n0
    _lib.check(call(L, args, stream))
    torch.cuda.synchronize()
    assert L.ofx_launch_count() == n0 + 1
