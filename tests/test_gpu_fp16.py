"""GPU: precision="fp16" -- fp16 GEMM / attention operands on the tensor cores, fp32 accumulation, fp32 residual
stream, LayerNorm / softmax statistics and heads: the arithmetic of the reference's evaluation under
torch.autocast("cuda", dtype=torch.float16) (base_train_config.py:25, use_amp=True).

Checked against the golden outputs of the unmodified reference, the oracle's stock-torch port, an fp64 matmul of
the fp16-rounded operands (ofx_gemm_f16) and a torch fp32 evaluation of the fused FFN block with operands rounded
to fp16 where the kernel rounds them (ofx_ffn_block_f16)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import torch_port
from oracle.make_golden import CASES, case_dims, case_inputs
from outfitx_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DM = 512


def _method(d_model):
    return "mean" if d_model == 512 else "concat"


def _cfg(d_model):
    import outfitx_b200 as o
    method = _method(d_model)
    return o.OutfitXConfig(item_encoder=o.ItemEncoderConfig(type=case_dims(method, d_model)[2],
                                                            aggregation_method=method))


@pytest.fixture(scope="module")
def models():
    """(d_model, precision) -> (B200 model, CPU oracle port), sharing the synthetic state_dict of the golden cases."""
    import outfitx_b200 as o
    cache = {}

    def get(d_model, precision):
        if (d_model, precision) not in cache:
            sd = synth.make_state_dict(d_model, case_dims(_method(d_model), d_model)[1], seed=0)
            m = o.OutfitX(_cfg(d_model), precision=precision)
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
            cache[(d_model, precision)] = (m.to(DEV), torch_port.ReferencePort.from_numpy(sd))
        return cache[(d_model, precision)]
    return get


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _rel(got, want):
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-12))


# ------------------------------------------------------------------ encoder
@pytest.mark.parametrize("name,method,d_model,batch", CASES)
def test_golden_reference_outputs(models, name, method, d_model, batch):
    g = np.load(os.path.join(GOLDEN, f"model_{name}.npz"))
    dpm, _, _ = case_dims(method, d_model)
    _, _, emb, mask, text, cand = case_inputs(method, batch, dpm=dpm)
    err = {}
    for prec in ("fp16", "bf16"):
        m, _ = models(d_model, prec)
        probs = m.score_cp(_t(emb), _t(mask)).cpu().numpy()
        pred, _, query = m.score_fitb(_t(emb), _t(mask), _t(text), _t(cand))
        err[prec] = float(np.abs(probs - g["probs"][:, 0]).max())
        if prec == "fp16":
            assert _rel(query.cpu().numpy(), g["query"]) <= 1e-2
            assert np.array_equal(pred.cpu().numpy(), g["fitb_argmin"])
    print(f"{name}: max|prob - golden| fp16 {err['fp16']:.2e}, bf16 {err['bf16']:.2e}")
    assert err["fp16"] <= 5e-3
    # 3 fewer significand bits: a mode that silently ran bf16 arithmetic would fail here
    assert err["fp16"] <= max(0.25 * err["bf16"], 2e-4)


@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_seeded_batch_against_oracle(models, d_model):
    """Ragged batch (n ~ U{2..16}: the S <= 8, S <= 16 and S = 17 attention bodies all run) against the CPU port."""
    B = 192 if d_model < 1536 else 96
    method = _method(d_model)
    dpm, d_embed, _ = case_dims(method, d_model)
    emb, mask, lengths = synth.make_outfits(B, method, dim_per_modality=dpm, seed=11)
    seen = set(int(x) for x in lengths)
    assert {16} <= seen and min(seen) <= 7
    text = synth.make_text_prefix(B, d_model // 2, seed=13)
    cand = synth.make_items(B * 4, dpm, seed=14).reshape(B, 4, d_embed)
    m, port = models(d_model, "fp16")
    t = torch.from_numpy
    want_p = torch.sigmoid(port.cp(t(emb), t(mask))).numpy()[:, 0]
    want_q = port.cir(t(emb), t(mask), t(text))
    want_pred, want_d = torch_port.fitb(want_q, t(cand))
    probs = m.score_cp(_t(emb), _t(mask)).cpu().numpy()
    pred, _, q = m.score_fitb(_t(emb), _t(mask), _t(text), _t(cand))
    assert np.abs(probs - want_p).max() <= 5e-3
    assert _rel(q.cpu().numpy(), want_q.numpy()) <= 1e-2
    flip = pred.cpu().numpy() != want_pred.numpy()
    d = np.sort(want_d.numpy(), -1)
    assert np.all((d[flip, 1] - d[flip, 0]) < 2e-3)
    assert flip.mean() <= 0.01


def test_config2_full_batch_against_cpu_port(models):
    """configs[1] as bench.py times it -- 8192 outfits, mean fusion on the fly, CP and FITB over 4 candidates --
    against the reference's stock-torch stack on the full batch.  The FITB bar (argmin identical on >= 99.9 %) is
    asserted over ALL sets, near-ties included; every differing set must still be a near-tie."""
    m, port = models(512, "fp16")
    B = 8192
    img, txt = synth.make_modalities(B, 512, seed=51)
    mask = synth.make_mask(synth.make_lengths(B, 52))
    text = synth.make_text_prefix(B, 256, seed=53)
    cand = synth.make_items(B * 4, 512, seed=54).reshape(B, 4, 1024)
    enc = {"image_embeddings": _t(img), "text_embeddings": _t(txt)}
    probs = m.score_cp(outfit_mask=_t(mask), encoder_input_dict=enc).cpu().numpy()
    pred, dists, _ = m.score_fitb(outfit_mask=_t(mask), target_item_text_embedding=_t(text),
                                  candidate_item_embedding=_t(cand), encoder_input_dict=enc)
    emb = synth.fuse(img, txt, "mean")
    emb[mask] = 0.0
    t = torch.from_numpy
    torch.set_num_threads(os.cpu_count() or 1)
    want_p = torch.sigmoid(port.cp(t(emb), t(mask)).float()).numpy()[:, 0]
    want_pred, want_d = torch_port.fitb(port.cir(t(emb), t(mask), t(text)), t(cand))
    agree = pred.cpu().numpy() == want_pred.numpy()
    dd = np.sort(want_d.numpy(), -1)
    gap = dd[:, 1] - dd[:, 0]
    dprob = np.abs(probs - want_p).max()
    print("fp16 FITB agreement %.5f (%d of %d differ); reference gaps of the differing sets: %s; max|dprob| %.2e; "
          "max|ddist| %.2e" % (agree.mean(), (~agree).sum(), B, np.round(np.sort(gap[~agree]), 5).tolist(), dprob,
                               np.abs(dists.cpu().numpy() - want_d.numpy()).max()))
    assert dprob <= 5e-3
    assert np.all(gap[~agree] < 2e-3)
    assert agree.mean() >= 0.999, f"FITB argmin agreement {agree.mean():.5f} ({(~agree).sum()} of {B} differ)"


def test_host_pipeline_equals_device_forward(models):
    """HostScoringPipeline takes an fp16 model as it is: packed host batches, chunked, first call eager + captured,
    later calls replaying CUDA graphs -- bit-identical to the device-resident fp16 forward."""
    from outfitx_b200.pipeline import HostScoringPipeline, pack_valid_rows
    m, _ = models(512, "fp16")
    B = 257
    img, txt = synth.make_modalities(B, 512, seed=41)
    lengths = synth.make_lengths(B, 42)
    lengths[:3] = (0, 16, 1)
    mask = synth.make_mask(lengths)
    text = synth.make_text_prefix(B, 256, 43)
    cand = synth.make_items(B * 4, 512, 44).reshape(B, 4, 1024)
    enc = {"image_embeddings": _t(img), "text_embeddings": _t(txt)}
    want_p = m.score_cp(outfit_mask=_t(mask), encoder_input_dict=enc).cpu()
    want_pred, _, _ = m.score_fitb(outfit_mask=_t(mask), target_item_text_embedding=_t(text),
                                   candidate_item_embedding=_t(cand), encoder_input_dict=enc)
    host = [torch.from_numpy(np.ascontiguousarray(a)) for a in (img, txt, mask, text, cand)]
    rows = pack_valid_rows(host[0], host[1], host[2])
    for chunk in (64, 1000):
        pipe = HostScoringPipeline(m, chunk=chunk)
        for _ in range(3):
            got = pipe.score_packed(rows[0], rows[1], rows[2], host[3], host[4])
            assert torch.equal(got["probs"], want_p) and torch.equal(got["pred"], want_pred.cpu())
        assert any(e[0] is not None for e in pipe._graphs.values())


# ------------------------------------------------------------------ ofx_gemm_f16
def _gemm(a, w, bias=None, mish=False, residual=None, out=None, out_f32=True):
    from outfitx_b200 import _lib
    m, k = a.shape
    n = w.shape[0]
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32 if out_f32 else torch.float16, device=a.device)
    rc = _lib.lib().ofx_gemm_f16(
        a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), m, n, k,
        bias.data_ptr() if bias is not None else None, int(mish),
        residual.data_ptr() if residual is not None else None, residual.stride(0) if residual is not None else 0,
        out.data_ptr(), out.stride(0), int(out_f32), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, out


@pytest.mark.parametrize("k", [64, 512, 2048])
@pytest.mark.parametrize("n", [128, 256, 384])
@pytest.mark.parametrize("m", [1, 127, 128, 129, 1000, 9477])
def test_gemm_f16_against_fp64(m, n, k):
    from outfitx_b200 import _lib
    g = torch.Generator(device=DEV).manual_seed(m * 31 + n * 7 + k)
    a = torch.randn(m, k, device=DEV, generator=g).half()
    w = (torch.randn(n, k, device=DEV, generator=g) / k ** 0.5).half()
    bias = torch.randn(n, device=DEV, generator=g)
    res = torch.randn(m, n, device=DEV, generator=g)
    lin = a.double() @ w.double().T
    lin_b = lin + bias.double()
    mish = F.mish(lin_b)

    def f32(got, want, atol=1e-4):
        torch.testing.assert_close(got.double(), want, rtol=1e-4, atol=atol)

    def f16(got, want):          # one fp16 rounding of the exact result
        assert got.dtype == torch.float16
        torch.testing.assert_close(got.double(), want.half().double(), rtol=1e-3, atol=1e-4)

    rc, out = _gemm(a, w)
    assert rc == 0
    f32(out, lin)
    f32(_gemm(a, w, bias)[1], lin_b)
    f32(_gemm(a, w, bias, mish=True)[1], mish, atol=3e-5)
    f32(_gemm(a, w, bias, residual=res)[1], lin_b + res.double())
    f32(_gemm(a, w, residual=res)[1], lin + res.double())
    x = res.clone()                                                     # in place, as the encoder updates x
    assert _gemm(a, w, bias, residual=x, out=x)[0] == 0
    f32(x, lin_b + res.double())
    f16(_gemm(a, w, out_f32=False)[1], lin)
    f16(_gemm(a, w, bias, out_f32=False)[1], lin_b)
    f16(_gemm(a, w, bias, mish=True, out_f32=False)[1], mish)
    # an fp16 output takes no residual
    assert _gemm(a, w, bias, residual=res, out_f32=False)[0] == -2
    assert b"residual" in _lib.lib().ofx_last_error()


def test_gemm_f16_rejects_bad_shapes():
    a = torch.zeros(128, 96, device=DEV, dtype=torch.float16)
    assert _gemm(a, a)[0] == -1                                         # K % 64 != 0


# ------------------------------------------------------------------ ofx_ffn_block_f16
def _ffn_params(seed, fp=2048, d_ffn=2024):
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    ln_w, ln_b = 1.0 + 0.1 * r(DM), 0.1 * r(DM)
    w1, b1 = r(fp, DM) / DM ** 0.5, 0.1 * r(fp)
    w2, b2 = r(DM, fp) / fp ** 0.5, 0.1 * r(DM)
    w1[d_ffn:] = 0; b1[d_ffn:] = 0; w2[:, d_ffn:] = 0      # the 2024 -> 2048 zero padding
    return ln_w, ln_b, w1.half().contiguous(), b1, w2.half().contiguous(), b2, g


def _ffn(x, ln_w, ln_b, w1, b1, w2, b2, h=None, nw=None, nb=None, ws_bytes=None):
    from outfitx_b200 import _lib
    L = _lib.lib()
    out = x.clone()
    n = L.ofx_ffn_block_workspace_bytes(out.shape[0], DM, w1.shape[0])
    assert n > 0
    # poisoned: the kernel must not depend on what the workspace held before
    ws = torch.full((n,), 0x5A, dtype=torch.uint8, device=DEV)
    p = lambda t: t.data_ptr() if t is not None else None
    rc = L.ofx_ffn_block_f16(out.data_ptr(), out.shape[0], DM, w1.shape[0], ln_w.data_ptr(), ln_b.data_ptr(),
                             w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), p(h), p(nw), p(nb),
                             ws.data_ptr(), ws.numel() if ws_bytes is None else ws_bytes,
                             torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, out


def _ffn_want(x, ln_w, ln_b, w1, b1, w2, b2):
    h = F.layer_norm(x, (DM,), ln_w, ln_b, 1e-5).half().float()
    u = F.mish(h @ w1.float().T + b1).half().float()
    return x + u @ w2.float().T + b2


@pytest.mark.parametrize("rows", [1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 128 * 74 + 5,
                                  256 * 37 * 2 + 130, 40000])
def test_ffn_block_f16_matches_fp32(rows):
    ln_w, ln_b, w1, b1, w2, b2, g = _ffn_params(rows)
    x = torch.randn(rows, DM, device=DEV, generator=g) * 0.7 + 0.05
    rc, got = _ffn(x, ln_w, ln_b, w1, b1, w2, b2)
    assert rc == 0
    torch.testing.assert_close(got, _ffn_want(x, ln_w, ln_b, w1, b1, w2, b2), rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("fp", [256, 512, 1024, 2048])
def test_ffn_block_f16_chunk_counts(fp):
    ln_w, ln_b, w1, b1, w2, b2, g = _ffn_params(fp, fp=fp, d_ffn=fp)
    x = torch.randn(777, DM, device=DEV, generator=g)
    rc, got = _ffn(x, ln_w, ln_b, w1, b1, w2, b2)
    assert rc == 0
    torch.testing.assert_close(got, _ffn_want(x, ln_w, ln_b, w1, b1, w2, b2), rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("rows", [1, 64, 129, 257, 1000, 128 * 74 + 5, 128 * 74 * 3 + 77])
def test_ffn_block_f16_emits_next_layer_norm(rows):
    """With h_next: the same x as the plain block (bit for bit), h_next == fp16(LayerNorm(x_new)) with the next
    layer's norm1 terms, nothing written past `rows` (several tiles per CTA pair at the larger row counts)."""
    ln_w, ln_b, w1, b1, w2, b2, g = _ffn_params(rows + 1)
    nw = 1.0 + 0.1 * torch.randn(DM, device=DEV, generator=g)
    nb = 0.1 * torch.randn(DM, device=DEV, generator=g)
    x = torch.randn(rows, DM, device=DEV, generator=g) * 0.7 + 0.05
    rc, plain = _ffn(x, ln_w, ln_b, w1, b1, w2, b2)
    assert rc == 0
    h = torch.full((rows + 3, DM), 7.0, device=DEV, dtype=torch.float16)      # 3 guard rows
    rc, out = _ffn(x, ln_w, ln_b, w1, b1, w2, b2, h, nw, nb)
    assert rc == 0
    assert torch.equal(out, plain)
    want = F.layer_norm(out, (DM,), nw, nb, 1e-5)
    torch.testing.assert_close(h[:rows].float(), want, rtol=1e-3, atol=1e-5)   # one fp16 rounding
    assert bool((h[rows:] == 7.0).all())


def test_ffn_block_f16_rejects_other_shapes_and_small_workspaces():
    from outfitx_b200 import _lib
    L = _lib.lib()
    x = torch.zeros(4, 1024, device=DEV)
    p = x.data_ptr()
    assert L.ofx_ffn_block_f16(p, 4, 1024, 2048, p, p, p, p, p, p, None, None, None, p, 1 << 30, None) == -1
    assert L.ofx_ffn_block_f16(p, 4, 512, 2000, p, p, p, p, p, p, None, None, None, p, 1 << 30, None) == -1
    assert L.ofx_ffn_block_workspace_bytes(4, 1024, 2048) == 0
    ln_w, ln_b, w1, b1, w2, b2, g = _ffn_params(5)
    x = torch.randn(4, DM, device=DEV, generator=g)
    assert _ffn(x, ln_w, ln_b, w1, b1, w2, b2, ws_bytes=16)[0] == -5      # checked before anything is launched
    h = torch.empty(4, DM, device=DEV, dtype=torch.float16)
    assert _ffn(x, ln_w, ln_b, w1, b1, w2, b2, h=h)[0] == -2             # h_next without the next norm's terms
