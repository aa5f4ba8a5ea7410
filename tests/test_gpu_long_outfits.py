"""GPU: outfits of up to 64 item slots (S = 1 + n <= 65 tokens per outfit) -- the reference's ``max_length`` set
above 16.  Checked against the reference's stock-torch stack (oracle.torch_port.ReferencePort), which takes any
length, in all three precisions and at the three model widths (head_dim 32, 64, 96).  Outfits of <= 16 items keep
the arithmetic of the 16-slot launch bit for bit, whatever the padding width."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import torch_port
from oracle.make_golden import case_dims
from outfitx_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
W = 64                                                           # the widest supported padding
EDGE = (1, 7, 8, 15, 16, 17, 31, 32, 33, 48, 63, 64)           # every short body and every long tile count
TOL_P = {"fp32": None, "fp16": 5e-3, "bf16": 2e-2}              # absolute on CP probabilities (fp32: 1e-3 relative)


def _method(d_model):
    return {512: "mean", 1024: "concat", 1536: "concat"}[d_model]


@pytest.fixture(scope="module")
def models():
    """(d_model, precision, n_layers) -> (B200 model, CPU oracle port) on one synthetic state_dict."""
    import outfitx_b200 as o
    cache, ports = {}, {}

    def get(d_model, precision, n_layers=6):
        key = (d_model, precision, n_layers)
        if key not in cache:
            method = _method(d_model)
            dpm, d_embed, enc = case_dims(method, d_model)
            sd = synth.make_state_dict(d_model, d_embed, seed=0, n_layers=n_layers)
            cfg = o.OutfitXConfig(item_encoder=o.ItemEncoderConfig(type=enc, aggregation_method=method),
                                  transformer=o.TransformerConfig(n_layers=n_layers), max_length=W)
            m = o.OutfitX(cfg, precision=precision)
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
            if (d_model, n_layers) not in ports:
                ports[(d_model, n_layers)] = torch_port.ReferencePort.from_numpy(sd, n_layers=n_layers)
            cache[key] = (m.to(DEV), ports[(d_model, n_layers)])
        return cache[key]
    return get


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _rel(got, want):
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-12))


def _batch(B, d_model, seed, lengths=None):
    """B outfits padded to W slots, n ~ U{1..64} with the EDGE lengths first; raw modalities and fused embeddings."""
    dpm, d_embed, _ = case_dims(_method(d_model), d_model)
    img, txt = synth.make_modalities(B, dpm, seed, max_items=W)
    if lengths is None:
        lengths = synth.make_lengths(B, seed + 1, lo=1, hi=W)
        lengths[:len(EDGE)] = EDGE
    mask = synth.make_mask(lengths, W)
    emb = synth.fuse(img, txt, _method(d_model))
    emb[mask] = 0.0
    text = synth.make_text_prefix(B, d_model // 2, seed + 2)
    cand = synth.make_items(B * 4, dpm, seed + 3).reshape(B, 4, d_embed)
    return img, txt, emb, mask, lengths, text, cand


def _check_against_port(m, port, precision, emb, mask, text, cand):
    t = torch.from_numpy
    want_logits = port.cp(t(emb), t(mask)).numpy()[:, 0]
    want_p = 1.0 / (1.0 + np.exp(-want_logits))
    want_q = port.cir(t(emb), t(mask), t(text))
    want_pred, want_d = torch_port.fitb(want_q, t(cand))
    want_q, want_pred, want_d = want_q.numpy(), want_pred.numpy(), want_d.numpy()
    probs = m.score_cp(_t(emb), _t(mask)).cpu().numpy()
    pred, dists, q = m.score_fitb(_t(emb), _t(mask), _t(text), _t(cand))
    pred, dists, q = pred.cpu().numpy(), dists.cpu().numpy(), q.cpu().numpy()
    err = np.abs(probs - want_p).max()
    print(f"{precision}: max|dprob| {err:.2e}, query rel {_rel(q, want_q):.2e}, dist rel {_rel(dists, want_d):.2e}, "
          f"FITB flips {(pred != want_pred).sum()} of {len(pred)}")
    if precision == "fp32":
        assert _rel(probs, want_p) <= 1e-3
        assert _rel(q, want_q) <= 1e-3
        assert _rel(dists, want_d) <= 1e-3
    else:
        assert err <= TOL_P[precision]
        assert _rel(q, want_q) <= (1e-2 if precision == "fp16" else 5e-2)
        assert _rel(dists, want_d) <= (1e-2 if precision == "fp16" else 5e-2)
    flip = pred != want_pred
    d = np.sort(want_d, -1)
    assert np.all((d[flip, 1] - d[flip, 0]) < 2e-3)          # the argmin flips only on near-ties


@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_long_outfits_against_cpu_port(models, d_model, precision):
    m, port = models(d_model, precision)
    B = 48 if d_model == 1536 else 64
    _, _, emb, mask, lengths, text, cand = _batch(B, d_model, seed=200 + d_model)
    assert set(EDGE) <= set(int(n) for n in lengths)
    _check_against_port(m, port, precision, emb, mask, text, cand)


@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_short_outfits_are_bit_identical_at_any_padding_width(models, d_model, precision):
    """Outfits of <= 16 items run the same attention arithmetic in the long launch as in the 16-slot one."""
    m, _ = models(d_model, precision)
    B = 96
    lengths = synth.make_lengths(B, 301, lo=1, hi=16)
    lengths[:4] = (1, 7, 15, 16)
    img, txt, emb, _, _, text, cand = _batch(B, d_model, seed=300, lengths=lengths)
    outs = []
    for width in (16, 17, 40, 64):
        mask = synth.make_mask(lengths, width)
        e = np.ascontiguousarray(emb[:, :width])
        probs, logits = m.score_cp(_t(e), _t(mask), return_logits=True)
        pred, dists, q = m.score_fitb(_t(e), _t(mask), _t(text), _t(cand))
        outs.append((width, logits, probs, pred, dists, q))
    for width, *got in outs[1:]:
        for a, b in zip(outs[0][1:], got):
            assert torch.equal(a, b), f"width {width} differs from width 16"


def test_items_in_any_slot_at_64_slots(models):
    """No positional encoding: valid items scattered over the 64 slots (their order kept) give the same bits."""
    m, _ = models(512, "bf16")
    B = 64
    _, _, emb, mask, lengths, text, cand = _batch(B, 512, seed=400)
    rng = np.random.Generator(np.random.PCG64(401))
    emb_s, mask_s = np.zeros_like(emb), np.ones_like(mask)
    for b, n in enumerate(lengths):
        slots = np.sort(rng.choice(W, size=int(n), replace=False))
        emb_s[b, slots], mask_s[b, slots] = emb[b, :n], False
    assert (mask_s != mask).any()
    a =m.score_cp(_t(emb), _t(mask))
    b = m.score_cp(_t(emb_s), _t(mask_s))
    assert torch.equal(a, b)
    qa = m.cir_embed(_t(emb), _t(mask), _t(text))
    qb = m.cir_embed(_t(emb_s), _t(mask_s), _t(text))
    assert torch.equal(qa, qb)


@pytest.mark.parametrize("d_model", [512, 1024])
def test_device_collate_and_fusion_at_64_slots(models, d_model):
    """item_ids (B, 64) over item tables and raw per-slot modalities fused on the fly give the bits of the gathered,
    fused embeddings."""
    from outfitx_b200.model import aggregate_embeddings
    m, _ = models(d_model, "bf16")
    method = _method(d_model)
    dpm, d_embed, _ = case_dims(method, d_model)
    B, n_table = 80, 1000
    lengths = synth.make_lengths(B, 501, lo=1, hi=W)
    lengths[:len(EDGE)] = EDGE
    mask = synth.make_mask(lengths, W)
    img_t, txt_t = synth.make_modalities(n_table, dpm, seed=502, max_items=1)
    img_t, txt_t = _t(img_t[:, 0]), _t(txt_t[:, 0])
    ids = np.random.Generator(np.random.PCG64(503)).integers(0, n_table, size=(B, W)).astype(np.int32)
    ids_t, mask_t = _t(ids), _t(mask)
    fused = aggregate_embeddings(img_t, txt_t, method, normalize=True)
    gathered = fused[ids_t.long()]
    gathered[mask_t] = 0.0
    text = _t(synth.make_text_prefix(B, d_model // 2, 504))
    cand = _t(synth.make_items(B * 4, dpm, 505).reshape(B, 4, d_embed))
    want_p = m.score_cp(gathered, mask_t)
    want = m.score_fitb(gathered, mask_t, text, cand)
    raw = {"image_embeddings": img_t[ids_t.long()], "text_embeddings": txt_t[ids_t.long()]}
    by_ids = {"image_embeddings": img_t, "text_embeddings": txt_t, "item_ids": ids_t}
    for enc in (raw, by_ids):
        assert torch.equal(m.score_cp(outfit_mask=mask_t, encoder_input_dict=enc), want_p)
        got = m.score_fitb(outfit_mask=mask_t, target_item_text_embedding=text, candidate_item_embedding=cand,
                           encoder_input_dict=enc)
        for a, b in zip(got, want):
            assert torch.equal(a, b)


def test_host_pipeline_packed_at_64_slots(models):
    from outfitx_b200.pipeline import HostScoringPipeline, pack_valid_rows
    m, _ = models(512, "bf16")
    B = 300
    img, txt, _, mask, lengths, text, cand = _batch(B, 512, seed=600)
    lengths[len(EDGE)] = 0
    mask = synth.make_mask(lengths, W)
    img[mask], txt[mask] = 0.0, 0.0
    host = [torch.from_numpy(np.ascontiguousarray(a)) for a in (img, txt, mask, text, cand)]
    want_p = m.score_cp(outfit_mask=_t(mask), encoder_input_dict={"image_embeddings": _t(img),
                                                                   "text_embeddings": _t(txt)}).cpu()
    want_pred = m.score_fitb(outfit_mask=_t(mask), target_item_text_embedding=_t(text), candidate_item_embedding=_t(cand),
                             encoder_input_dict={"image_embeddings": _t(img), "text_embeddings": _t(txt)})[0].cpu()
    ir, tr, lens = pack_valid_rows(host[0], host[1], host[2])
    pipe = HostScoringPipeline(m, chunk=128)
    for _ in range(2):                          # eager + capture, then graph replay
        got = pipe.score_packed(ir, tr, lens, host[3], host[4], max_items=W)
        assert torch.equal(got["probs"], want_p) and torch.equal(got["pred"], want_pred)
    # back to 16 slots on the same pipeline: the graphs of the wider staging buffers are not replayed
    short = np.minimum(lengths, 16)
    m16 = synth.make_mask(short, 16)
    i16, t16 = np.ascontiguousarray(img[:, :16]), np.ascontiguousarray(txt[:, :16])
    i16[m16], t16[m16] = 0.0, 0.0
    ir16, tr16, lens16 = pack_valid_rows(torch.from_numpy(i16), torch.from_numpy(t16), torch.from_numpy(m16))
    want16 = m.score_cp(outfit_mask=_t(m16), encoder_input_dict={"image_embeddings": _t(i16), "text_embeddings": _t(t16)})
    got16 = pipe.score_packed(ir16, tr16, lens16)
    assert torch.equal(got16["probs"], want16.cpu())
    with pytest.raises(ValueError, match="1..64"):
        pipe.score_packed(ir, tr, lens, max_items=W + 1)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_pruned_last_layer_alone_at_64_slots(models, precision):
    """n_layers = 1: the only layer is the pruned one (prefix-token queries only), over up to 65 keys."""
    m, port = models(512, precision, n_layers=1)
    _, _, emb, mask, _, text, cand = _batch(64, 512, seed=700)
    _check_against_port(m, port, precision, emb, mask, text, cand)


def test_scale_4096_mixed_outfits(models):
    """Multi-wave launches with long and short outfits mixed: 4096 outfits, n ~ U{2..64}."""
    m, port = models(512, "bf16")
    B = 4096
    emb, mask, lengths = synth.make_outfits(B, "mean", seed=800, max_items=W)
    assert lengths.min() >= 2 and lengths.max() <= W
    probs = m.score_cp(_t(emb), _t(mask)).cpu().numpy()
    n = 256
    want = port.cp(torch.from_numpy(emb[:n]), torch.from_numpy(mask[:n])).numpy()[:, 0]
    want_p = 1.0 / (1.0 + np.exp(-want))
    assert np.abs(probs[:n] - want_p).max() <= 2e-2
    assert np.isfinite(probs).all()


def test_65_slots_are_refused(models):
    from outfitx_b200 import _lib
    m, _ = models(512, "bf16")
    emb = torch.zeros(2, W + 1, 512, device=DEV)
    mask = torch.zeros(2, W + 1, dtype=torch.bool, device=DEV)
    with pytest.raises(ValueError, match="64"):
        m.score_cp(emb, mask)
    L = _lib.lib()
    s = _lib.Shape(512, 1024, 16, 6, 2024, W + 1, _lib.PREC_BF16)
    args = _lib.ForwardArgs()
    assert L.ofx_encoder_forward(C.byref(s), None, C.byref(args), None, 0, None) == -1      # OFX_E_SHAPE
    assert b"max_items 65" in L.ofx_last_error()
