"""GPU: the fused feed-forward block (ofx_ffn_block_bf16: LayerNorm -> linear1 -> mish -> linear2
-> +residual in one tcgen05 cta_group::2 kernel) against a torch fp32 evaluation of the same
arithmetic (torch TransformerEncoderLayer._ff_block as the reference configures it,
/root/reference/src/models/outfit_x.py:32-45), with the operands rounded to bf16 where the
kernel rounds them (LN output, weights, hidden activation)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DM, FP = 512, 2048


def _ws(rows, fp):
    from outfitx_b200 import _lib
    n = _lib.lib().ofx_ffn_block_workspace_bytes(rows, DM, fp)
    assert n > 0
    # poisoned on purpose: the kernel must not depend on what the scratch ring / counters held before
    return torch.full((n,), 0x5A, dtype=torch.uint8, device="cuda")


def _run(x, ln_w, ln_b, w1, b1, w2, b2):
    from outfitx_b200 import _lib
    out = x.clone()
    ws = _ws(out.shape[0], w1.shape[0])
    _lib.check(_lib.lib().ofx_ffn_block_bf16(
        out.data_ptr(), out.shape[0], DM, w1.shape[0], ln_w.data_ptr(), ln_b.data_ptr(), w1.data_ptr(),
        b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out


def _want(x, ln_w, ln_b, w1, b1, w2, b2):
    h = F.layer_norm(x, (DM,), ln_w, ln_b, 1e-5).to(torch.bfloat16).float()
    u = F.mish(h @ w1.float().T + b1).to(torch.bfloat16).float()
    return x + u @ w2.float().T + b2


def _params(seed, fp=FP, d_ffn=2024):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    ln_w, ln_b = 1.0 + 0.1 * r(DM), 0.1 * r(DM)
    w1 = (r(fp, DM) / DM ** 0.5)
    b1 = 0.1 * r(fp)
    w2 = (r(DM, fp) / fp ** 0.5)
    b2 = 0.1 * r(DM)
    w1[d_ffn:] = 0; b1[d_ffn:] = 0; w2[:, d_ffn:] = 0      # the 2024 -> 2048 zero padding
    return ln_w, ln_b, w1.to(torch.bfloat16).contiguous(), b1, w2.to(torch.bfloat16).contiguous(), b2, g


@pytest.mark.parametrize("rows", [1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 128 * 74 + 5, 256 * 37 * 2 + 130, 40000])
def test_ffn_block_matches_fp32(rows):
    ln_w, ln_b, w1, b1, w2, b2, g = _params(rows)
    x = torch.randn(rows, DM, device="cuda", generator=g) * 0.7 + 0.05
    got = _run(x, ln_w, ln_b, w1, b1, w2, b2)
    want = _want(x, ln_w, ln_b, w1, b1, w2, b2)
    torch.testing.assert_close(got, want, rtol=6e-3, atol=6e-3)


def test_ffn_block_other_chunk_counts():
    for fp in (256, 512, 1024):
        ln_w, ln_b, w1, b1, w2, b2, g = _params(fp, fp=fp, d_ffn=fp)
        x = torch.randn(777, DM, device="cuda", generator=g)
        torch.testing.assert_close(_run(x, ln_w, ln_b, w1, b1, w2, b2),
                                   _want(x, ln_w, ln_b, w1, b1, w2, b2), rtol=6e-3, atol=6e-3)


def test_ffn_block_rejects_other_shapes():
    from outfitx_b200 import _lib
    x = torch.zeros(4, 1024, device="cuda")
    rc = _lib.lib().ofx_ffn_block_bf16(x.data_ptr(), 4, 1024, 2048, x.data_ptr(), x.data_ptr(), x.data_ptr(),
                                       x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), 1 << 30, None)
    assert rc == -1
    assert _lib.lib().ofx_ffn_block_workspace_bytes(4, 1024, 2048) == 0
    x = torch.zeros(4, 512, device="cuda")
    rc = _lib.lib().ofx_ffn_block_bf16(x.data_ptr(), 4, 512, 2048, x.data_ptr(), x.data_ptr(), x.data_ptr(),
                                       x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), 16, None)
    assert rc == -5         # workspace too small (checked before anything is launched)


@pytest.mark.parametrize("rows", [1, 64, 129, 257, 1000, 128 * 74 + 5, 128 * 74 * 3 + 77])
def test_ffn_block_emits_next_layer_norm(rows):
    """ofx_ffn_block_ln_bf16: same x as the plain block, and h_next == bf16(LayerNorm(x_new)) with the next
    layer's norm1 terms (rows of several tiles per CTA pair exercise the deferred per-tile hand-over)."""
    from outfitx_b200 import _lib
    ln_w, ln_b, w1, b1, w2, b2, g = _params(rows + 1)
    nw = 1.0 + 0.1 * torch.randn(DM, device="cuda", generator=g)
    nb = 0.1 * torch.randn(DM, device="cuda", generator=g)
    x = torch.randn(rows, DM, device="cuda", generator=g) * 0.7 + 0.05
    plain = _run(x, ln_w, ln_b, w1, b1, w2, b2)
    out = x.clone()
    h = torch.full((rows + 3, DM), 7.0, device="cuda", dtype=torch.bfloat16)     # 3 guard rows
    ws = _ws(rows, w1.shape[0])
    _lib.check(_lib.lib().ofx_ffn_block_ln_bf16(
        out.data_ptr(), rows, DM, w1.shape[0], ln_w.data_ptr(), ln_b.data_ptr(), w1.data_ptr(), b1.data_ptr(),
        w2.data_ptr(), b2.data_ptr(), h.data_ptr(), nw.data_ptr(), nb.data_ptr(), ws.data_ptr(), ws.numel(),
        torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(out, plain)
    want = F.layer_norm(out, (DM,), nw, nb, 1e-5)
    torch.testing.assert_close(h[:rows].float(), want, rtol=8e-3, atol=2e-5)    # one bf16 rounding
    assert (h[:rows].float() - want).abs().max() < 0.02 * (1 + want.abs().max())
    assert bool((h[rows:] == 7.0).all())                                          # nothing past `rows`
