"""CPU: the 1..64 item-slot range through the C ABI size queries and the synthetic-input helpers."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from outfitx_b200 import synth


@pytest.mark.parametrize("precision", [0, 1, 2])
@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_workspace_grows_with_max_items_up_to_64(d_model, precision):
    from outfitx_b200 import _lib
    L = _lib.lib()

    def ws(max_items, batch=1000):
        s = _lib.Shape(d_model, 1024, 16, 6, 2024, max_items, precision)
        return L.ofx_encoder_workspace_bytes(C.byref(s), batch)

    sizes = [ws(n) for n in range(1, 65)]
    assert all(x > 0 for x in sizes)
    assert all(a <= b for a, b in zip(sizes, sizes[1:]))
    assert sizes[-1] > sizes[15]
    assert ws(0) == 0 and ws(65) == 0
    assert b"max_items 65" in L.ofx_last_error()


@pytest.mark.parametrize("precision", [0, 1, 2])
def test_packed_weights_do_not_depend_on_max_items(precision):
    from outfitx_b200 import _lib
    L = _lib.lib()
    sizes = {L.ofx_packed_weights_bytes(C.byref(_lib.Shape(1024, 1024, 16, 6, 2024, n, precision)))
             for n in (1, 16, 17, 40, 64)}
    assert len(sizes) == 1 and sizes.pop() > 0


def test_synth_width_arguments():
    img, txt = synth.make_modalities(5, 64, seed=9, max_items=40)
    assert img.shape == txt.shape == (5, 40, 64)
    mask = synth.make_mask(np.array([0, 3, 40]), 40)
    assert mask.shape == (3, 40) and (~mask).sum(1).tolist() == [0, 3, 40]
    emb, mask, lengths = synth.make_outfits(200, "mean", dim_per_modality=128, seed=3, max_items=64)
    assert emb.shape == (200, 64, 128) and mask.shape == (200, 64)
    assert lengths.min() >= 2 and lengths.max() <= 64 and lengths.max() > 16
    assert np.array_equal((~mask).sum(1), lengths) and not emb[mask].any()


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def test_synth_defaults_are_unchanged():
    """The default width is 16 and gives the bytes the helpers gave before they took a width."""
    assert _digest(*synth.make_modalities(4, 64, seed=1)) == "385a9adf669fe9df"
    assert _digest(synth.make_mask(np.array([0, 5, 16]))) == "251ec4237694d9df"
    assert _digest(*synth.make_outfits(20, "mean", 128, seed=7)) == "2842bdec81e56925"
    assert _digest(*synth.make_outfits(6, "concat", 64, seed=2, fixed_len=9)) == "ce88575c60735e50"
    img, txt = synth.make_modalities(3, 32, seed=1)
    g = np.random.Generator(np.random.PCG64(1))
    assert np.array_equal(img, g.standard_normal((3, 16, 32), dtype=np.float32))
    assert np.array_equal(txt, g.standard_normal((3, 16, 32), dtype=np.float32))
    lengths = np.array([0, 5, 16])
    assert np.array_equal(synth.make_mask(lengths), np.arange(16)[None, :] >= lengths[:, None])
    emb, mask, lengths = synth.make_outfits(50, "concat", seed=7)
    emb16, mask16, lengths16 = synth.make_outfits(50, "concat", seed=7, max_items=16)
    assert emb.shape == (50, 16, 1024) and lengths.max() <= 16
    assert np.array_equal(emb, emb16) and np.array_equal(mask, mask16) and np.array_equal(lengths, lengths16)
    assert np.array_equal(lengths, synth.make_lengths(50, 8))
