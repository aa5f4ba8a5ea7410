"""CPU: precision="fp16" through the Python API and the C ABI without a GPU -- the mode is accepted, its packed
weights and workspace have the bf16 sizes, an unknown precision is rejected with a message, and the two fp16
building blocks refuse to run without an sm_100 device."""
import ctypes as C

import pytest


def test_model_accepts_fp16_and_still_rejects_unknown_modes():
    import outfitx_b200 as o
    m = o.OutfitX(o.OutfitXConfig(item_encoder=o.ItemEncoderConfig(type="clip", aggregation_method="mean")),
                  precision="fp16")
    assert m.precision == "fp16"
    with pytest.raises(ValueError, match="'bf16', 'fp16' or 'fp32'"):
        o.OutfitX(precision="fp8")


@pytest.mark.parametrize("d_model", [512, 1024, 1536])
def test_fp16_sizes_equal_bf16_sizes(d_model):
    from outfitx_b200 import _lib
    L = _lib.lib()
    s16 = _lib.Shape(d_model, 1024, 16, 6, 2024, 16, _lib.PREC_FP16)
    sbf = _lib.Shape(d_model, 1024, 16, 6, 2024, 16, _lib.PREC_BF16)
    n16 = L.ofx_packed_weights_bytes(C.byref(s16))
    assert n16 > 0 and n16 == L.ofx_packed_weights_bytes(C.byref(sbf))
    for batch in (1, 8192):
        w16 = L.ofx_encoder_workspace_bytes(C.byref(s16), batch)
        assert w16 > 0 and w16 == L.ofx_encoder_workspace_bytes(C.byref(sbf), batch)


def test_unknown_precision_is_rejected_with_a_message():
    from outfitx_b200 import _lib
    L = _lib.lib()
    s = _lib.Shape(512, 1024, 16, 6, 2024, 16, 3)
    assert L.ofx_packed_weights_bytes(C.byref(s)) == 0
    assert b"precision 3" in L.ofx_last_error()
    assert L.ofx_encoder_workspace_bytes(C.byref(s), 64) == 0


def test_fp16_building_blocks_need_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from outfitx_b200 import _lib
    L = _lib.lib()
    buf = (C.c_float * 4096)()
    p = C.addressof(buf)
    assert L.ofx_gemm_f16(p, 64, p, 64, 4, 128, 64, None, 0, None, 0, p, 128, 1, None) == -3
    assert L.ofx_last_error()
    assert L.ofx_ffn_block_f16(p, 4, 512, 2048, p, p, p, p, p, p, None, None, None, p, 256, None) == -3
    assert L.ofx_ffn_block_workspace_bytes(4, 512, 2048) == 256
