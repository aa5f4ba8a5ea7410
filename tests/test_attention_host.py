"""CPU: ofx_attention refuses every invalid argument before it looks for a device, and the fp64 attention reference of
test_gpu_attention.py (tests/attention_ref.py) equals torch's scaled_dot_product_attention with a key-padding mask."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/attention_ref.py
from attention_ref import (E_ARCH, N_HEAD, attention_ref, call, packed_layout, refusal_cases,  # noqa: E402
                           token_rows, valid_args)


def _host_ptrs():
    buf = torch.zeros(1 << 22, dtype=torch.uint8)                     # host memory: never dereferenced here
    base = (buf.data_ptr() + 255) // 256 * 256
    return buf, {"off": base, "owner": base + 4096, "n_tok": base + 8192, "q": base + 16384, "out": base + 16384}


@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("d_model", [512, 1536])
def test_refusals_come_before_the_device_check(precision, d_model):
    from outfitx_b200 import _lib
    L = _lib.lib()
    _buf, ptrs = _host_ptrs()
    launches = L.ofx_launch_count()
    for what, args, code in refusal_cases(precision, d_model, ptrs):
        assert call(L, args) == code, what
        assert b"ofx_attention" in L.ofx_last_error(), what
    assert L.ofx_launch_count() == launches
    if torch.cuda.is_available():
        return
    # accepted arguments reach the device check: there is no CPU path
    assert call(L, valid_args(precision, d_model, ptrs)) == E_ARCH
    if precision == "fp32":                                            # fp32 rows are 16-byte aligned at pitch % 4
        assert call(L, {**valid_args(precision, d_model, ptrs), "ldo": d_model + 4}) == E_ARCH


def test_packed_layout():
    lengths = [2, 0, 3]
    off, owner, n_tok = packed_layout(lengths)
    assert off.tolist() == [0, 2, 2, 5] and n_tok == 8
    assert owner[3:].tolist() == [0, 0, 2, 2, 2]
    rows, valid = token_rows(lengths)
    assert rows[valid].tolist() == [0, 3, 4, 1, 2, 5, 6, 7]


@pytest.mark.parametrize("d_model", [512, 1024, 1536])
@pytest.mark.parametrize("row0_only", [0, 1])
def test_reference_equals_sdpa(d_model, row0_only):
    """The reference against F.scaled_dot_product_attention on padded fp64 tensors with the key-padding mask."""
    hd = d_model // N_HEAD
    g = torch.Generator().manual_seed(d_model + row0_only)
    lengths = np.array([0, 1, 7, 16, 17, 64, 33, 2])
    _, _, n_tok = packed_layout(lengths)
    B = len(lengths)
    k = torch.randn(n_tok, d_model, generator=g, dtype=torch.float64)
    v = torch.randn(n_tok, d_model, generator=g, dtype=torch.float64)
    q = 3 * torch.randn(B if row0_only else n_tok, d_model, generator=g, dtype=torch.float64)
    ref, M, A, S, W = attention_ref(q, k, v, lengths, row0_only)

    rows, valid = token_rows(lengths)
    rows_t, valid_t = torch.from_numpy(rows), torch.from_numpy(valid)
    heads = lambda x: x.reshape(B, -1, N_HEAD, hd).transpose(1, 2)
    Q = heads(q[:B]) if row0_only else heads(q[rows_t])
    want = F.scaled_dot_product_attention(Q, heads(k[rows_t]), heads(v[rows_t]), attn_mask=valid_t[:, None, None, :])
    want = want.transpose(1, 2).reshape(B, -1, d_model)
    if row0_only:
        want = want[:, 0]
    else:
        flat = torch.empty(n_tok, d_model, dtype=torch.float64)
        flat[rows_t[valid_t]] = want[valid_t]
        want = flat
    torch.testing.assert_close(ref, want, rtol=1e-12, atol=1e-12)
    assert ref.shape == (B if row0_only else n_tok, d_model)
    assert torch.all(M >= ref.abs() - 1e-12) and torch.all(A > 0) and torch.all(W >= M - 1e-12)
    outfit = np.arange(B) if row0_only else packed_layout(lengths)[1]     # the outfit of each output row
    assert S[:, 0].tolist() == (lengths[outfit] + 1).tolist()
