"""ctypes binding of ``libofx.so`` (``include/ofx.h``).  No torch types cross this boundary:
only raw device pointers, sizes and the caller's CUDA stream handle.

There is NO fallback: if the library is missing this module raises, and every compute entry
point fails with OFX_E_ARCH on a host without an sm_100 GPU.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# OFX_LIB_PATH: an instrumented build of the SAME library (e.g. -DOFX_FFN_EPROF), for profiling runs
LIB_PATH = os.environ.get("OFX_LIB_PATH") or os.path.join(HERE, "libofx.so")

OFX_OK = 0
PREC_BF16, PREC_FP32, PREC_FP16 = 0, 1, 2
TASK_CP, TASK_CIR = 0, 1
FUSE_CONCAT, FUSE_MEAN = 0, 1
METRIC_DOT, METRIC_L2 = 0, 1
W_PER_LAYER, W_GLOBAL = 12, 5

# state_dict key suffixes in the order of the OFX_W_* / OFX_G_* enums of ofx.h
LAYER_KEYS = ("self_attn.in_proj_weight", "self_attn.in_proj_bias", "self_attn.out_proj.weight",
              "self_attn.out_proj.bias", "linear1.weight", "linear1.bias", "linear2.weight",
              "linear2.bias", "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")
GLOBAL_KEYS = ("outfit_token", "target_item_image_emb", "cp_ffn.1.weight", "cp_ffn.1.bias",
               "cir_ffn.0.weight")


class OfxError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libofx error {code}: {message}")
        self.code = code


class Shape(C.Structure):
    _fields_ = [("d_model", C.c_int32), ("d_embed", C.c_int32), ("n_head", C.c_int32),
                ("n_layers", C.c_int32), ("d_ffn", C.c_int32), ("max_items", C.c_int32),
                ("precision", C.c_int32)]


class ForwardArgs(C.Structure):
    _fields_ = [("task", C.c_int32), ("batch", C.c_int32), ("emb", C.c_void_p), ("img", C.c_void_p),
                ("txt", C.c_void_p), ("fuse_mode", C.c_int32), ("normalize", C.c_int32),
                ("mask", C.c_void_p), ("text", C.c_void_p), ("logits", C.c_void_p),
                ("probs", C.c_void_p), ("query", C.c_void_p), ("cand", C.c_void_p),
                ("n_cand", C.c_int32), ("fitb_dist", C.c_void_p), ("fitb_argmin", C.c_void_p),
                ("item_ids", C.c_void_p), ("n_table_rows", C.c_int64),
                ("cand_ids", C.c_void_p), ("n_cand_rows", C.c_int64)]


_SIGNATURES = {
    "ofx_version": (C.c_int, []),
    "ofx_last_error": (C.c_char_p, []),
    "ofx_launch_count": (C.c_int64, []),
    "ofx_device_ok": (C.c_int, [C.c_int]),
    "ofx_packed_weights_bytes": (C.c_size_t, [C.POINTER(Shape)]),
    "ofx_pack_weights": (C.c_int, [C.POINTER(Shape), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "ofx_fuse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                           C.c_void_p, C.c_void_p]),
    "ofx_encoder_workspace_bytes": (C.c_size_t, [C.POINTER(Shape), C.c_int32]),
    "ofx_encoder_forward": (C.c_int, [C.POINTER(Shape), C.c_void_p, C.POINTER(ForwardArgs),
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_gallery_packed_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "ofx_gallery_pack": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "ofx_search_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "ofx_topk_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                  C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_exact_search_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "ofx_exact_search": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_topk_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "ofx_category_gallery_packed_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "ofx_category_gallery_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ofx_category_search_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "ofx_category_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    "ofx_category_exact_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int32,
                                            C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                            C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                            C.c_void_p]),
    "ofx_pool_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ofx_loss_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "ofx_focal_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_set_wise_ranking_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                            C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                            C.c_size_t, C.c_void_p]),
    "ofx_cp_metrics": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ofx_ffn_block_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "ofx_ffn_block_bf16": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_ffn_block_ln_bf16": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_gemm_bf16": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64,
                                C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "ofx_gemm_f16": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                               C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64,
                               C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "ofx_ffn_block_f16": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_gemm_f32_tc_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "ofx_gemm_f32_tc": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ofx_attention": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                C.c_void_p, C.c_int64, C.c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded library (built on demand when nvcc is available, never substituted)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            from . import build as _build
            _build.build()
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here = header / library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != OFX_OK:
        raise OfxError(rc, lib().ofx_last_error().decode("utf-8", "replace"))
