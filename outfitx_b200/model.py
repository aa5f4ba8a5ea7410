"""Drop-in ``OutfitX`` for the outfit-scoring path of the reference's ``src/models/outfit_x.py``.

Same constructor, ``forward(task, **kwargs)`` dispatch (``:97-104``), ``_cp_forward``
(``:120-144``) / ``_cir_forward`` (``:147-172``) signatures, ``device`` property, parameter
names and shapes (``load_state_dict(ckpt['model'])`` of a reference checkpoint works;
SURVEY.md App. C).  The arithmetic runs in ``libofx.so`` (hand-written sm_100a CUDA behind a C
ABI); torch only owns memory and streams.  There is no CPU or eager fallback: tensors must be
on a B200 and the library must load.

Added on top of the reference API (its callers do these by hand, SURVEY.md D12):
``score_cp`` (sigmoid, compatibility_prediction_trainer.py:408), ``score_fitb``
(cdist -> argmin, fill_in_the_blank_trainer.py:50-53), ``cir_embed``; the raw-modality entry
(``encoder_input_dict={'image_embeddings', 'text_embeddings'}``) fuses precomputed CLIP
image / text embeddings on the fly (normalise + concat | mean, model_utils.py:26-45).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch
from torch import nn

from . import _lib
from .configs import OutfitXConfig
from .datatypes import (OutfitCompatibilityPredictionTask, OutfitComplementaryItemRetrievalTask,
                        OutfitFillInTheBlankTask, OutfitPrecomputeEmbeddingTask)

_PRECISIONS = {"bf16": _lib.PREC_BF16, "fp32": _lib.PREC_FP32, "fp16": _lib.PREC_FP16}
_FUSE = {"concat": _lib.FUSE_CONCAT, "mean": _lib.FUSE_MEAN}


class _SelfAttnParams(nn.Module):
    """Parameter holder with nn.MultiheadAttention's names and default init."""

    def __init__(self, d: int):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * d, d))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * d))
        self.out_proj = nn.Linear(d, d)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.constant_(self.out_proj.bias, 0.0)


class _LayerParams(nn.Module):
    """Parameter holder with nn.TransformerEncoderLayer's names (never called)."""

    def __init__(self, d: int, d_ffn: int):
        super().__init__()
        self.self_attn = _SelfAttnParams(d)
        self.linear1 = nn.Linear(d, d_ffn)
        self.linear2 = nn.Linear(d_ffn, d)
        self.norm1 = nn.LayerNorm(d, eps=1e-5)
        self.norm2 = nn.LayerNorm(d, eps=1e-5)


class _EncoderParams(nn.Module):
    def __init__(self, d: int, d_ffn: int, n_layers: int):
        super().__init__()
        self.layers = nn.ModuleList([_LayerParams(d, d_ffn) for _ in range(n_layers)])


class _ItemEncoderInfo(nn.Module):
    """Stands where the reference keeps its frozen CLIP/SigLIP ItemEncoder (out of scope: it is
    upstream of the precomputed embeddings).  Keeps cfg and the d_embed rule (item_encoder.py:38-40)."""

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg

    @property
    def d_embed(self) -> int:
        return self.cfg.d_embed

    def forward(self, *a, **k):
        raise NotImplementedError(
            "the pretrained image/text encoders are upstream of outfitx_b200; pass precomputed "
            "embeddings (outfit_embedding, or encoder_input_dict={'image_embeddings','text_embeddings'})")


def _task_name(task) -> str:
    return getattr(task, "__name__", str(task))


class OutfitX(nn.Module):
    def __init__(self, cfg: Optional[OutfitXConfig] = None, precision: str = "bf16"):
        super().__init__()
        self.cfg = cfg if cfg is not None else OutfitXConfig()
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be 'bf16', 'fp16' or 'fp32', got {precision!r}")
        self.precision = precision
        t = self.cfg.transformer
        if str(getattr(t.activation, "__name__", t.activation)) != "mish":
            raise ValueError("only the reference activation (mish) is implemented")
        self.item_encoder = _ItemEncoderInfo(self.cfg.item_encoder)
        d = self.item_encoder.d_embed
        self.transformer_encoder = _EncoderParams(d, t.d_ffn, t.n_layers)
        self.outfit_token = nn.Parameter(torch.randn(d) * 0.02)
        self.cp_ffn = nn.Sequential(nn.Dropout(t.dropout), nn.Linear(d, 1))
        self.cir_ffn = nn.Sequential(nn.Linear(d, self.cfg.d_embed, bias=False))
        self.target_item_image_emb = nn.Parameter(torch.randn(d // 2) * 0.02)
        self.forward_ = {
            "OutfitCompatibilityPredictionTask": self._cp_forward,
            "OutfitComplementaryItemRetrievalTask": self._cir_forward,
            "OutfitFillInTheBlankTask": self._cir_forward,
            "OutfitPrecomputeEmbeddingTask": self.precompute_embeddings,
        }
        self._packed = None       # (key, uint8 device tensor)
        self._params_cache = None
        self._workspace = None    # uint8 device tensor, grown on demand
        self.requires_grad_(False)
        self.eval()

    # ------------------------------------------------------------------ reference surface
    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def forward(self, task, *args, **kwargs):
        try:
            fn = self.forward_[_task_name(task)]
        except KeyError:
            raise KeyError(task) from None  # the reference raises KeyError here (outfit_x.py:103)
        return fn(*args, **kwargs)

    def precompute_embeddings(self, images=None, texts=None):
        return self.item_encoder(images, texts)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        # a real reference checkpoint also carries the frozen encoders under item_encoder.*
        sd = {k: v for k, v in state_dict.items() if not k.startswith("item_encoder.")}
        out = super().load_state_dict(sd, strict=strict, assign=assign)
        self._packed = None
        self._params_cache = None
        return out

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("outfitx_b200.OutfitX is inference-only (scoring path)")
        return super().train(False)

    def _cp_forward(self, outfit_embedding: Optional[torch.Tensor] = None,
                    outfit_mask: Optional[torch.Tensor] = None,
                    encoder_input_dict: Optional[dict] = None) -> torch.Tensor:
        """-> (B, 1) logits (no sigmoid: outfit_x.py:57-61)."""
        out = self._run(_lib.TASK_CP, outfit_embedding, outfit_mask, encoder_input_dict)
        return out["logits"].unsqueeze(1)

    def _cir_forward(self, outfit_embedding: Optional[torch.Tensor] = None,
                     outfit_mask: Optional[torch.Tensor] = None,
                     target_item_text_embedding: Optional[torch.Tensor] = None,
                     encoder_input_dict: Optional[dict] = None) -> torch.Tensor:
        """-> (B, cfg.d_embed) query embeddings."""
        out = self._run(_lib.TASK_CIR, outfit_embedding, outfit_mask, encoder_input_dict,
                        text=target_item_text_embedding)
        return out["query"]

    # ------------------------------------------------------------------ caller idioms
    def score_cp(self, outfit_embedding=None, outfit_mask=None, encoder_input_dict=None,
                 return_logits: bool = False):
        """sigmoid(logit) per outfit, (B,) -- compatibility_prediction_trainer.py:408."""
        out = self._run(_lib.TASK_CP, outfit_embedding, outfit_mask, encoder_input_dict, probs=True)
        return (out["probs"], out["logits"]) if return_logits else out["probs"]

    def cir_embed(self, outfit_embedding=None, outfit_mask=None, target_item_text_embedding=None,
                  encoder_input_dict=None):
        return self._cir_forward(outfit_embedding, outfit_mask, target_item_text_embedding,
                                 encoder_input_dict)

    def score_fitb(self, outfit_embedding=None, outfit_mask=None, target_item_text_embedding=None,
                   candidate_item_embedding=None, encoder_input_dict=None):
        """cdist(q[:,None], cand).squeeze(1) -> argmin (fill_in_the_blank_trainer.py:50-53).
        -> (pred (B,) int64, dists (B, n_cand) fp32, query (B, De))."""
        if candidate_item_embedding is None:
            raise ValueError("candidate_item_embedding (B, n_cand, d_embed) is required")
        out = self._run(_lib.TASK_CIR, outfit_embedding, outfit_mask, encoder_input_dict,
                        text=target_item_text_embedding, cand=candidate_item_embedding)
        return out["fitb_argmin"], out["fitb_dist"], out["query"]

    # ------------------------------------------------------------------ plumbing
    def _shape(self) -> _lib.Shape:
        t = self.cfg.transformer
        return _lib.Shape(self.item_encoder.d_embed, self.cfg.d_embed, t.n_head, t.n_layers,
                          t.d_ffn, self.cfg.max_length, _PRECISIONS[self.precision])

    def _param_list(self):
        # walked once: named_parameters() costs ~0.3 ms, which at 8 forwards per 8192-outfit step was 2.4 ms of
        # pure host time in the hot loop (tools/time_e2e.py)
        if self._params_cache is None:
            sd = dict(self.named_parameters())
            keys = [f"transformer_encoder.layers.{l}.{k}" for l in range(self.cfg.transformer.n_layers)
                    for k in _lib.LAYER_KEYS] + list(_lib.GLOBAL_KEYS)
            self._params_cache = [sd[k] for k in keys]
        return self._params_cache

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)      # .to() / .cuda() / .float(): parameters may be replaced
        self._params_cache = None
        self._packed = None
        return out

    def _packed_weights(self, dev: torch.device) -> torch.Tensor:
        params = self._param_list()
        key = (dev, self.precision, tuple((p.data_ptr(), p._version) for p in params))
        if self._packed is not None and self._packed[0] == key:
            return self._packed[1]
        shape = self._shape()
        L = _lib.lib()
        n = L.ofx_packed_weights_bytes(C.byref(shape))
        if n == 0:
            raise _lib.OfxError(-1, L.ofx_last_error().decode())
        buf = torch.empty(n, dtype=torch.uint8, device=dev)
        srcs = []
        for p in params:
            if p.device != dev:
                raise RuntimeError(f"parameter on {p.device}, inputs on {dev}: call model.to(device) first")
            srcs.append(p.detach().to(torch.float32).contiguous())
        ptrs = (C.c_void_p * len(srcs))(*[s.data_ptr() for s in srcs])
        _lib.check(L.ofx_pack_weights(C.byref(shape), ptrs, buf.data_ptr(),
                                      torch.cuda.current_stream(dev).cuda_stream))
        torch.cuda.current_stream(dev).synchronize()  # srcs may be temporaries
        self._packed = (key, buf)
        return buf

    def _get_workspace(self, shape: _lib.Shape, batch: int, dev) -> torch.Tensor:
        need = _lib.lib().ofx_encoder_workspace_bytes(C.byref(shape), batch)
        ws = self._workspace
        if ws is None or ws.device != dev or ws.numel() < need:
            self._workspace = ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
        return ws

    @staticmethod
    def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor: outfitx_b200 has no CPU path")
        return t.detach().to(torch.float32).contiguous()

    @torch.no_grad()
    def _run(self, task, emb, mask, enc_dict, text=None, cand=None, probs=False):
        L = _lib.lib()
        shape = self._shape()
        d = shape.d_model
        img = txt = item_ids = cand_ids = None
        n_table = 0
        fuse_mode, normalize = _lib.FUSE_CONCAT, 1
        if enc_dict is not None:
            try:
                img, txt = enc_dict["image_embeddings"], enc_dict["text_embeddings"]
            except KeyError:
                raise ValueError("encoder_input_dict must hold precomputed 'image_embeddings' and "
                                 "'text_embeddings' (B, L, dim_per_modality)") from None
            method = enc_dict.get("aggregation_method", self.cfg.item_encoder.aggregation_method)
            if method not in _FUSE:
                raise ValueError(f"Unsupported aggregation method: {method}. Use 'concat' or 'mean'.")
            fuse_mode = _FUSE[method]
            normalize = int(enc_dict.get("normalize", self.cfg.item_encoder.norm_out))
            img, txt = self._f32(img, "image_embeddings"), self._f32(txt, "text_embeddings")
            dpm = self.cfg.item_encoder.dim_per_modality
            if (2 * dpm if method == "concat" else dpm) != d:
                raise ValueError(f"aggregation '{method}' gives width != d_model {d}")
            item_ids = enc_dict.get("item_ids")
            if item_ids is not None:
                # device-side collate (SURVEY.md N2): image / text embeddings are item TABLES
                # (n_items, dpm) resident in HBM, item_ids (B, L) selects the rows of each slot
                if img.shape != txt.shape or img.dim() != 2 or img.shape[-1] != dpm:
                    raise ValueError(f"with item_ids, image/text embeddings must both be tables (n_items, {dpm})")
                if not item_ids.is_cuda or item_ids.dim() != 2:
                    raise ValueError("item_ids must be a CUDA tensor (B, L)")
                item_ids = item_ids.to(torch.int32).contiguous()
                B, n_items = item_ids.shape
                n_table = img.shape[0]
            else:
                if img.shape != txt.shape or img.dim() != 3 or img.shape[-1] != dpm:
                    raise ValueError(f"image/text embeddings must both be (B, L, {dpm})")
                B, n_items = img.shape[0], img.shape[1]
            dev = img.device
            emb = None
        else:
            if emb is None:
                raise ValueError("outfit_embedding is required")
            emb = self._f32(emb, "outfit_embedding")
            if emb.dim() != 3 or emb.shape[-1] != d:
                raise ValueError(f"outfit_embedding must be (B, L, {d}), got {tuple(emb.shape)}")
            B, n_items = emb.shape[0], emb.shape[1]
            dev = emb.device
        if n_items < 1 or n_items > 64:
            raise ValueError(f"outfits hold 1..64 item slots (max_length {self.cfg.max_length}), got {n_items}")
        shape.max_items = n_items
        if mask is None or tuple(mask.shape) != (B, n_items):
            raise ValueError(f"outfit_mask must be (B, L) = ({B}, {n_items}), True = padding")
        if not mask.is_cuda:
            raise RuntimeError("outfit_mask must be a CUDA tensor")
        mask_u8 = (mask if mask.dtype == torch.bool else mask != 0).contiguous().view(torch.uint8)

        out = {}
        args = _lib.ForwardArgs()
        args.task, args.batch = task, B
        args.emb = emb.data_ptr() if emb is not None else None
        args.img = img.data_ptr() if img is not None else None
        args.txt = txt.data_ptr() if txt is not None else None
        args.fuse_mode, args.normalize = fuse_mode, normalize
        args.mask = mask_u8.data_ptr()
        if item_ids is not None:
            args.item_ids, args.n_table_rows = item_ids.data_ptr(), n_table
        keep = [emb, img, txt, mask_u8, item_ids]
        if task == _lib.TASK_CP:
            out["logits"] = torch.empty(B, dtype=torch.float32, device=dev)
            args.logits = out["logits"].data_ptr()
            if probs:
                out["probs"] = torch.empty(B, dtype=torch.float32, device=dev)
                args.probs = out["probs"].data_ptr()
        else:
            if text is None:
                raise ValueError("target_item_text_embedding is required for CIR / FITB")
            text = self._f32(text, "target_item_text_embedding")
            if tuple(text.shape) != (B, d // 2):
                raise ValueError(f"target_item_text_embedding must be ({B}, {d // 2})")
            args.text = text.data_ptr()
            out["query"] = torch.empty(B, shape.d_embed, dtype=torch.float32, device=dev)
            args.query = out["query"].data_ptr()
            keep.append(text)
            if cand is not None:
                if isinstance(cand, (tuple, list)):        # (table (n_rows, De), ids (B, n_cand))
                    cand, cand_ids = cand
                    cand = self._f32(cand, "candidate table")
                    if cand.dim() != 2 or cand.shape[1] != shape.d_embed:
                        raise ValueError(f"candidate table must be (n_rows, {shape.d_embed})")
                    if not cand_ids.is_cuda or cand_ids.dim() != 2 or cand_ids.shape[0] != B:
                        raise ValueError(f"candidate ids must be a CUDA tensor ({B}, n_cand)")
                    cand_ids = cand_ids.to(torch.int32).contiguous()
                    n_cand = cand_ids.shape[1]
                    args.cand_ids, args.n_cand_rows = cand_ids.data_ptr(), cand.shape[0]
                    keep.append(cand_ids)
                else:
                    cand = self._f32(cand, "candidate_item_embedding")
                    if cand.dim() != 3 or cand.shape[0] != B or cand.shape[2] != shape.d_embed:
                        raise ValueError(f"candidate_item_embedding must be ({B}, n_cand, {shape.d_embed})")
                    n_cand = cand.shape[1]
                args.cand, args.n_cand = cand.data_ptr(), n_cand
                out["fitb_dist"] = torch.empty(B, n_cand, dtype=torch.float32, device=dev)
                out["fitb_argmin"] = torch.empty(B, dtype=torch.int64, device=dev)
                args.fitb_dist = out["fitb_dist"].data_ptr()
                args.fitb_argmin = out["fitb_argmin"].data_ptr()
                keep.append(cand)
        if B == 0:
            return out
        with torch.cuda.device(dev):
            packed = self._packed_weights(dev)
            ws = self._get_workspace(shape, B, dev)
            _lib.check(L.ofx_encoder_forward(C.byref(shape), packed.data_ptr(), C.byref(args),
                                             ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream(dev).cuda_stream))
        return out


def aggregate_embeddings(image_embeddings: Optional[torch.Tensor] = None,
                         text_embeddings: Optional[torch.Tensor] = None,
                         aggregation_method: str = "concat", normalize: bool = False) -> torch.Tensor:
    """``src/utils/model_utils.py:26-45`` on the GPU (``ofx_fuse``).  ``normalize=True`` adds the
    per-modality ``F.normalize`` the reference encoders apply first (base_image_encoder.py:46-47).
    'mean' is the elementwise (img + txt) / 2 the reference intends (SURVEY.md D5)."""
    if image_embeddings is None or text_embeddings is None:
        raise ValueError("At least one of image_embeds or text_embeds must be provided."
                         if image_embeddings is None and text_embeddings is None else
                         "outfitx_b200 fuses two modalities: pass both image and text embeddings")
    if aggregation_method not in _FUSE:
        raise ValueError(f"Unsupported aggregation method: {aggregation_method}. Use 'concat' or 'mean'.")
    if not image_embeddings.is_cuda:
        raise RuntimeError("embeddings must be CUDA tensors: outfitx_b200 has no CPU path")
    img = image_embeddings.detach().to(torch.float32).contiguous()
    txt = text_embeddings.detach().to(torch.float32).contiguous()
    if img.shape != txt.shape:
        raise ValueError("image and text embeddings must have the same shape")
    dpm = img.shape[-1]
    rows = img.numel() // dpm
    width = 2 * dpm if aggregation_method == "concat" else dpm
    out = torch.empty(*img.shape[:-1], width, dtype=torch.float32, device=img.device)
    with torch.cuda.device(img.device):
        _lib.check(_lib.lib().ofx_fuse(img.data_ptr(), txt.data_ptr(), rows, dpm,
                                       _FUSE[aggregation_method], int(normalize), out.data_ptr(),
                                       torch.cuda.current_stream(img.device).cuda_stream))
    return out
