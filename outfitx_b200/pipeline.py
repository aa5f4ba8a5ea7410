"""Host-to-result scoring pipeline: the H2D boundary of the reference's callers, overlapped.

The reference moves every collated batch to the GPU and then runs the model on it
(``v.to(local_rank)`` followed by ``model(**input_dict)``,
``src/trains/trainers/compatibility_prediction_trainer.py:140-145``; the demo does the same,
``src/demo/app.py:124-130``), so copy and compute are serialised.  At 64 KB of fp32 embeddings
per outfit (16 slots x (512 + 512) floats) the copy is the longer of the two on a PCIe-attached
B200, so this module splits a host batch into chunks and double-buffers them: chunk i+1 crosses
PCIe on a copy stream while chunk i is scored on the compute stream, and results return through
pinned host buffers.  Everything it calls is the public ``OutfitX`` API; it adds no arithmetic.

``score_packed`` takes the batch WITHOUT its zero padding: the valid item rows of all outfits back to back,
``(sum n_i, dim_per_modality)`` per modality, plus ``lengths (B,)`` -- what a collate produces when it skips the
``pad_value.expand(...)`` of ``outfit_x_base_processor.py:57-81``.  A chunk of outfits is then ONE contiguous
row range per modality (one DMA each) and 44 % fewer PCIe bytes at n ~ U{2..16}; on the device the rows are
addressed through the item-id gather of the device-side collate (slot (b, s) reads row ``off[b] + s``), so the
arithmetic -- and every output bit -- is that of the padded path.  (Round 1 tried to skip the padding with a kernel
that read the pinned padded tensors in place; the persistent scoring kernels starve it of SMs, 16.97 vs 14.95 ms.
The copy engines need no SM, so the fix belongs in the host layout.)
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib


class HostScoringPipeline:
    """Scores host-resident batches with ``model`` (an ``outfitx_b200.OutfitX`` on a CUDA device).

    ``chunk``: outfits per device chunk.  Inputs should be pinned (``tensor.pin_memory()``) for
    the copies to be asynchronous; pageable tensors work but serialise.
    """

    def __init__(self, model, chunk: int = 2048, use_graphs: bool = True):
        """``use_graphs``: the packed path replays one CUDA graph per (staging slot, chunk size) instead of issuing the
        ~120 launches of a CP + FITB pass one by one -- at 2048 outfits per chunk the host needed as long to issue a
        chunk as the GPU to run it.  Same kernels, same arguments (the staging buffers are persistent), same bits."""
        self.use_graphs = use_graphs
        self.tail_min = chunk      # smallest chunk of a tapered tail (see _plan); = chunk: uniform chunks
        self._graphs = {}
        self._graph_width = None   # max_items of the captured graphs: their staging buffers are sized by it
        if chunk < 1:
            raise ValueError("chunk must be >= 1")
        self.model, self.chunk = model, chunk
        dev = model.device
        if dev.type != "cuda":
            raise RuntimeError("the model must be on a CUDA device: outfitx_b200 has no CPU path")
        self.dev = dev
        self.copy_stream = torch.cuda.Stream(dev)
        self.compute_stream = torch.cuda.Stream(dev)
        # device staging buffers.  Four, not two: with a tapered tail the copy of chunk i must not wait for the scoring
        # of chunk i - 2 (the step is copy-bound: every stall of the copy engine is added to it)
        self.n_slots = 4
        self._slots = [dict() for _ in range(self.n_slots)]
        self._free = [torch.cuda.Event() for _ in range(self.n_slots)]    # slot may be overwritten
        self._ready = [torch.cuda.Event() for _ in range(self.n_slots)]   # slot's copies have landed
        self._host = {}                          # pinned scratch for the ids / masks derived from lengths

    def _plan(self, batch: int, taper: bool):
        """Chunk boundaries [(lo, hi)]: uniform chunks, optionally with a tail cut into halves down to ``tail_min``.
        Measured on configs[1] (tools/time_e2e.py, 8192 outfits, graphs on): every chunk costs ~0.6-1 ms on top of its
        share of the work (a CP + FITB pass is ~120 kernels whose prologues / tails do not shrink with the batch), and
        PCIe delivers ~43 GB/s while the scoring kernels run (55 GB/s alone), so 4 chunks of 2048 (12.1 ms) beat both
        a tapered tail (2048 x 3 + 1024 x 2: 13.3 ms, ... + 512 x 2: 14.6 ms) and fewer, larger chunks."""
        out, lo = [], 0
        while batch - lo > self.chunk:
            out.append((lo, lo + self.chunk))
            lo += self.chunk
        rest = batch - lo
        if taper:
            while rest > self.tail_min:
                half = max(self.tail_min, (rest // 2 + 127) // 128 * 128)
                out.append((lo, lo + half))
                lo, rest = lo + half, rest - half
        if rest > 0:
            out.append((lo, lo + rest))
        return out

    def _stage(self, slot: int, name: str, src: torch.Tensor) -> torch.Tensor:
        buf = self._slots[slot].get(name)
        if buf is None or buf.shape[1:] != src.shape[1:] or buf.dtype != src.dtype or buf.shape[0] < src.shape[0]:
            buf = torch.empty((self.chunk,) + tuple(src.shape[1:]), dtype=src.dtype, device=self.dev)
            self._slots[slot][name] = buf
        view = buf[: src.shape[0]]
        view.copy_(src, non_blocking=True)
        return view

    def _stage_rows(self, slot: int, name: str, src: torch.Tensor, cap_rows: int) -> torch.Tensor:
        """Like _stage for a ragged row range: the buffer holds up to cap_rows rows."""
        buf = self._slots[slot].get(name)
        if buf is None or buf.shape[1:] != src.shape[1:] or buf.dtype != src.dtype or buf.shape[0] < max(cap_rows, src.shape[0]):
            buf = torch.empty((max(cap_rows, src.shape[0], 1),) + tuple(src.shape[1:]), dtype=src.dtype, device=self.dev)
            self._slots[slot][name] = buf
        view = buf[: src.shape[0]]
        if src.shape[0]:
            view.copy_(src, non_blocking=True)
        return view

    def _pinned(self, name: str, shape, dtype) -> torch.Tensor:
        t = self._host.get(name)
        if t is None or t.shape != tuple(shape) or t.dtype != dtype:
            t = torch.empty(shape, dtype=dtype).pin_memory()
            self._host[name] = t
        return t

    @torch.no_grad()
    def score(self, image_embeddings: torch.Tensor, text_embeddings: torch.Tensor, outfit_mask: torch.Tensor,
              target_item_text_embedding: Optional[torch.Tensor] = None,
              candidate_item_embedding: Optional[torch.Tensor] = None,
              out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """CP probabilities (and, when ``target_item_text_embedding`` + ``candidate_item_embedding``
        are given, FITB predictions) for a HOST batch of raw per-modality embeddings
        ``(B, L, dim_per_modality)``.  Returns pinned host tensors ``probs (B,)`` [, ``pred (B,)``];
        the call returns once they are valid."""
        B = image_embeddings.shape[0]
        fitb = candidate_item_embedding is not None
        if fitb and target_item_text_embedding is None:
            raise ValueError("FITB scoring needs target_item_text_embedding")
        if out is None:
            out = {"probs": torch.empty(B, dtype=torch.float32).pin_memory()}
            if fitb:
                out["pred"] = torch.empty(B, dtype=torch.int64).pin_memory()
        cur = torch.cuda.current_stream(self.dev)
        self.copy_stream.wait_stream(cur)
        self.compute_stream.wait_stream(cur)
        for i, lo in enumerate(range(0, B, self.chunk)):
            hi = min(B, lo + self.chunk)
            s = i % self.n_slots
            with torch.cuda.stream(self.copy_stream):
                if i >= self.n_slots:
                    self.copy_stream.wait_event(self._free[s])
                d = {"mask": self._stage(s, "mask", outfit_mask[lo:hi])}
                d["img"] = self._stage(s, "img", image_embeddings[lo:hi])
                d["txt"] = self._stage(s, "txt", text_embeddings[lo:hi])
                if fitb:
                    d["text"] = self._stage(s, "text", target_item_text_embedding[lo:hi])
                    d["cand"] = self._stage(s, "cand", candidate_item_embedding[lo:hi])
                self._ready[s].record(self.copy_stream)
            with torch.cuda.stream(self.compute_stream):
                self.compute_stream.wait_event(self._ready[s])
                enc = {"image_embeddings": d["img"], "text_embeddings": d["txt"]}
                probs = self.model.score_cp(outfit_mask=d["mask"], encoder_input_dict=enc)
                out["probs"][lo:hi].copy_(probs, non_blocking=True)
                if fitb:
                    pred, _, _ = self.model.score_fitb(outfit_mask=d["mask"], target_item_text_embedding=d["text"],
                                                       candidate_item_embedding=d["cand"], encoder_input_dict=enc)
                    out["pred"][lo:hi].copy_(pred, non_blocking=True)
                self._free[s].record(self.compute_stream)
        cur.wait_stream(self.compute_stream)
        self.compute_stream.synchronize()
        return out

    @torch.no_grad()
    def score_packed(self, image_rows: torch.Tensor, text_rows: torch.Tensor, lengths: torch.Tensor,
                     target_item_text_embedding: Optional[torch.Tensor] = None,
                     candidate_item_embedding: Optional[torch.Tensor] = None,
                     out: Optional[Dict[str, torch.Tensor]] = None, max_items: int = 16) -> Dict[str, torch.Tensor]:
        """As ``score`` for a HOST batch in the packed layout: ``image_rows`` / ``text_rows``
        ``(sum(lengths), dim_per_modality)`` hold the valid items of outfit 0, then outfit 1, ...;
        ``lengths (B,)`` integers in ``[0, max_items]`` (a collate truncates to ``max_items`` first, 16 by default,
        ``outfit_x_base_processor.py:57-81``); ``max_items`` lies in 1..64.  Bit-identical to ``score`` on the
        padded tensors."""
        if not 1 <= max_items <= 64:
            raise ValueError(f"max_items must lie in 1..64, got {max_items}")
        lens = lengths.detach().to("cpu", torch.int64).flatten()
        B = lens.numel()
        if B and (int(lens.min()) < 0 or int(lens.max()) > max_items):
            raise ValueError(f"lengths must lie in [0, {max_items}]")
        total = int(lens.sum())
        if image_rows.shape != text_rows.shape or image_rows.dim() != 2 or image_rows.shape[0] != total:
            raise ValueError(f"image_rows / text_rows must both be (sum(lengths) = {total}, dim_per_modality)")
        fitb = candidate_item_embedding is not None
        if fitb and target_item_text_embedding is None:
            raise ValueError("FITB scoring needs target_item_text_embedding")
        if out is None:
            out = {"probs": torch.empty(B, dtype=torch.float32).pin_memory()}
            if fitb:
                out["pred"] = torch.empty(B, dtype=torch.int64).pin_memory()
        # host side of the collate, vectorised: row offsets, the padding mask and the chunk-local row id of every slot
        plan = self._plan(B, taper=self.use_graphs)
        mask_h = self._pinned("mask", (B, max_items), torch.bool)
        ids_h = self._pinned("ids", (B, max_items), torch.int32)
        off = packed_layout(lens, plan, max_items, mask_h, ids_h)
        cap_rows = self.chunk * max_items
        if max_items != self._graph_width:
            # a new width reallocates the mask / ids / row staging buffers that the captured graphs read
            self._graphs.clear()
            self._graph_width = max_items
        cur = torch.cuda.current_stream(self.dev)
        self.copy_stream.wait_stream(cur)
        self.compute_stream.wait_stream(cur)
        for i, (lo, hi) in enumerate(plan):
            r0, r1 = int(off[lo]), int(off[hi])
            s = i % self.n_slots
            with torch.cuda.stream(self.copy_stream):
                if i >= self.n_slots:
                    self.copy_stream.wait_event(self._free[s])
                d = {"mask": self._stage(s, "pmask", mask_h[lo:hi]), "ids": self._stage(s, "pids", ids_h[lo:hi]),
                     "img": self._stage_rows(s, "pimg", image_rows[r0:r1], cap_rows),
                     "txt": self._stage_rows(s, "ptxt", text_rows[r0:r1], cap_rows)}
                if fitb:
                    d["text"] = self._stage(s, "text", target_item_text_embedding[lo:hi])
                    d["cand"] = self._stage(s, "cand", candidate_item_embedding[lo:hi])
                self._ready[s].record(self.copy_stream)
            with torch.cuda.stream(self.compute_stream):
                self.compute_stream.wait_event(self._ready[s])
                # the slot's row buffers are the "table" of the device-side collate (ids never point past the chunk's rows)
                enc = {"image_embeddings": self._slots[s]["pimg"], "text_embeddings": self._slots[s]["ptxt"], "item_ids": d["ids"]}

                def run():
                    probs = self.model.score_cp(outfit_mask=d["mask"], encoder_input_dict=enc)
                    pred = None
                    if fitb:
                        pred, _, _ = self.model.score_fitb(outfit_mask=d["mask"], target_item_text_embedding=d["text"],
                                                           candidate_item_embedding=d["cand"], encoder_input_dict=enc)
                    return probs, pred

                key = (s, hi - lo, fitb, tuple(image_rows.shape[1:]), image_rows.dtype,
                       tuple(candidate_item_embedding.shape[1:]) if fitb else None)
                entry = self._graphs.get(key) if self.use_graphs else None
                if entry is not None and entry[0] is not None:
                    entry[0].replay()
                    probs, pred = entry[1], entry[2]
                else:
                    probs, pred = run()
                    if self.use_graphs and entry is None:
                        # first time this (slot, chunk size) is seen: the eager pass above was the warm-up; capture the
                        # same calls on the same persistent buffers for the following steps
                        try:
                            g = torch.cuda.CUDAGraph()
                            self.compute_stream.synchronize()
                            with torch.cuda.graph(g, stream=self.compute_stream):
                                gp, gq = run()
                            self._graphs[key] = (g, gp, gq)
                        except Exception:
                            self._graphs[key] = (None, None, None)      # not capturable here: stay eager
                            torch.cuda.synchronize(self.dev)
                out["probs"][lo:hi].copy_(probs, non_blocking=True)
                if fitb:
                    out["pred"][lo:hi].copy_(pred, non_blocking=True)
                self._free[s].record(self.compute_stream)
        cur.wait_stream(self.compute_stream)
        self.compute_stream.synchronize()
        return out

    @torch.no_grad()
    def score_ids(self, item_ids: torch.Tensor, outfit_mask: torch.Tensor, image_table: torch.Tensor,
                  text_table: torch.Tensor, target_item_text_embedding: Optional[torch.Tensor] = None,
                  candidate_ids: Optional[torch.Tensor] = None, candidate_table: Optional[torch.Tensor] = None,
                  out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """As ``score`` but with the collate on the device (SURVEY.md N2): the item embedding tables
        ``(n_items, dim_per_modality)`` [and the fused candidate table ``(n_items, d_embed)``] are
        DEVICE tensors resident in HBM -- the counterpart of the embedding dict the reference's
        trainers keep in host memory (``compatibility_prediction_trainer.py:329-349``) -- and a
        batch is ``item_ids (B, L)`` int32 + ``outfit_mask`` [+ ``candidate_ids (B, n_cand)``] on the
        HOST.  Only ids cross PCIe (64 B per outfit instead of 64 KB)."""
        B = item_ids.shape[0]
        fitb = candidate_ids is not None
        if fitb and (target_item_text_embedding is None or candidate_table is None):
            raise ValueError("FITB scoring needs target_item_text_embedding and candidate_table")
        if out is None:
            out = {"probs": torch.empty(B, dtype=torch.float32).pin_memory()}
            if fitb:
                out["pred"] = torch.empty(B, dtype=torch.int64).pin_memory()
        cur = torch.cuda.current_stream(self.dev)
        self.copy_stream.wait_stream(cur)
        self.compute_stream.wait_stream(cur)
        for i, lo in enumerate(range(0, B, self.chunk)):
            hi = min(B, lo + self.chunk)
            s = i % self.n_slots
            with torch.cuda.stream(self.copy_stream):
                if i >= self.n_slots:
                    self.copy_stream.wait_event(self._free[s])
                d = {"ids": self._stage(s, "ids", item_ids[lo:hi]), "mask": self._stage(s, "idmask", outfit_mask[lo:hi])}
                if fitb:
                    d["text"] = self._stage(s, "text", target_item_text_embedding[lo:hi])
                    d["cids"] = self._stage(s, "cids", candidate_ids[lo:hi])
                self._ready[s].record(self.copy_stream)
            with torch.cuda.stream(self.compute_stream):
                self.compute_stream.wait_event(self._ready[s])
                enc = {"image_embeddings": image_table, "text_embeddings": text_table, "item_ids": d["ids"]}
                probs = self.model.score_cp(outfit_mask=d["mask"], encoder_input_dict=enc)
                out["probs"][lo:hi].copy_(probs, non_blocking=True)
                if fitb:
                    pred, _, _ = self.model.score_fitb(outfit_mask=d["mask"], target_item_text_embedding=d["text"],
                                                       candidate_item_embedding=(candidate_table, d["cids"]),
                                                       encoder_input_dict=enc)
                    out["pred"][lo:hi].copy_(pred, non_blocking=True)
                self._free[s].record(self.compute_stream)
        cur.wait_stream(self.compute_stream)
        self.compute_stream.synchronize()
        return out


def packed_layout(lengths: torch.Tensor, plan, max_items: int, mask_out: torch.Tensor, ids_out: torch.Tensor) -> torch.Tensor:
    """Host arithmetic of the packed layout (CPU tensors only).  ``lengths (B,)`` int64, ``plan`` = [(lo, hi)] chunk
    boundaries in outfits.  Fills ``mask_out (B, max_items)`` bool (True = padded slot, the reference's convention,
    ``outfit_x_base_processor.py:70-81``) and ``ids_out (B, max_items)`` int32: slot (b, s) of a chunk reads row
    ``off[b] - off[chunk start] + s`` of the chunk's staged rows (slots past the length are masked, whatever their id).
    Returns ``off (B + 1,)``, the exclusive prefix sum of the lengths = each outfit's first row."""
    B = lengths.numel()
    off = torch.zeros(B + 1, dtype=torch.int64)
    torch.cumsum(lengths, 0, out=off[1:])
    slot = torch.arange(max_items, dtype=torch.int64)
    torch.ge(slot[None, :], lengths[:, None], out=mask_out)
    starts = torch.tensor([lo for lo, _ in plan], dtype=torch.int64)
    sizes = torch.tensor([hi - lo for lo, hi in plan], dtype=torch.int64)
    chunk_base = off[starts].repeat_interleave(sizes)             # first row of each outfit's chunk
    ids_out.copy_((off[:B, None] - chunk_base[:, None] + slot[None, :]).to(torch.int32))
    return off


def pack_valid_rows(image_embeddings: torch.Tensor, text_embeddings: torch.Tensor, outfit_mask: torch.Tensor):
    """Padded host batch ``(B, L, dpm)`` x 2 + ``outfit_mask (B, L)`` (True = pad) -> the packed layout of
    ``HostScoringPipeline.score_packed``: ``(image_rows, text_rows, lengths)``.  Valid slots keep their order.
    (A convenience for callers that already hold padded tensors; a collate should build the rows directly.)"""
    keep = ~outfit_mask.bool()
    return (image_embeddings[keep].contiguous(), text_embeddings[keep].contiguous(), keep.sum(-1).to(torch.int32))
