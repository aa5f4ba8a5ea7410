"""CIR gallery search: exact top-k by L2 distance or dot product, single GPU or gallery-sharded.

Restates the reference's retrieval idiom ``torch.cdist(Q, G)`` -> ``torch.topk(k, largest=False)``
(``src/trains/trainers/complementary_item_retrieval_trainer.py:240-242``,
``src/demo/app.py:189-190``) as the arg-max of ``q.g - 0.5|g|^2`` ('l2', same ranking as
ascending distance) or ``q.g`` ('dot'); ties resolve to the lowest gallery index.

Sharding (no reference counterpart -- its inference is single-GPU,
``complementary_item_retrieval_trainer.py:350-351``): rank r owns gallery rows
``[r*ceil(N/W), ...)``, every rank searches its shard for ALL queries, the per-shard
``(nq, k)`` lists are exchanged with ONE all-gather and merged by ``(-score, index)``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib

_METRIC = {"dot": _lib.METRIC_DOT, "l2": _lib.METRIC_L2}
MAX_K = 64


def shard_rows(n_rows: int, rank: int, world: int) -> Tuple[int, int]:
    """Row range [lo, hi) of the gallery owned by `rank` (contiguous, ceil-divided)."""
    per = (n_rows + world - 1) // world
    lo = min(rank * per, n_rows)
    return lo, min(lo + per, n_rows)


class Gallery:
    """A gallery shard resident in HBM: bf16 rows + 0.5|g|^2 for the tensor-core pass and
    (optionally) the fp32 rows for the exact fp64 re-rank.

    A categorised gallery (``build(..., categories=...)``) is searched per category: its packed rows are
    sorted stably by category, ``perm`` maps a packed row to the shard row, ``seg_off`` (n_categories + 1)
    delimits each category's packed rows and ``cat_max`` holds each category's max 0.5|g|^2 (the
    certificate's bound).  ``rows_f32`` stays in the caller's row order."""

    def __init__(self, packed: torch.Tensor, n_rows: int, dim: int, id_offset: int,
                 rows_f32: Optional[torch.Tensor], n_categories: Optional[int] = None,
                 perm: Optional[torch.Tensor] = None, seg_off: Optional[torch.Tensor] = None,
                 cat_max: Optional[torch.Tensor] = None):
        self.packed, self.n_rows, self.dim = packed, n_rows, dim
        self.id_offset, self.rows_f32 = id_offset, rows_f32
        self.n_categories, self.perm, self.seg_off, self.cat_max = n_categories, perm, seg_off, cat_max

    @property
    def device(self):
        return self.packed.device

    @classmethod
    def build(cls, embeddings: torch.Tensor, id_offset: int = 0, keep_fp32: bool = True,
              categories: Optional[torch.Tensor] = None, n_categories: Optional[int] = None) -> "Gallery":
        """embeddings: (n_rows, dim) fp32 CUDA tensor holding THIS rank's rows.
        categories: optional (n_rows,) integer CUDA tensor of category ids in [0, n_categories); the gallery is
        then searched per category (``local_search(..., query_category=...)``).  n_categories defaults to
        max id + 1; give it explicitly when shards of one catalogue are built separately, so that every shard
        accepts the same query categories.  Checking the ids costs one small device->host sync."""
        if not embeddings.is_cuda:
            raise RuntimeError("gallery embeddings must be a CUDA tensor: outfitx_b200 has no CPU path")
        g = embeddings.detach().to(torch.float32).contiguous()
        n, dim = g.shape
        L = _lib.lib()
        stream = torch.cuda.current_stream(g.device).cuda_stream
        if categories is not None:
            cat, n_cat = _gallery_categories(categories, n, g.device, n_categories)
            nbytes = L.ofx_category_gallery_packed_bytes(n, dim, n_cat)
            packed = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=g.device)
            perm = torch.empty(n, dtype=torch.int32, device=g.device)
            seg_off = torch.empty(n_cat + 1, dtype=torch.int64, device=g.device)
            cat_max = torch.empty(n_cat, dtype=torch.float32, device=g.device)
            with torch.cuda.device(g.device):
                _lib.check(L.ofx_category_gallery_pack(g.data_ptr(), cat.data_ptr(), n, dim, n_cat, packed.data_ptr(),
                                                       perm.data_ptr(), seg_off.data_ptr(), cat_max.data_ptr(), stream))
                if not keep_fp32:
                    torch.cuda.current_stream(g.device).synchronize()
            return cls(packed, n, dim, id_offset, g if keep_fp32 else None, n_cat, perm, seg_off, cat_max)
        if n_categories is not None:
            raise ValueError("n_categories is given without categories")
        nbytes = L.ofx_gallery_packed_bytes(n, dim)
        packed = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=g.device)
        with torch.cuda.device(g.device):
            _lib.check(L.ofx_gallery_pack(g.data_ptr(), n, dim, packed.data_ptr(), stream))
            if not keep_fp32:
                torch.cuda.current_stream(g.device).synchronize()
        return cls(packed, n, dim, id_offset, g if keep_fp32 else None)

    @classmethod
    def build_sharded(cls, embeddings: torch.Tensor, rank: int, world: int, keep_fp32: bool = True,
                      categories: Optional[torch.Tensor] = None, n_categories: Optional[int] = None):
        """Takes the FULL gallery (n, dim) and keeps rank's slice -- for tests / small galleries;
        large galleries should be generated or loaded shard by shard and passed to build()."""
        lo, hi = shard_rows(embeddings.shape[0], rank, world)
        if categories is None:
            return cls.build(embeddings[lo:hi], id_offset=lo, keep_fp32=keep_fp32, n_categories=n_categories)
        if n_categories is None and categories.numel():
            n_categories = int(categories.max()) + 1          # of the whole catalogue, the same on every rank
        return cls.build(embeddings[lo:hi], id_offset=lo, keep_fp32=keep_fp32, categories=categories[lo:hi],
                         n_categories=n_categories)


MAX_CATEGORIES = 65536


def _check_ids(ids: torch.Tensor, n: int, dev, what: str) -> None:
    if not isinstance(ids, torch.Tensor) or not ids.is_cuda or ids.device != torch.device(dev):
        raise ValueError(f"{what} must be a CUDA tensor on {dev}")
    if ids.shape != (n,):
        raise ValueError(f"{what} must have shape ({n},), got {tuple(ids.shape)}")
    if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
        raise ValueError(f"{what} must be an integer tensor, got {ids.dtype}")


def _gallery_categories(categories, n: int, dev, n_categories: Optional[int]):
    _check_ids(categories, n, dev, "categories")
    if n_categories is None:
        n_categories = int(categories.max()) + 1 if n else 1
    if not 1 <= n_categories <= MAX_CATEGORIES:
        raise ValueError(f"n_categories must be in [1, {MAX_CATEGORIES}], got {n_categories}")
    if n and (int(categories.min()) < 0 or int(categories.max()) >= n_categories):
        raise ValueError(f"categories holds an id outside [0, {n_categories})")
    return categories.to(torch.int32).contiguous(), n_categories


def _query_categories(query_category, nq: int, dev, n_categories: int) -> torch.Tensor:
    _check_ids(query_category, nq, dev, "query_category")
    # the range check reads two numbers back; inside CUDA-graph capture it is skipped (the kernels answer an
    # out-of-range category with padding and never read outside the gallery)
    if nq and not torch.cuda.is_current_stream_capturing():
        if int(query_category.min()) < 0 or int(query_category.max()) >= n_categories:
            raise ValueError(f"query_category holds an id outside [0, {n_categories})")
    return query_category.to(torch.int32).contiguous()


class _Workspace:
    buf: Optional[torch.Tensor] = None


def _workspace(nbytes: int, dev) -> torch.Tensor:
    b = _Workspace.buf
    if b is None or b.device != dev or b.numel() < nbytes:
        _Workspace.buf = b = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
    return b


class SearchStats:
    """Counters of the exactness certificate (process-wide, for tests and the bench line)."""
    queries = 0          # exact-mode queries searched
    uncertified = 0      # of those, how many the bound could not prove and went to the exhaustive fallback

    @classmethod
    def reset(cls):
        cls.queries = cls.uncertified = 0


@torch.no_grad()
def local_search(queries: torch.Tensor, gallery: Gallery, k: int = 10, metric: str = "l2",
                 exact: bool = True, return_certified: bool = False, query_category: Optional[torch.Tensor] = None):
    """Top-k of every query over one shard -> (idx (nq,k) int64 GLOBAL ids, score (nq,k) fp64).

    exact=True re-scores the tensor-core pass's candidates in fp64 from the fp32 rows and PROVES, per query,
    that nothing the bf16 pass dropped can reach the k-th best exact score (rigorous bf16 error bound, see
    ``ofx_topk_search``); the few queries it cannot prove (gallery rows closer than bf16 resolves) are
    re-searched exhaustively in fp64 (``ofx_exact_search``), so the indices ARE those of an fp64 exhaustive
    search.  Reading the certificate flags costs one small device->host sync per call.
    exact=False returns the bf16-pass ranking (no certificate, no sync).
    return_certified=True appends the (nq,) bool tensor "proved by the bound alone".
    query_category: (nq,) integer CUDA tensor, required for (and only for) a gallery built with categories:
    query q is ranked against the shard's rows of category query_category[q] only
    (``ofx_category_search``); -1 / -inf pad a list past the category's rows here."""
    if metric not in _METRIC:
        raise ValueError(f"metric must be 'dot' or 'l2', got {metric!r}")
    if not 1 <= k <= MAX_K:
        raise ValueError(f"k must be in [1, {MAX_K}]")
    if not queries.is_cuda:
        raise RuntimeError("queries must be a CUDA tensor: outfitx_b200 has no CPU path")
    q = queries.detach().to(torch.float32).contiguous()
    if q.dim() != 2 or q.shape[1] != gallery.dim:
        raise ValueError(f"queries must be (nq, {gallery.dim})")
    if exact and gallery.rows_f32 is None:
        raise ValueError("exact search needs Gallery.build(..., keep_fp32=True)")
    if gallery.n_categories is not None and query_category is None:
        raise ValueError("a gallery built with categories is searched with query_category")
    if gallery.n_categories is None and query_category is not None:
        raise ValueError("query_category needs a gallery built with categories")
    nq, dev = q.shape[0], q.device
    qc = _query_categories(query_category, nq, dev, gallery.n_categories) if query_category is not None else None
    L = _lib.lib()
    score = torch.empty(nq, k, dtype=torch.float64, device=dev)
    idx = torch.empty(nq, k, dtype=torch.int64, device=dev)
    proved = torch.zeros(nq, dtype=torch.bool, device=dev)
    if nq == 0:
        return (idx, score, proved) if return_certified else (idx, score)
    cert = torch.zeros(nq, dtype=torch.uint8, device=dev) if exact else None
    g32 = gallery.rows_f32.data_ptr() if exact else None
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream(dev).cuda_stream
        if qc is None:
            nbytes = L.ofx_search_workspace_bytes(gallery.n_rows, gallery.dim, nq, k)
            ws = _workspace(nbytes, dev)
            _lib.check(L.ofx_topk_search(
                gallery.packed.data_ptr(), g32, gallery.n_rows, gallery.dim, gallery.id_offset, q.data_ptr(), nq, k,
                _METRIC[metric], score.data_ptr(), idx.data_ptr(), cert.data_ptr() if exact else None, ws.data_ptr(),
                ws.numel(), st))
        else:
            nbytes = L.ofx_category_search_workspace_bytes(gallery.dim, gallery.n_categories, nq, k)
            ws = _workspace(nbytes, dev)
            _lib.check(L.ofx_category_search(
                gallery.packed.data_ptr(), gallery.perm.data_ptr(), gallery.seg_off.data_ptr(),
                gallery.cat_max.data_ptr(), gallery.n_categories, g32, gallery.n_rows, gallery.dim, gallery.id_offset,
                q.data_ptr(), qc.data_ptr(), nq, k, _METRIC[metric], score.data_ptr(), idx.data_ptr(),
                cert.data_ptr() if exact else None, ws.data_ptr(), ws.numel(), st))
        if exact:
            proved = cert.bool()
            sel = torch.nonzero(~proved).flatten().to(torch.int32)       # the one host sync of an exact search
            SearchStats.queries += nq
            SearchStats.uncertified += int(sel.numel())
            if sel.numel():
                nb = L.ofx_exact_search_workspace_bytes(gallery.n_rows, sel.numel(), k)
                ws2 = torch.empty(max(nb, 256), dtype=torch.uint8, device=dev)
                if qc is None:
                    _lib.check(L.ofx_exact_search(
                        gallery.rows_f32.data_ptr(), gallery.n_rows, gallery.dim, gallery.id_offset, q.data_ptr(),
                        sel.data_ptr(), sel.numel(), k, _METRIC[metric], score.data_ptr(), idx.data_ptr(), None,
                        ws2.data_ptr(), ws2.numel(), st))
                else:
                    _lib.check(L.ofx_category_exact_search(
                        gallery.rows_f32.data_ptr(), gallery.perm.data_ptr(), gallery.seg_off.data_ptr(),
                        gallery.n_categories, gallery.n_rows, gallery.dim, gallery.id_offset, q.data_ptr(),
                        qc.data_ptr(), sel.data_ptr(), sel.numel(), k, _METRIC[metric], score.data_ptr(),
                        idx.data_ptr(), None, ws2.data_ptr(), ws2.numel(), st))
    return (idx, score, proved) if return_certified else (idx, score)


@torch.no_grad()
def merge_lists(idx: torch.Tensor, score: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(R, nq, k') lists -> (nq, k) by (-score, idx); idx < 0 marks padding."""
    R, nq, kk = idx.shape
    if not idx.is_cuda:
        raise RuntimeError("lists must be CUDA tensors: outfitx_b200 has no CPU path")
    if kk != k:
        raise ValueError("merge_lists expects per-shard lists of length k")
    out_i = torch.empty(nq, k, dtype=torch.int64, device=idx.device)
    out_s = torch.empty(nq, k, dtype=torch.float64, device=idx.device)
    with torch.cuda.device(idx.device):
        _lib.check(_lib.lib().ofx_topk_merge(
            score.contiguous().data_ptr(), idx.contiguous().data_ptr(), R, nq, k, out_s.data_ptr(),
            out_i.data_ptr(), torch.cuda.current_stream(idx.device).cuda_stream))
    return out_i, out_s


class ShardedSearch:
    """Gallery-sharded search over a torch.distributed process group (one process per GPU).

    `local` and `merge` are the two device steps; they are injectable so the host-side exchange
    logic can be exercised on CPU with gloo (tests/test_sharded_host.py)."""

    def __init__(self, group=None, local=local_search, merge=merge_lists):
        self.group, self._local, self._merge = group, local, merge

    def search(self, queries, gallery, k: int = 10, metric: str = "l2", exact: bool = True, query_category=None):
        import torch.distributed as dist
        if query_category is None:
            idx, score = self._local(queries, gallery, k, metric, exact)
        else:
            idx, score = self._local(queries, gallery, k, metric, exact, query_category=query_category)
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world == 1:
            return idx, score
        # one collective: ids and the fp64 scores' bit patterns travel as one int64 payload
        payload = torch.stack([idx, score.view(torch.int64)]).contiguous()       # (2, nq, k)
        gathered = torch.empty((world * 2,) + tuple(idx.shape), dtype=torch.int64, device=idx.device)
        dist.all_gather_into_tensor(gathered, payload, group=self.group)   # concatenated along dim 0
        gathered = gathered.view((world, 2) + tuple(idx.shape))
        all_i = gathered[:, 0].contiguous()
        all_s = gathered[:, 1].contiguous().view(torch.float64)
        return self._merge(all_i, all_s, k)


def cir_search(queries, gallery: Gallery, k: int = 10, metric: str = "l2", exact: bool = True,
               group=None, query_category=None):
    """Top-k gallery items per query.  With an initialised process group the gallery is taken to
    be sharded across its ranks (each rank passes its own shard and the same queries).  With a
    categorised gallery, query_category (nq,) picks the category each query is ranked in -- the
    reference's per-category retrieval (complementary_item_retrieval_trainer.py:192-249)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        return ShardedSearch(group).search(queries, gallery, k, metric, exact, query_category=query_category)
    return local_search(queries, gallery, k, metric, exact, query_category=query_category)


# ---------------------------------------------------------------------------------------------
# Per-category candidate pools + Recall@k (SURVEY.md N1)
# ---------------------------------------------------------------------------------------------
MAX_POOL_ROWS = 4096
MAX_POOL_K = 64


class PoolSet:
    """The reference's ``candidate_pools`` (one pool of <= 3000 item embeddings per category,
    ``polyvore_complementary_item_retrieval_dataset.py:111-153``) resident in HBM: all pools
    concatenated into one ``(total_rows, dim)`` fp32 matrix plus row offsets."""

    def __init__(self, rows: torch.Tensor, offsets: torch.Tensor, sizes):
        self.rows, self.offsets, self.sizes = rows, offsets, list(sizes)

    @property
    def n_pools(self) -> int:
        return len(self.sizes)

    @classmethod
    def build(cls, pools) -> "PoolSet":
        """pools: sequence of ``(n_c, dim)`` CUDA fp32 tensors (pool c = category c)."""
        if len(pools) == 0:
            raise ValueError("need at least one pool")
        if any(not p.is_cuda for p in pools):
            raise RuntimeError("pools must be CUDA tensors: outfitx_b200 has no CPU path")
        sizes = [int(p.shape[0]) for p in pools]
        if max(sizes) > MAX_POOL_ROWS or min(sizes) < 1:
            raise ValueError(f"pools hold 1..{MAX_POOL_ROWS} rows")
        rows = torch.cat([p.detach().to(torch.float32) for p in pools]).contiguous()
        off = torch.zeros(len(sizes) + 1, dtype=torch.int64)
        off[1:] = torch.tensor(sizes, dtype=torch.int64).cumsum(0)
        return cls(rows, off.to(rows.device), sizes)


@torch.no_grad()
def pool_search(queries: torch.Tensor, query_pool: torch.Tensor, pools: PoolSet, k: int = 50,
                metric: str = "l2") -> Tuple[torch.Tensor, torch.Tensor]:
    """Top-k of every query inside ITS pool -> (idx (nq,k) int64 pool-local, -1 past the pool size;
    score (nq,k) fp64).  Same ranking as ``torch.topk(torch.cdist(q, pool), k, largest=False)``
    (``complementary_item_retrieval_trainer.py:240-242``), exact, ties to the lowest index."""
    if metric not in _METRIC:
        raise ValueError(f"metric must be 'dot' or 'l2', got {metric!r}")
    if not 1 <= k <= MAX_POOL_K:
        raise ValueError(f"k must be in [1, {MAX_POOL_K}]")
    if not queries.is_cuda:
        raise RuntimeError("queries must be a CUDA tensor: outfitx_b200 has no CPU path")
    q = queries.detach().to(torch.float32).contiguous()
    qp = query_pool.to(device=q.device, dtype=torch.int32).contiguous()
    if q.dim() != 2 or q.shape[1] != pools.rows.shape[1] or qp.shape != (q.shape[0],):
        raise ValueError("queries must be (nq, dim) and query_pool (nq,)")
    nq = q.shape[0]
    if nq and (int(qp.min()) < 0 or int(qp.max()) >= pools.n_pools):
        raise ValueError("query_pool holds a pool index out of range")
    idx = torch.empty(nq, k, dtype=torch.int64, device=q.device)
    score = torch.empty(nq, k, dtype=torch.float64, device=q.device)
    if nq == 0:
        return idx, score
    with torch.cuda.device(q.device):
        _lib.check(_lib.lib().ofx_pool_search(
            pools.rows.data_ptr(), pools.offsets.data_ptr(), pools.n_pools, max(pools.sizes), q.data_ptr(),
            qp.data_ptr(), nq, q.shape[1], k, _METRIC[metric], score.data_ptr(), idx.data_ptr(),
            torch.cuda.current_stream(q.device).cuda_stream))
    return idx, score


def recall_at_k(topk_idx: torch.Tensor, gt_idx: torch.Tensor, top_k_list=(1, 5, 10, 15, 30, 50)) -> dict:
    """``Recall@k`` exactly as ``compute_recall_metrics`` scores it
    (``complementary_item_retrieval_trainer.py:244-249``): the fraction of queries whose
    ground-truth pool index is among the first k retrieved indices."""
    gt = gt_idx.to(topk_idx.device).view(-1, 1)
    out = {}
    for k in top_k_list:
        if k > topk_idx.shape[1]:
            raise ValueError(f"Recall@{k} needs at least {k} retrieved indices")
        out[f"Recall@{k}"] = float((topk_idx[:, :k] == gt).any(dim=-1).float().mean().item()) if gt.numel() else 0.0
    return out


def load_embedding_pickles(paths, device=None):
    """The reference's precomputed-embedding wire format (SURVEY.md N3): each file is
    ``pickle.dump({'ids': [int], 'embeddings': np.float32 (N, 2*dim_per_modality)})`` written by
    ``precompute_embedding_script.py:47-53`` as ``{model_name}_embedding_subset_{rank}.pkl`` and read
    back by ``compatibility_prediction_trainer.py:329-349`` / ``demo/app.py:51-71``.
    -> (ids int64 (N,), embeddings fp32 (N, 2*dpm) [on `device` if given], id -> row dict).
    The text embedding of an item is the second half of its row (``polyvore_item_dataset.py:75``)."""
    import pickle

    import numpy as np
    ids, embs = [], []
    for path in paths:
        with open(path, "rb") as f:
            d = pickle.load(f)
        ids.extend(int(i) for i in d["ids"])
        embs.append(np.asarray(d["embeddings"], dtype=np.float32))
    emb = torch.from_numpy(np.concatenate(embs, axis=0))
    if len(ids) != emb.shape[0]:
        raise ValueError("ids and embeddings disagree in length")
    if device is not None:
        emb = emb.to(device)
    return torch.tensor(ids, dtype=torch.int64), emb, {i: r for r, i in enumerate(ids)}
