"""GPU parity of the category-restricted search (ofx_category_search / ofx_category_exact_search) against the
per-category fp64 oracle (tests/category_oracle.py): indices bit-exact, scores within 1e-13 relative."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/category_oracle.py
from category_oracle import category_search  # noqa: E402
from outfitx_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def _interleaved(sizes, seed):
    """Category ids with the given sizes, in random row order (ids must come back through perm)."""
    cat = np.repeat(np.arange(len(sizes)), sizes)
    _rng(seed).shuffle(cat)
    return cat.astype(np.int64)


def _gallery(n, metric, seed):
    gal = synth.make_items(n, 512, seed=seed)
    if metric == "l2":     # break the |g|^2 == 2 degeneracy so that the bias term matters
        gal = gal * (1.0 + 0.2 * synth.make_queries(n, 1, seed=seed + 1)).astype(np.float32)
    return gal


def _plant_ties(gal, g_cat, n_pairs, seed):
    """Exact copies of rows inside their own category, later in row order: the earlier id must win the tie."""
    r = _rng(seed)
    src = r.choice(len(gal) // 2, n_pairs, replace=False)
    dst = len(gal) // 2 + r.choice(len(gal) // 2, n_pairs, replace=False)
    gal[dst] = gal[src]
    g_cat[dst] = g_cat[src]
    return src


def _search(q, q_cat, gal, g_cat, k, metric="l2", exact=True, id_offset=0, n_cat=None):
    from outfitx_b200.search import Gallery, local_search
    G = Gallery.build(_t(gal), id_offset=id_offset, categories=_t(g_cat), n_categories=n_cat)
    idx, score = local_search(_t(q), G, k, metric, exact, query_category=_t(q_cat))
    torch.cuda.synchronize()
    return idx.cpu().numpy(), score.cpu().numpy()


def _check(got, want):
    assert np.array_equal(got[0], want[0])
    fin = np.isfinite(want[1])
    assert np.array_equal(fin, np.isfinite(got[1]))
    np.testing.assert_allclose(got[1][fin], want[1][fin], rtol=1e-13, atol=1e-11)


def _sizes(n, n_cat):
    """Skewed (Zipf) sizes with empty categories and categories smaller than k; at 150 categories one category
    holds over 90 % of the rows."""
    if n_cat == 1:
        return [n]
    if n_cat == 3:
        return [n - 5, 5, 0]
    w = 1.0 / np.arange(1, n_cat + 1) ** 1.1
    if n_cat >= 150:
        w[0] = 10.0 * w[1:].sum()
    s = np.floor(w / w.sum() * n).astype(np.int64)
    s[[1, n_cat // 2]] = 0                      # empty
    s[[2, n_cat - 1]] = [3, 1]                  # smaller than k
    s[0] += n - s.sum()
    return s.tolist()


@pytest.mark.parametrize("n_cat,k,metric", [
    (1, 10, "l2"), (3, 1, "dot"), (11, 50, "l2"), (11, 10, "dot"), (150, 64, "dot"), (150, 10, "l2")])
def test_category_shapes(n_cat, k, metric):
    n, nq = 60_000, 300
    sizes = _sizes(n, n_cat)
    if n_cat == 150:
        assert sizes[0] > 0.9 * n
    g_cat = _interleaved(sizes, seed=n_cat + 1)
    gal = _gallery(n, metric, seed=n_cat + 2)
    src = _plant_ties(gal, g_cat, 200, seed=n_cat + 3)
    q = synth.make_queries(nq, 1024, seed=n_cat + 4) * np.float32(0.05)
    q_cat = _rng(n_cat + 5).integers(0, n_cat, nq)
    q[:20] = gal[src[:20]] * np.float32(0.7) + q[:20]        # ties near the top of the list
    q_cat[:20] = g_cat[src[:20]]
    got = _search(q, q_cat, gal, g_cat, k, metric, id_offset=12345, n_cat=n_cat)
    want = category_search(q, q_cat, gal, g_cat, k, metric, id_offset=12345)
    _check(got, want)


def test_query_mixes():
    """All queries in one category; queries in categories without rows (padding only)."""
    n, nq, k, n_cat = 30_000, 200, 10, 6
    g_cat = _interleaved([9000, 0, 12000, 8999, 1, 0], seed=1)
    gal = _gallery(n, "l2", seed=2)
    q = synth.make_queries(nq, 1024, seed=3) * np.float32(0.05)
    for q_cat in (np.full(nq, 2), np.where(np.arange(nq) % 2 == 0, 1, 5), np.arange(nq) % n_cat):
        got = _search(q, q_cat, gal, g_cat, k, id_offset=7, n_cat=n_cat)
        _check(got, category_search(q, q_cat, gal, g_cat, k, id_offset=7))
    assert np.all(got[0][q_cat == 1] == -1) and np.all(np.isneginf(got[1][q_cat == 5]))


def test_near_duplicates_reach_the_segment_fallback():
    """Thousands of near-duplicates (closer than bf16 resolves) inside one category: the certificate cannot prove
    the queries that look at them, so the exhaustive fp64 fallback -- restricted to the category's segment --
    answers them, and the result is still the oracle's."""
    from outfitx_b200.search import Gallery, SearchStats, local_search
    n, n_dup, k, n_cat = 200_000, 3000, 10, 7
    gal = synth.make_items(n, 512, seed=11)
    r = _rng(12)
    g_cat = r.integers(1, n_cat, n)
    rows = r.choice(n, size=n_dup, replace=False)
    base = gal[rows[0]].copy()
    gal[rows] = base[None, :] + (r.standard_normal((n_dup, 1024)) * 1e-4).astype(np.float32)
    g_cat[rows] = 0
    g_cat[r.choice(np.setdiff1d(np.arange(n), rows), 20_000, replace=False)] = 0
    q = synth.make_queries(40, 1024, seed=13) * np.float32(0.05)
    q[:8] = base[None, :] * np.float32(0.7) + q[:8] * np.float32(0.1)
    q_cat = np.where(np.arange(40) < 8, 0, r.integers(0, n_cat, 40))
    G = Gallery.build(_t(gal), categories=_t(g_cat))
    SearchStats.reset()
    idx, score, proved = local_search(_t(q), G, k, "l2", True, return_certified=True, query_category=_t(q_cat))
    _check((idx.cpu().numpy(), score.cpu().numpy()), category_search(q, q_cat, gal, g_cat, k))
    assert SearchStats.queries == 40
    assert SearchStats.uncertified > 0
    assert not proved.cpu().numpy()[:8].any()


def test_one_category_equals_flat_search():
    from outfitx_b200.search import Gallery, local_search
    n, nq, k = 70_001, 129, 32
    gal = synth.make_items(n, 512, seed=21, dup=500)
    q = _t(synth.make_queries(nq, 1024, seed=22))
    flat_i, flat_s = local_search(q, Gallery.build(_t(gal), id_offset=5), k)
    G = Gallery.build(_t(gal), id_offset=5, categories=torch.zeros(n, dtype=torch.int32, device=DEV))
    cat_i, cat_s = local_search(q, G, k, query_category=torch.zeros(nq, dtype=torch.int64, device=DEV))
    assert torch.equal(cat_i, flat_i)
    torch.testing.assert_close(cat_s, flat_s, rtol=1e-13, atol=1e-11)


def test_agrees_with_pool_search():
    """The reference's evaluation pools (<= 4096 rows) as the categories of one gallery: the ids are
    pool_search's pool-local ids plus the pool's offset."""
    from outfitx_b200.search import Gallery, PoolSet, local_search, pool_search
    sizes = [3000, 17, 4096, 1, 2500]
    pools = [synth.make_items(s, 512, seed=30 + i) for i, s in enumerate(sizes)]
    off = np.concatenate([[0], np.cumsum(sizes)])
    nq, k = 150, 50
    q = synth.make_queries(nq, 1024, seed=40) * np.float32(0.05)
    q_pool = _rng(41).integers(0, len(sizes), nq)
    for metric in ("l2", "dot"):
        p_i, p_s = pool_search(_t(q), _t(q_pool), PoolSet.build([_t(p) for p in pools]), k, metric)
        G = Gallery.build(_t(np.concatenate(pools)), categories=_t(np.repeat(np.arange(len(sizes)), sizes)))
        c_i, c_s = local_search(_t(q), G, k, metric, query_category=_t(q_pool))
        p_i, c_i = p_i.cpu().numpy(), c_i.cpu().numpy()
        want = np.where(p_i >= 0, p_i + off[q_pool][:, None], -1)
        assert np.array_equal(c_i, want)
        fin = p_i >= 0
        np.testing.assert_allclose(c_s.cpu().numpy()[fin], p_s.cpu().numpy()[fin], rtol=1e-13, atol=1e-11)


def test_emulated_sharding():
    """Per-shard categorised search with global ids, then the merge kernel -- equal to the unsharded search and
    the oracle for worlds 1/2/4/8.  Categories are contiguous runs of rows, so most are absent from most
    shards."""
    from outfitx_b200.search import Gallery, local_search, merge_lists, shard_rows
    n, nq, k, n_cat = 40_003, 200, 10, 11
    g_cat = np.sort(_interleaved(_sizes(n, n_cat), seed=51))
    gal = _gallery(n, "l2", seed=52)
    q = synth.make_queries(nq, 1024, seed=53) * np.float32(0.05)
    q_cat = _rng(54).integers(0, n_cat, nq)
    want = category_search(q, q_cat, gal, g_cat, k)
    full, fc, qq, qc = _t(gal), _t(g_cat), _t(q), _t(q_cat)
    single = local_search(qq, Gallery.build(full, categories=fc, n_categories=n_cat), k, query_category=qc)
    _check((single[0].cpu().numpy(), single[1].cpu().numpy()), want)
    for world in (1, 2, 4, 8):
        parts = []
        for r in range(world):
            lo, hi = shard_rows(n, r, world)
            G = Gallery.build(full[lo:hi], id_offset=lo, categories=fc[lo:hi], n_categories=n_cat)
            parts.append(local_search(qq, G, k, query_category=qc))
        mi, ms = merge_lists(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
        assert torch.equal(mi, single[0]) and torch.equal(ms, single[1])


WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["OFX_ROOT"])
from outfitx_b200 import synth
from outfitx_b200.search import Gallery, cir_search, local_search, shard_rows
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
ok = True
for n, nq, k, metric, n_cat in ((60_001, 300, 10, "l2", 11), (9_000, 64, 50, "dot", 150)):
    gal = synth.make_items(n, 512, seed=n, dup=min(500, n // 4))
    cat = np.sort(np.random.Generator(np.random.PCG64(n)).integers(0, n_cat, n))   # some categories on one rank only
    q = torch.from_numpy(synth.make_queries(nq, 1024, seed=n + 1)).to(dev)
    qc = torch.arange(nq, device=dev) % n_cat
    lo, hi = shard_rows(n, rank, world)
    shard = Gallery.build(torch.from_numpy(gal[lo:hi]).to(dev), id_offset=lo,
                          categories=torch.from_numpy(cat[lo:hi]).to(dev), n_categories=n_cat)
    idx, score = cir_search(q, shard, k=k, metric=metric, query_category=qc)
    whole = Gallery.build(torch.from_numpy(gal).to(dev), categories=torch.from_numpy(cat).to(dev), n_categories=n_cat)
    full_i, full_s = local_search(q, whole, k, metric, query_category=qc)
    same = torch.equal(idx, full_i) and torch.equal(score, full_s)
    flag = torch.tensor([1 if same else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = ok and bool(flag.item())
    if rank == 0:
        print(f"case n={n} nq={nq} k={k} {metric} categories={n_cat}: sharded == single: {bool(flag.item())}", flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_nccl_sharded_category_search_equals_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, OFX_ROOT=ROOT, NCCL_DEBUG="WARN")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("sharded == single: True") == 2


def test_graph_capture_replays_eager():
    from outfitx_b200.search import Gallery, local_search
    n, nq, k, n_cat = 50_000, 500, 10, 11
    g_cat = _interleaved(_sizes(n, n_cat), seed=61)
    G = Gallery.build(_t(_gallery(n, "l2", seed=62)), categories=_t(g_cat))
    q = _t(synth.make_queries(nq, 1024, seed=63))
    qc = _t(_rng(64).integers(0, n_cat, nq))
    eager_i, eager_s = local_search(q, G, k, exact=False, query_category=qc)      # also sizes the workspace
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            g_i, g_s = local_search(q, G, k, exact=False, query_category=qc)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        g_i.fill_(-7)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(g_i, eager_i) and torch.equal(g_s, eager_s)


def test_scale_one_million_rows():
    """4096 queries over 1 M rows in 11 categories; 64 queries are checked against an exhaustive fp64 scan of
    their category."""
    from outfitx_b200.search import Gallery, local_search
    n, nq, k, n_cat = 1_000_000, 4096, 10, 11
    g = torch.Generator(device=DEV).manual_seed(7)
    gal = torch.nn.functional.normalize(torch.randn(n, 2, 512, device=DEV, generator=g), dim=-1).reshape(n, 1024)
    cat = torch.randint(0, n_cat, (n,), device=DEV, generator=g)
    q = torch.randn(nq, 1024, device=DEV, generator=g) * 0.05
    qc = torch.randint(0, n_cat, (nq,), device=DEV, generator=g)
    G = Gallery.build(gal, categories=cat)
    idx, score, proved = local_search(q, G, k, return_certified=True, query_category=qc)
    print(f"certified by the bound alone: {float(proved.float().mean()):.4f} of {nq} queries")
    check = torch.arange(0, nq, nq // 64, device=DEV)
    for c in range(n_cat):
        sel = check[qc[check] == c]
        if sel.numel() == 0:
            continue
        rows = torch.nonzero(cat == c).flatten()
        gc = gal[rows].double()
        s = q[sel].double() @ gc.T - 0.5 * (gc * gc).sum(-1)
        top = torch.topk(s, k, dim=-1)
        assert torch.equal(idx[sel], rows[top.indices])
        torch.testing.assert_close(score[sel], top.values, rtol=1e-12, atol=1e-10)


def test_argument_errors():
    from outfitx_b200.search import Gallery, cir_search, local_search
    gal = _t(synth.make_items(1000, 512, seed=70))
    cat = torch.arange(1000, device=DEV) % 4
    q = _t(synth.make_queries(8, 1024, seed=71))
    qc = torch.arange(8, device=DEV) % 4
    Gc = Gallery.build(gal, categories=cat)
    Gf = Gallery.build(gal)
    assert Gc.n_categories == 4
    with pytest.raises(ValueError, match="query_category"):
        local_search(q, Gc, 10)                                       # categorised gallery, no query categories
    with pytest.raises(ValueError, match="categories"):
        local_search(q, Gf, 10, query_category=qc)                     # flat gallery, query categories
    with pytest.raises(ValueError, match="shape"):
        local_search(q, Gc, 10, query_category=qc[:7])
    with pytest.raises(ValueError, match="integer"):
        local_search(q, Gc, 10, query_category=qc.float())
    with pytest.raises(ValueError, match="CUDA"):
        local_search(q, Gc, 10, query_category=qc.cpu())
    with pytest.raises(ValueError, match="outside"):
        local_search(q, Gc, 10, query_category=qc + 1)
    with pytest.raises(ValueError, match="outside"):
        cir_search(q, Gc, 10, query_category=qc - 1)
    with pytest.raises(ValueError, match="outside"):
        Gallery.build(gal, categories=cat, n_categories=3)
    with pytest.raises(ValueError, match="outside"):
        Gallery.build(gal, categories=cat - 1, n_categories=4)
    with pytest.raises(ValueError, match="n_categories"):
        Gallery.build(gal, categories=cat, n_categories=65537)
    with pytest.raises(ValueError, match="shape"):
        Gallery.build(gal, categories=cat[:999])
    with pytest.raises(ValueError, match="integer"):
        Gallery.build(gal, categories=cat.double())
