"""CPU: the category-search reference against the reference's own idiom, the category entry points' size
queries and their refusal to run without an sm_100 device, and the host routing of query categories."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/category_oracle.py
from category_oracle import category_search  # noqa: E402
from outfitx_b200 import synth


def test_restatement_equals_grouped_cdist_topk():
    """complementary_item_retrieval_trainer.py:192-249: group the queries by category, then
    topk(cdist(q, category items), k, largest=False) inside each group -- on rows whose distances are
    clearly distinct, so torch.topk's tie order does not matter."""
    n, nq, n_cat, k = 600, 40, 5, 7
    r = np.random.Generator(np.random.PCG64(3))
    gal = synth.make_items(n, 64, seed=4)
    g_cat = r.integers(0, n_cat, n)
    g_cat[g_cat == 4] = 3                              # category 4 is empty
    q = synth.make_queries(nq, 128, seed=5)
    q_cat = r.integers(0, n_cat, nq)
    for metric in ("l2", "dot"):
        idx, score = category_search(q, q_cat, gal, g_cat, k, metric=metric, id_offset=100)
        for c in range(n_cat):
            qs, rows = np.nonzero(q_cat == c)[0], np.nonzero(g_cat == c)[0]
            if len(qs) == 0:
                continue
            if len(rows) == 0:
                assert np.all(idx[qs] == -1) and np.all(np.isneginf(score[qs]))
                continue
            qt, gt = torch.from_numpy(q[qs]).double(), torch.from_numpy(gal[rows]).double()
            d = torch.cdist(qt, gt) if metric == "l2" else -(qt @ gt.T)
            want = torch.topk(d, min(k, len(rows)), largest=False).indices.numpy()
            assert np.array_equal(idx[qs, :want.shape[1]], rows[want] + 100)


def test_category_size_queries_without_gpu():
    from outfitx_b200 import _lib
    L = _lib.lib()
    n, dim = 100_000, 1024
    assert L.ofx_category_gallery_packed_bytes(n, dim, 150) >= n * (dim + 64) * 2
    assert L.ofx_category_gallery_packed_bytes(n, dim, 65536) > L.ofx_category_gallery_packed_bytes(n, dim, 1)
    assert L.ofx_category_gallery_packed_bytes(n, dim, 0) == 0
    assert L.ofx_category_gallery_packed_bytes(n, dim, 65537) == 0     # the documented category limit
    w = L.ofx_category_search_workspace_bytes(dim, 11, 8192, 10)
    assert w > 8192 * (dim + 64) * 2
    # the worst case grows with the number of categories the queries may spread over
    assert L.ofx_category_search_workspace_bytes(dim, 150, 8192, 10) > w
    assert L.ofx_category_search_workspace_bytes(dim, 11, 8192, 64) > w      # longer candidate lists
    assert L.ofx_category_search_workspace_bytes(dim, 11, 8192, 65) == 0     # k out of range
    assert L.ofx_category_search_workspace_bytes(dim, 65537, 8, 10) == 0
    assert L.ofx_category_search_workspace_bytes(dim, 11, 0, 10) > 0


def test_category_entries_refuse_without_sm100():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from outfitx_b200 import _lib
    L = _lib.lib()
    buf = (C.c_uint8 * (1 << 20))()
    p = (C.addressof(buf) + 255) // 256 * 256          # 256-byte aligned host address; never dereferenced
    rc = L.ofx_category_gallery_pack(p, p, 4, 128, 3, p, p, p, p, None)
    assert rc == -3 and b"device" in L.ofx_last_error()   # OFX_E_ARCH
    rc = L.ofx_category_search(p, p, p, p, 3, p, 4, 128, 0, p, p, 2, 10, 1, p, p, p, p, 1 << 19, None)
    assert rc == -3
    rc = L.ofx_category_exact_search(p, p, p, 3, 4, 128, 0, p, p, p, 1, 10, 1, p, p, p, p, 1 << 19, None)
    assert rc == -3
    # argument errors are reported before the device check
    assert L.ofx_category_gallery_pack(p, p, 4, 128, 65537, p, p, p, p, None) == -1
    assert L.ofx_category_search(p, p, p, p, 3, p, 4, 100, 0, p, p, 2, 10, 1, p, p, p, p, 1 << 19, None) == -1


def test_sharded_search_forwards_query_category_only_when_given():
    """ShardedSearch calls the local step exactly as before without categories (five positional arguments),
    and passes query_category through when it is given."""
    from outfitx_b200.search import ShardedSearch
    calls = []

    def local(*args, **kw):
        calls.append((len(args), kw))
        return torch.zeros(2, 3, dtype=torch.int64), torch.zeros(2, 3, dtype=torch.float64)

    s = ShardedSearch(local=local, merge=None)
    s.search(torch.zeros(2, 4), None, 3, "l2", True)
    qc = torch.tensor([0, 1])
    s.search(torch.zeros(2, 4), None, 3, "l2", True, query_category=qc)
    assert calls[0] == (5, {})
    assert calls[1][0] == 5 and calls[1][1]["query_category"] is qc
