"""TEST INFRASTRUCTURE ONLY -- reference of the category-restricted search (``ofx_category_search``).

The reference ranks a CIR query only against the items of its target category
(``complementary_item_retrieval_trainer.py:192-249``: group by category, ``cdist`` -> ``topk(largest=False)``
per group).  Restated on the fp64 oracle ``oracle.restatement.search`` applied per category, with the
category's local row numbers mapped back to gallery ids: ties go to the lowest gallery id, -1 / -inf pad
a list past the category's rows.
"""
import numpy as np

from oracle import restatement as R


def category_search(q, q_cat, gallery, g_cat, k, metric="l2", id_offset=0):
    """-> (idx (nq, k) int64 gallery ids + id_offset, score (nq, k) fp64)."""
    q = np.ascontiguousarray(q, np.float32)
    gallery = np.ascontiguousarray(gallery, np.float32)
    q_cat, g_cat = np.asarray(q_cat), np.asarray(g_cat)
    idx = np.full((len(q), k), -1, np.int64)
    score = np.full((len(q), k), -np.inf, np.float64)
    for c in np.unique(q_cat):
        qs = np.nonzero(q_cat == c)[0]
        rows = np.nonzero(g_cat == c)[0]             # ascending: local order is gallery order
        if len(rows) == 0:
            continue
        kk = min(k, len(rows))
        i, s = R.search(q[qs], gallery[rows], k=kk, metric=metric)
        idx[qs, :kk] = rows[i] + id_offset
        score[qs, :kk] = s
    return idx, score
