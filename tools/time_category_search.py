"""Time the category-restricted search (ofx_category_search) against the flat search of the same gallery.

    python tools/time_category_search.py [--rows 10000000] [--queries 8192] [--k 10] [--reps 5] [--out FILE]

One gallery of --rows random 1024-d items (two L2-normalised 512-d halves, like the bench), exact top-k
(fp64 re-rank + certificate + fallback, the product path), two category distributions:
  (a) 11 equal categories, query categories uniform;
  (b) 150 Zipf-sized categories (size ~ 1/rank), query categories drawn in proportion to size.
The flat search of the same rows is timed in the same process, alternated with (a) and (b), and compared as
a (query x row) rate: a category search of query q covers the N_c rows of its category only.
FLOPs: useful = 2 sum_c nq_c N_c (dim + 64) (the +64 is the bias k-block of the packed rows); padded = what the
tensor cores really run, 2 sum_c groups_c 256 (tiles_c 256) (dim + 64) with groups of two 128-query blocks (CTA
pairs) and 256-row tiles.  Shares are of the data-sheet dense BF16 rate of one B200 (2250 TFLOP/s at 1000 W).
CUDA events; the card's name and power limit are read in the same run.  A 64-query fp64 spot check (exhaustive
torch fp64 scan of each query's category) verifies every distribution.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from outfitx_b200.search import Gallery, SearchStats, local_search  # noqa: E402

PEAK_BF16 = 2250e12
DIM = 1024


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return {"name": name, "nvidia_smi": r.stdout.strip()}
    except (OSError, subprocess.SubprocessError) as e:
        return {"name": name, "nvidia_smi": f"unavailable: {e}"}


def make_gallery(n, gen):
    gal = torch.empty(n, DIM, device="cuda")
    for lo in range(0, n, 1 << 20):
        hi = min(n, lo + (1 << 20))
        x = torch.randn(hi - lo, 2, DIM // 2, device="cuda", generator=gen)
        gal[lo:hi] = torch.nn.functional.normalize(x, dim=-1).reshape(hi - lo, DIM)
    return gal


def distributions(n, nq, gen):
    out = {}
    cat = torch.arange(n, device="cuda") % 11
    out["a_11_equal"] = (cat[torch.randperm(n, device="cuda", generator=gen)],
                         torch.randint(0, 11, (nq,), device="cuda", generator=gen), 11)
    w = 1.0 / torch.arange(1, 151, dtype=torch.float64)
    sizes = torch.floor(w / w.sum() * n).long()
    sizes[0] += n - int(sizes.sum())
    cat = torch.repeat_interleave(torch.arange(150, device="cuda"), sizes.cuda())
    qc = torch.multinomial((sizes.double() / n).cuda(), nq, replacement=True, generator=gen)
    out["b_150_zipf"] = (cat[torch.randperm(n, device="cuda", generator=gen)], qc, 150)
    return out


def flops(cat, qc, n_cat, dim):
    rows = torch.bincount(cat, minlength=n_cat).double().cpu()
    nq_c = torch.bincount(qc, minlength=n_cat).double().cpu()
    useful = 2.0 * float((nq_c * rows).sum()) * (dim + 64)
    groups = torch.where(rows > 0, torch.ceil(nq_c / 256.0), torch.zeros_like(rows))
    padded = 2.0 * float((groups * 256.0 * torch.ceil(rows / 256.0) * 256.0).sum()) * (dim + 64)
    return useful, padded, float((nq_c * rows).sum())


def timed(fn, reps):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def spot_check(gal, cat, q, qc, idx, k, n_check=64):
    sel_all = torch.arange(0, q.shape[0], max(1, q.shape[0] // n_check), device="cuda")[:n_check]
    bad = 0
    for c in torch.unique(qc[sel_all]).tolist():
        sel = sel_all[qc[sel_all] == c]
        rows = torch.nonzero(cat == c).flatten()
        top_i = []
        for lo in range(0, rows.numel(), 1 << 20):      # exhaustive fp64 scan of the category, in chunks
            gc = gal[rows[lo:lo + (1 << 20)]].double()
            s = q[sel].double() @ gc.T - 0.5 * (gc * gc).sum(-1)
            t = torch.topk(s, min(k, s.shape[1]), dim=-1)
            top_i.append((t.values, rows[lo:lo + (1 << 20)][t.indices]))
        v = torch.cat([t[0] for t in top_i], 1)
        i = torch.cat([t[1] for t in top_i], 1)
        o = torch.topk(v, min(k, v.shape[1]), dim=-1).indices
        bad += int((torch.gather(i, 1, o) != idx[sel, :o.shape[1]]).any(-1).sum())
    return sel_all.numel(), bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--queries", type=int, default=8192)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200): there is no CPU measurement")
    gen = torch.Generator(device="cuda").manual_seed(1)
    n, nq, k = a.rows, a.queries, a.k
    gal = make_gallery(n, gen)
    q = torch.randn(nq, DIM, device="cuda", generator=gen) * 0.05
    dists = distributions(n, nq, gen)
    flat = Gallery.build(gal)
    cats = {name: (Gallery.build(gal, categories=c, n_categories=m), c, qc, m) for name, (c, qc, m) in dists.items()}
    runs = {"flat": lambda: local_search(q, flat, k)}
    for name, (G, c, qc, m) in cats.items():
        runs[name] = (lambda G=G, qc=qc: local_search(q, G, k, query_category=qc))
    for fn in runs.values():
        timed(fn, a.warmup)
    times = {name: [] for name in runs}
    stats = {}
    for _ in range(a.reps):                 # alternated: one call of each per round
        for name, fn in runs.items():
            SearchStats.reset()
            times[name] += timed(fn, 1)
            stats[name] = (SearchStats.queries, SearchStats.uncertified)
    res = {"card": card(), "rows": n, "queries": nq, "k": k, "reps": a.reps}
    flat_ms = min(times["flat"])
    res["flat"] = {"ms_min": flat_ms, "ms_all": times["flat"], "queries_per_s": nq / (flat_ms * 1e-3),
                   "query_rows_per_s": nq * n / (flat_ms * 1e-3), "uncertified": stats["flat"][1]}
    for name, (G, c, qc, m) in cats.items():
        ms = min(times[name])
        useful, padded, qr = flops(c, qc, m, DIM)
        idx, _ = local_search(q, G, k, query_category=qc)
        n_chk, bad = spot_check(gal, c, q, qc, idx, k)
        res[name] = {"ms_min": ms, "ms_all": times[name], "queries_per_s": nq / (ms * 1e-3),
                     "query_rows_per_s": qr / (ms * 1e-3), "rate_vs_flat": (qr / (ms * 1e-3)) / (nq * n / (flat_ms * 1e-3)),
                     "useful_tflops": useful / (ms * 1e-3) / 1e12, "useful_share_of_peak": useful / (ms * 1e-3) / PEAK_BF16,
                     "padded_tflops": padded / (ms * 1e-3) / 1e12, "padded_share_of_peak": padded / (ms * 1e-3) / PEAK_BF16,
                     "padded_over_useful": padded / useful, "uncertified": stats[name][1],
                     "spot_check": f"{n_chk - bad}/{n_chk} queries equal to the exhaustive fp64 scan of their category",
                     "spot_check_failures": bad}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if all(res[name]["spot_check_failures"] == 0 for name in cats) else 1)


if __name__ == "__main__":
    main()
