#!/usr/bin/env python
"""Benchmark of the outfit-scoring hot path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--skip cir,cir3,large,fp32]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on rank 0.  Primary metric: CP outfits/s on BASELINE.json configs[1]
(CP + FITB(4 candidates) scoring, 8192 outfits per GPU, bf16, mean fusion; weak scaling, no
collective).  The same line carries one object per remaining config, each with its own `roofline`,
`cpu_baseline` and a `verified` flag computed OUTSIDE the timed region against an independent check:

  cir    configs[3]: 8192 queries, exact top-10 over a 10 M-item gallery sharded across the N GPUs with one
         NCCL all-gather (strong scaling); verified against the exhaustive fp64 scan of 64 queries.
  cir3   configs[2] (N = 1 only): 4096 ENCODER-PRODUCED queries (d_model 1024 CIR forward) + exact top-10 over
         1 M items, embed + search timed together.
  large  configs[4] (N = 1 only): large-encoder CP sweep, d_model 1024, 16 items, batch 256 .. 32768.
  fp32   (N = 1 only) the headline step with precision="fp32": linear layers as bf16 hi / lo split GEMMs on tcgen05.

`--impl reference` times the reference's CPU path (oracle/torch_port.py: the stock torch modules the
reference itself is built from -- the reference is pure Python and cannot travel to the GPU box) on the host
cores for the same metric.

`--dump-outputs DIR` writes what the primary step returned in its last timed step on rank 0 (CP probabilities,
FITB argmin, FITB distances, CIR query embeddings) as DIR/<name>.npy, so that two builds can be compared output for
output: the inputs are seeded, identical from run to run for the same arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: everything libraries print to fd 1 (e.g. NCCL's version
# banner) is sent to stderr instead, and the result line goes to the saved descriptor.
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

from outfitx_b200 import synth  # noqa: E402

D_MODEL, D_EMBED, DPM, F_FFN, N_LAYERS = 512, 1024, 512, 2024, 6
N_CAND, TOPK = 4, 10


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return {"burst": float(p["bf16_tflops"]), "sustained": float(p["bf16_tflops_sustained"]),
                "hbm": float(p["hbm_gbs"]), "source": "measured"}
    except Exception:
        return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the committed ncu --set full
    capture of the SAME shipped kernel (profiles/r2_traffic.json, written by tools/ncu_summary.py), else None:
    the number is never a constant in this file."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        e = t.get(kernel_key)
        return (int(e["dram_bytes"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


def flops_alg(n, dm=D_MODEL, f=F_FFN, de=D_EMBED, task="cp"):
    """Minimum exact work per outfit with n valid items (SURVEY.md 8d): layers 0-4 dense over the
    1+n valid tokens, layer 5 pruned to the prefix-token query row; padding never counted."""
    n = np.asarray(n, np.float64)
    s = 1.0 + n
    dense = 5 * s * (8 * dm * dm + 4 * dm * f + 4 * s * dm)
    last = s * 4 * dm * dm + 2 * dm * dm + 4 * s * dm + 2 * dm * dm + 4 * dm * f
    head = 2 * dm if task == "cp" else (2 * dm * de + (3 * N_CAND * de if task == "fitb" else 0))
    return dense + last + head


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.15)        # the first sample takes ~100 ms to appear; keep it out of the timed region's start
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw)}


def timed(fn, steps, warmup, dist_ok, dev, sampler=None):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, CUDA events on the
    launching stream, MAX over ranks.  -> total ms."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    if dist_ok:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.__enter__()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    if dist_ok:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if sampler:
        sampler.__exit__()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist_ok:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def time_ffn_block(L, rows, dev, reps=20):
    """ofx_ffn_block_ln_bf16 -- the form layers 0-4 of the step launch: the fused FFN block that also emits
    norm1 of the next layer -- on `rows` token rows (d_model 512, d_ffn 2024 padded to 2048), inputs rotated
    over 4 buffers (4 x rows x 2 KB > L2).  Algorithmic flops = 4 * rows * 512 * 2024 (the padded columns and
    the LayerNorms are not counted); algorithmic HBM bytes = rows * 5 KB (fp32 row in, fp32 row out, bf16
    LayerNorm row out)."""
    from outfitx_b200 import _lib
    g = torch.Generator(device=dev).manual_seed(11)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    ln_w, ln_b = 1.0 + 0.1 * r(D_MODEL), 0.1 * r(D_MODEL)
    w1 = (r(2048, D_MODEL) / D_MODEL ** 0.5); w1[F_FFN:] = 0
    w2 = (r(D_MODEL, 2048) / 2048 ** 0.5); w2[:, F_FFN:] = 0
    b1 = 0.1 * r(2048); b1[F_FFN:] = 0
    b2 = 0.1 * r(D_MODEL)
    w1, w2 = w1.to(torch.bfloat16).contiguous(), w2.to(torch.bfloat16).contiguous()
    bufs = [r(rows, D_MODEL) for _ in range(4)]
    st = torch.cuda.current_stream(dev).cuda_stream
    h_next = torch.empty(rows, D_MODEL, device=dev, dtype=torch.bfloat16)
    ws = torch.empty(max(int(L.ofx_ffn_block_workspace_bytes(rows, D_MODEL, 2048)), 256), dtype=torch.uint8, device=dev)

    def run(x):
        _lib.check(L.ofx_ffn_block_ln_bf16(x.data_ptr(), rows, D_MODEL, 2048, ln_w.data_ptr(), ln_b.data_ptr(),
                                           w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                           h_next.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                                           ws.data_ptr(), ws.numel(), st))
    for x in bufs:
        run(x)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        run(bufs[i % 4])
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    flops = 4.0 * rows * D_MODEL * F_FFN
    return {"kernel": "ffn_block_kernel", "rows": rows, "us_per_launch": ms * 1e3, "flops_per_launch": flops,
            "tflops": flops / (ms * 1e-3) / 1e12}


def make_cp_inputs(batch, dev, seed):
    """configs[1] inputs: raw (un-normalised) 512-d CLIP image / text embeddings per item,
    n ~ U{2..16} valid items left-aligned, 256-d target text, 4 FITB candidates of 1024-d."""
    g = torch.Generator(device=dev).manual_seed(seed)
    img = torch.randn(batch, 16, DPM, device=dev, generator=g)
    txt = torch.randn(batch, 16, DPM, device=dev, generator=g)
    lengths = synth.make_lengths(batch, seed + 1)
    mask = torch.from_numpy(synth.make_mask(lengths)).to(dev)
    text = torch.nn.functional.normalize(torch.randn(batch, D_MODEL // 2, device=dev, generator=g), dim=-1)
    cand = torch.randn(batch, N_CAND, 2, DPM, device=dev, generator=g)
    cand = torch.nn.functional.normalize(cand, dim=-1).reshape(batch, N_CAND, 2 * DPM).contiguous()
    return img, txt, mask, text, cand, lengths


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, seed=0):
    """Writes `arrays` (name -> tensor with one row per outfit) as DIR/<name>.npy, float64 where the tensor is
    float64 and float32 otherwise.  Above DUMP_BYTES in all, every array keeps the same fixed, seeded sample of
    rows (ascending), and their row numbers are written as rows.npy."""
    host = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    host = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in host.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(v.nbytes // max(n, 1) for v in host.values())
    budget = DUMP_BYTES - 4096                  # room for the .npy headers
    if n * row_bytes > budget:
        keep = budget // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        host = {k: v[rows] for k, v in host.items()}
        host["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def make_model(dev, d_model=D_MODEL, precision="bf16"):
    import outfitx_b200 as o
    method = "mean" if d_model == 512 else "concat"
    cfg = o.OutfitXConfig(item_encoder=o.ItemEncoderConfig(type="clip", aggregation_method=method))
    m = o.OutfitX(cfg, precision=precision)
    sd = synth.make_state_dict(d_model, D_EMBED, seed=0)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return m.to(dev), sd


def make_gallery_shard(n_total, rank, world, dev, chunk=500_000):
    """Rows [lo, hi) of the synthetic gallery: per-modality-normalised halves (|g|^2 = 2)."""
    from outfitx_b200.search import shard_rows
    lo, hi = shard_rows(n_total, rank, world)
    out = torch.empty(hi - lo, 2 * DPM, dtype=torch.float32, device=dev)
    for c0 in range(lo, hi, chunk):
        c1 = min(hi, c0 + chunk)
        g = torch.Generator(device=dev).manual_seed(5 * 2 ** 32 + c0)
        x = torch.randn(c1 - c0, 2, DPM, device=dev, generator=g)
        out[c0 - lo:c1 - lo] = torch.nn.functional.normalize(x, dim=-1).reshape(c1 - c0, 2 * DPM)
    return out, lo


# ------------------------------------------------------------------------------------------ CPU legs (oracle)
def cpu_cp_run(sd, img, txt, mask, text, cand, reps=2):
    """The reference's CPU path (stock torch modules, fp32, all host threads) on the GIVEN host tensors:
    mean fusion, CP logits -> sigmoid, CIR query -> cdist -> argmin.  -> (outfits/s, threads, probs, pred, dists)."""
    from oracle import torch_port
    torch.set_num_threads(os.cpu_count() or 1)
    port = torch_port.ReferencePort.from_numpy(sd)
    method = "mean" if sd["outfit_token"].shape[0] == img.shape[-1] else "concat"
    emb = synth.fuse(img.numpy(), txt.numpy(), method)
    emb[mask.numpy()] = 0.0
    emb = torch.from_numpy(emb)
    best, keep = float("inf"), None
    for r in range(reps + 1):       # pass 0 is the warm-up (and the only pass when reps = 0: results only)
        t0 = time.perf_counter()
        probs = torch.sigmoid(port.cp(emb, mask).float())[:, 0]
        pred = dists = None
        if text is not None:
            q = port.cir(emb, mask, text)
            pred, dists = torch_port.fitb(q, cand)
        dt = time.perf_counter() - t0
        if r > 0 or reps == 0:
            best = min(best, dt)
        keep = (probs, pred, dists)
    return img.shape[0] / best, torch.get_num_threads(), keep[0], keep[1], keep[2]


def cpu_cp_synthetic(sd, sample, seed, reps=1):
    img, txt = synth.make_modalities(sample, DPM, seed)
    mask = synth.make_mask(synth.make_lengths(sample, seed + 1))
    text = synth.make_text_prefix(sample, D_MODEL // 2, seed + 2)
    cand = synth.make_items(sample * N_CAND, DPM, seed + 3).reshape(sample, N_CAND, 2 * DPM)
    t = torch.from_numpy
    v, threads, *_ = cpu_cp_run(sd, t(img), t(txt), t(mask), t(text), t(cand), reps=reps)
    return v, threads


def cpu_cir_sample(nq_s=256, n_s=200_000, reps=2):
    """Reference idiom topk(cdist(Q, G)) chunked, on a bounded slice; cost is linear in nq*N."""
    from oracle import torch_port
    torch.set_num_threads(os.cpu_count() or 1)
    gal = torch.from_numpy(synth.make_items(n_s, DPM, seed=5))
    q = torch.from_numpy(synth.make_queries(nq_s, 2 * DPM, seed=6))
    best = float("inf")
    for r in range(reps + 1):
        t0 = time.perf_counter()
        torch_port.search_cdist_topk(q, gal, k=TOPK)
        dt = time.perf_counter() - t0
        if r > 0 or reps == 0:
            best = min(best, dt)
    return nq_s * n_s / best  # (query, item) pairs per second


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, all host threads."""
    if rank != 0:
        return
    sd = synth.make_state_dict(D_MODEL, D_EMBED, seed=0)
    sample = args.cpu_sample
    t0 = time.perf_counter()
    vals = []
    for _ in range(args.warmup + args.steps):
        v, threads = cpu_cp_synthetic(sd, sample, seed=1, reps=1)
        vals.append(v)
        if time.perf_counter() - t0 > 150:
            break
    vals = vals[min(args.warmup, len(vals) - 1):]
    value = float(np.mean(vals))
    pairs = cpu_cir_sample()
    cir_q = pairs / args.cir_rows
    line = {
        "impl": "reference", "metric": "CP outfits/sec", "value": value, "unit": "outfits/s",
        "n_gpus": world, "steps": len(vals), "warmup": args.warmup, "ms_per_step": 1e3 * sample / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "configs[1]: CP + FITB(4 cand) scoring, mean fusion, d_model 512",
                   "sample": f"{sample} outfits per step (bounded sample of the 8192-outfit batch)"},
        "cpu_baseline": {"value": value, "unit": "outfits/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} outfits, CP + FITB, fp32 stock-torch port of the reference"},
        "e2e": {"value": value, "unit": "outfits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cir": {"metric": f"CIR queries/sec top-{TOPK} over {args.cir_rows} items", "value": cir_q,
                "unit": "queries/s", "kind": "port",
                "sample": "topk(cdist) on 256 q x 200k items, scaled linearly in nq*N"},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------ search legs
def exhaustive_check(queries, gal, result_idx, result_score, k, n_check, dist_ok, dev):
    """OUTSIDE the timed region: the exhaustive fp64 CUDA-core scan (ofx_exact_search -- no tensor cores, no
    candidate lists, no thresholds) of n_check queries spread over the batch, on every rank's shard, merged across
    ranks exactly like the real result.  -> True when indices AND fp64 scores equal the benchmarked result's."""
    import torch.distributed as dist
    from outfitx_b200 import _lib
    from outfitx_b200.search import merge_lists
    L = _lib.lib()
    nq = queries.shape[0]
    sel = torch.linspace(0, nq - 1, n_check, device=dev).round().to(torch.int32).unique()
    score = torch.empty(nq, k, dtype=torch.float64, device=dev)
    idx = torch.empty(nq, k, dtype=torch.int64, device=dev)
    ws = torch.empty(max(int(L.ofx_exact_search_workspace_bytes(gal.n_rows, sel.numel(), k)), 256), dtype=torch.uint8, device=dev)
    _lib.check(L.ofx_exact_search(gal.rows_f32.data_ptr(), gal.n_rows, gal.dim, gal.id_offset, queries.data_ptr(),
                                  sel.data_ptr(), sel.numel(), k, _lib.METRIC_L2, score.data_ptr(), idx.data_ptr(), None,
                                  ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream))
    s64 = sel.long()
    li, ls = idx[s64].contiguous(), score[s64].contiguous()
    if dist_ok:
        world = dist.get_world_size()
        payload = torch.stack([li, ls.view(torch.int64)]).contiguous()
        gathered = torch.empty((world * 2,) + tuple(li.shape), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(gathered, payload)
        gathered = gathered.view((world, 2) + tuple(li.shape))
        li, ls = merge_lists(gathered[:, 0].contiguous(), gathered[:, 1].contiguous().view(torch.float64), k)
    # indices must be identical; the fp64 scores come from two different summation orders (warp-strided re-rank vs
    # the scan's 16-byte lanes), so they may differ in the last bits
    ok = bool(torch.equal(li, result_idx[s64]) and torch.allclose(ls, result_score[s64], rtol=1e-12, atol=1e-10))
    return ok, int(sel.numel())


def bench_search(ctx, args, n_rows, queries, k_steps, label, peak_kind, embed=None):
    """Gallery-sharded exact top-k.  `embed`: optional callable producing the queries inside the timed step."""
    from outfitx_b200.search import Gallery, SearchStats, ShardedSearch
    L, dev, rank, world, dist_ok, pk = ctx["L"], ctx["dev"], ctx["rank"], ctx["world"], ctx["dist_ok"], ctx["pk"]
    rows, lo = make_gallery_shard(n_rows, rank, world, dev)
    gal = Gallery.build(rows, id_offset=lo, keep_fp32=True)
    searcher = ShardedSearch()
    state = {}

    def step():
        q = embed() if embed is not None else queries
        state["q"] = q
        state["res"] = searcher.search(q, gal, TOPK, "l2", True)

    step()
    torch.cuda.synchronize(dev)
    n1 = L.ofx_launch_count()
    SearchStats.reset()
    ms = timed(step, k_steps, 3, dist_ok, dev)
    launches = (L.ofx_launch_count() - n1) * k_steps // (k_steps + 3)
    unc = SearchStats.uncertified / max(SearchStats.queries, 1)
    nq = state["q"].shape[0]
    value = nq * k_steps / (ms * 1e-3)
    flops = 2.0 * nq * gal.n_rows * D_EMBED           # this rank's shard
    tf = flops * k_steps / (ms * 1e-3) / 1e12

    # the search alone (the dominant kernel's share when the step also embeds the queries)
    search_ms = ms
    if embed is not None:
        qfix = state["q"]
        search_ms = timed(lambda: searcher.search(qfix, gal, TOPK, "l2", True), k_steps, 1, dist_ok, dev)
        tf = flops * k_steps / (search_ms * 1e-3) / 1e12

    q_host = state["q"].cpu().pin_memory()
    idx_host = torch.empty(nq, TOPK, dtype=torch.int64).pin_memory()
    e2e = None
    if embed is None:
        def e2e_step():
            q = q_host.to(dev, non_blocking=True)
            idx, _ = searcher.search(q, gal, TOPK, "l2", True)
            idx_host.copy_(idx, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        e2e_ms = timed(e2e_step, k_steps, 1, dist_ok, dev)
        e2e = {"value": nq * k_steps / (e2e_ms * 1e-3), "unit": "queries/s",
               "h2d_bytes_per_step": q_host.numel() * 4, "d2h_bytes_per_step": idx_host.numel() * 8}

    ok, n_chk = exhaustive_check(state["q"], gal, state["res"][0], state["res"][1], TOPK, 64, dist_ok, dev)
    peak = pk[peak_kind]
    traffic, tsrc = ncu_traffic(f"search_sweep_{n_rows}") if world == 1 else (None, None)
    out = {
        "metric": f"CIR queries/sec top-{TOPK} over {n_rows} items", "value": value, "unit": "queries/s",
        "steps": k_steps, "ms_per_step": ms / k_steps,
        "config": {"workload": label, "rows_per_gpu": gal.n_rows, "l2": "gallery shard (bf16) larger than L2"},
        "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                     "traffic": traffic, "traffic_source": tsrc,
                     "algorithmic_bytes_per_launch": gal.n_rows * (1024 + 64) * 2,
                     "kernel": "tc_kernel<256,6,2,SchedSearch,EpiTopK<32>,pair> (+ EpiBlockMax seeding launch, merge_rerank), per GPU",
                     "flops_per_launch": flops, "ms_search": search_ms / k_steps,
                     "peak_kind": f"{peak_kind} bf16, {pk['source']}"},
        "gpu_launches": int(launches),
        "verified": ok,
        "verified_how": f"indices (exactly) and fp64 scores (to 1e-12) of {n_chk} queries equal an exhaustive fp64 CUDA-core scan of "
                        f"every rank's shard (ofx_exact_search), merged across {world} rank(s); outside the timed region",
        "uncertified_frac": unc,
    }
    if e2e:
        out["e2e"] = e2e
    del rows, gal
    torch.cuda.empty_cache()
    return out


def bench_large(ctx, args):
    """configs[4]: large-encoder CP sweep (d_model 1024 = clip + concat, 6 layers, 16 items per outfit)."""
    dev, pk = ctx["dev"], ctx["pk"]
    model, sd = make_model(dev, 1024)
    sweep, best = [], None
    for B in (256, 512, 1024, 2048, 4096, 8192, 16384, 32768):
        g = torch.Generator(device=dev).manual_seed(B)
        emb = torch.nn.functional.normalize(torch.randn(B, 16, 2, DPM, device=dev, generator=g), dim=-1).reshape(B, 16, 1024)
        mask = torch.zeros(B, 16, dtype=torch.bool, device=dev)          # n = 16 valid items
        reps = max(3, min(20, 65536 // B))
        ms = timed(lambda: model.score_cp(emb, mask), reps, 3, False, dev) / reps
        fl = float(flops_alg(np.full(B, 16), dm=1024, task="cp").sum())
        e = {"batch": B, "ms": ms, "outfits_per_s": B / ms * 1e3, "tflops_alg": fl / ms / 1e9,
             "frac_of_burst_peak": fl / ms / 1e9 / pk["burst"]}
        sweep.append(e)
        if best is None or e["outfits_per_s"] > best["outfits_per_s"]:
            best = e
        if B == 256:
            keep = (emb[:256].cpu(), mask[:256].cpu(), model.score_cp(emb[:256], mask[:256]).cpu())
        del emb, mask
    # CPU port on the B = 256 point (d_model 1024: ~130 outfits/s), which also verifies the GPU probabilities
    from oracle import torch_port
    torch.set_num_threads(os.cpu_count() or 1)
    port = torch_port.ReferencePort.from_numpy(sd)
    t0 = time.perf_counter()
    want = torch.sigmoid(port.cp(keep[0], keep[1]).float())[:, 0]
    dt = time.perf_counter() - t0
    dprob = float((keep[2] - want).abs().max())
    del model
    torch.cuda.empty_cache()
    return {
        "metric": "CP outfits/sec, large encoder (d_model 1024)", "value": best["outfits_per_s"], "unit": "outfits/s",
        "config": {"workload": "configs[4]: d_model 1024 (clip concat), 6 layers, 16 heads, d_ffn 2024, 16 items per "
                               "outfit, CP, bf16, batch sweep 256..32768 on 1 GPU", "best_batch": best["batch"],
                   "l2": "inputs of B >= 2048 (>= 134 MB) larger than L2"},
        "sweep": sweep,
        "roofline": {"bound": "tensor", "achieved": best["tflops_alg"], "peak": pk["burst"], "unit": "TFLOP/s",
                     "frac": best["frac_of_burst_peak"], "frac_of_sustained_peak": best["tflops_alg"] / pk["sustained"],
                     "traffic": None,
                     "kernel": "whole CP pass at the best batch (flops_alg: minimum exact work, SURVEY 8d); the pass is "
                               "LayerNorm + pair GEMMs (tc_kernel<256,..,pair>) + attention_mma_kernel<64>",
                     "peak_kind": f"burst bf16, {pk['source']}"},
        "cpu_baseline": {"value": 256 / dt, "unit": "outfits/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "256 outfits x 16 items, CP, fp32 stock-torch port (one pass, no warm-up)"},
        "verified": dprob <= 2e-2,
        "verified_how": f"max |prob - CPU port| = {dprob:.2e} over the 256-outfit point (bar 2e-2)",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="outfits per GPU per step (configs[1])")
    ap.add_argument("--cir-rows", type=int, default=10_000_000)
    ap.add_argument("--cir-queries", type=int, default=8192)
    ap.add_argument("--cir-steps", type=int, default=0, help="0 = min(steps, 5)")
    ap.add_argument("--skip", default="", help="comma list of cir, cir3, large, fp32, cpu")
    ap.add_argument("--no-cir", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=512)
    ap.add_argument("--e2e-chunk", type=int, default=2048, help="outfits per device chunk of the host pipeline")
    ap.add_argument("--sweep-out", default="", help="also append the configs[4] sweep points to this .jsonl file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the primary step's outputs of its last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    skip = set(x for x in args.skip.split(",") if x)
    if args.no_cir:
        skip |= {"cir", "cir3"}
    if args.no_cpu:
        skip.add("cpu")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from outfitx_b200 import _lib
    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist_ok = world > 1
    if dist_ok:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    pk = peaks()
    ctx = {"L": L, "dev": dev, "rank": rank, "world": world, "dist_ok": dist_ok, "pk": pk}

    # ------------------------------------------------------------------ CP + FITB (primary)
    model, sd = make_model(dev)
    B = args.batch
    img, txt, mask, text, cand, lengths = make_cp_inputs(B, dev, seed=1000 + rank)
    enc = {"image_embeddings": img, "text_embeddings": txt}
    state = {}

    def cp_step():
        state["probs"] = model.score_cp(outfit_mask=mask, encoder_input_dict=enc)
        state["fitb"] = model.score_fitb(outfit_mask=mask, target_item_text_embedding=text,
                                         candidate_item_embedding=cand, encoder_input_dict=enc)

    cp_step()
    torch.cuda.synchronize(dev)
    n0 = L.ofx_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    cp_ms = timed(cp_step, args.steps, args.warmup, dist_ok, dev, sampler)
    launches_cp = (L.ofx_launch_count() - n0) * args.steps // (args.steps + args.warmup)
    if args.dump_outputs and rank == 0:
        pred, dists, query = state["fitb"]
        dump_outputs(args.dump_outputs, {"cp_probs": state["probs"], "fitb_pred": pred, "fitb_dists": dists,
                                         "cir_query": query})
    cp_value = world * B * args.steps / (cp_ms * 1e-3)
    flops_step = float(flops_alg(lengths, task="cp").sum() + flops_alg(lengths, task="fitb").sum())
    cp_tflops = flops_step * args.steps / (cp_ms * 1e-3) / 1e12     # per GPU (every rank does B outfits)
    clocks = sampler.summary() if sampler else None

    # dominant kernel, timed alone with CUDA events on its launching stream: the fused FFN block
    # (ffn_block_kernel) on this batch's valid-token count
    dom = time_ffn_block(L, int(B + lengths.sum()), dev)

    # end to end through the public API with HOST buffers (pinned), copies inside the timed region.
    # Headline `e2e`: the packed host layout (valid item rows only + lengths: what a collate that skips the zero
    # padding hands over); `e2e_padded`: the reference collate's padded (B, 16, dpm) tensors.
    from outfitx_b200.pipeline import HostScoringPipeline, pack_valid_rows
    host = {k: v.cpu().pin_memory() for k, v in dict(img=img, txt=txt, mask=mask, text=text, cand=cand).items()}
    img_rows, txt_rows, lens_h = pack_valid_rows(host["img"], host["txt"], host["mask"])
    img_rows, txt_rows = img_rows.pin_memory(), txt_rows.pin_memory()
    res_host = {"probs": torch.empty(B, dtype=torch.float32).pin_memory(),
                "pred": torch.empty(B, dtype=torch.int64).pin_memory()}
    d2h = sum(v.numel() * v.element_size() for v in res_host.values())
    pipe = HostScoringPipeline(model, chunk=args.e2e_chunk)
    nbytes = lambda *ts: sum(t.numel() * t.element_size() for t in ts)
    h2d_packed = nbytes(img_rows, txt_rows, host["text"], host["cand"]) + B * 16 * 5      # + ids (int32) and mask bytes
    h2d_padded = nbytes(*host.values())

    def e2e_packed_step():
        pipe.score_packed(img_rows, txt_rows, lens_h, host["text"], host["cand"], out=res_host)

    def e2e_padded_step():
        pipe.score(host["img"], host["txt"], host["mask"], host["text"], host["cand"], out=res_host)

    e2e_ms = timed(e2e_packed_step, args.steps, 2, dist_ok, dev)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)
    packed_same = bool(torch.equal(res_host["probs"], state["probs"].cpu()) and torch.equal(res_host["pred"], state["fitb"][0].cpu()))
    e2e_pad_ms = timed(e2e_padded_step, args.steps, 2, dist_ok, dev)
    e2e_pad_value = world * B * args.steps / (e2e_pad_ms * 1e-3)

    # the same step with the collate on the device (SURVEY.md N2): item tables resident in HBM, only
    # item ids / masks / text prefixes / candidate ids cross PCIe.  Reported beside `e2e`, not as it.
    n_table = 200_000
    g2 = torch.Generator(device=dev).manual_seed(77 + rank)
    tab_img = torch.randn(n_table, DPM, device=dev, generator=g2)
    tab_txt = torch.randn(n_table, DPM, device=dev, generator=g2)
    tab_cand = torch.nn.functional.normalize(torch.randn(n_table, 2, DPM, device=dev, generator=g2), dim=-1)
    tab_cand = tab_cand.reshape(n_table, 2 * DPM).contiguous()
    ids_host = torch.randint(0, n_table, (B, 16), dtype=torch.int32).pin_memory()
    cids_host = torch.randint(0, n_table, (B, N_CAND), dtype=torch.int32).pin_memory()
    ids_h2d = ids_host.numel() * 4 + cids_host.numel() * 4 + host["mask"].numel() + host["text"].numel() * 4
    pipe_ids = HostScoringPipeline(model, chunk=B)   # ids are 64 B per outfit: nothing to overlap, one chunk
    res_ids = {k: torch.empty_like(v).pin_memory() for k, v in res_host.items()}

    def cp_e2e_ids_step():
        pipe_ids.score_ids(ids_host, host["mask"], tab_img, tab_txt, host["text"], cids_host, tab_cand, out=res_ids)

    e2e_ids_ms = timed(cp_e2e_ids_step, args.steps, 2, dist_ok, dev)
    e2e_ids_value = world * B * args.steps / (e2e_ids_ms * 1e-3)
    del tab_img, tab_txt, tab_cand

    # CPU baseline = the reference's stock-torch stack on the FIRST cpu_sample outfits of this very batch; the same
    # run verifies the GPU results (outside every timed region)
    cpu, verified, vhow = None, None, None
    if rank == 0 and "cpu" not in skip:
        # N > 1: rank 0 still checks its own results (one untimed pass of the port); the baseline is an N = 1 figure
        n = min(args.cpu_sample, B)
        v, threads, want_p, want_pred, want_d = cpu_cp_run(sd, host["img"][:n], host["txt"][:n], host["mask"][:n],
                                                           host["text"][:n], host["cand"][:n], reps=2 if world == 1 else 0)
        if world == 1:
            cpu = {"value": v, "unit": "outfits/s", "cores": threads, "kind": "port",
                   "sample": f"the first {n} outfits of the 8192-outfit batch, CP + FITB, fp32, "
                             "stock-torch port of the reference (oracle/torch_port.py)"}
        dprob = float((state["probs"][:n].cpu() - want_p).abs().max())
        agree = (state["fitb"][0][:n].cpu() == want_pred)
        dd = torch.sort(want_d, -1).values
        gaps = (dd[:, 1] - dd[:, 0])[~agree]
        near = bool((gaps < 2e-2).all()) if gaps.numel() else True
        verified = bool(dprob <= 2e-2 and near and packed_same)
        vhow = (f"first {n} outfits vs the CPU port: max |prob - ref| = {dprob:.2e} (bar 2e-2); FITB argmin equal on "
                f"{float(agree.float().mean()):.4f} of them, every difference a near-tie (gap of the two best reference "
                f"distances < 2e-2: {near}); packed-layout e2e results bit-identical to the device-resident ones: {packed_same}")
    # the same step in precision="fp32": every nn.Linear on the tensor cores as a bf16 hi / lo split GEMM (N = 1 only)
    fp32 = None
    if world == 1 and "fp32" not in skip:
        m32, _ = make_model(dev, precision="fp32")
        st32 = {}

        def fp32_step():
            st32["probs"] = m32.score_cp(outfit_mask=mask, encoder_input_dict=enc)
            st32["fitb"] = m32.score_fitb(outfit_mask=mask, target_item_text_embedding=text,
                                          candidate_item_embedding=cand, encoder_input_dict=enc)

        k32 = max(2, min(args.steps, 3))
        ms32 = timed(fp32_step, k32, 3, False, dev) / k32
        fp32 = {"metric": "CP outfits/sec, precision=fp32", "value": B / (ms32 * 1e-3), "unit": "outfits/s", "ms_per_step": ms32,
                "dtype": "f32 operands as bf16 hi + lo pieces on tcgen05 (3 products, fp32 accumulation); attention, LayerNorm, "
                         "heads in fp32 on the CUDA cores",
                "config": {"workload": "configs[1] (CP + FITB, 8192 outfits) with precision='fp32'"}}
        if cpu is not None:
            dp = float((st32["probs"][:n].cpu() - want_p).abs().max())
            same = bool((st32["fitb"][0][:n].cpu() == want_pred).all())
            fp32["verified"] = bool(dp <= 1e-4 and same)
            fp32["verified_how"] = (f"first {n} outfits vs the CPU port (fp32): max |prob - ref| = {dp:.2e} (bar 1e-4), "
                                    f"FITB argmin identical: {same}")
        del m32, st32
    del host, img_rows, txt_rows
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ CIR (secondary, sharded)
    cir = cir3 = large = None
    if "cir" not in skip:
        k_steps = args.cir_steps or min(args.steps, 5)
        g = torch.Generator(device=dev).manual_seed(6)
        queries = torch.randn(args.cir_queries, D_EMBED, device=dev, generator=g) * 0.05
        cir = bench_search(ctx, args, args.cir_rows, queries, k_steps,
                           f"configs[3]: {args.cir_queries} queries, exact top-{TOPK} (L2) over a {args.cir_rows}-item "
                           f"1024-d gallery row-sharded over {world} GPU(s), one NCCL all-gather + merge", "sustained")
        cir["scaling"] = "strong"
        if rank == 0 and "cpu" not in skip and world == 1:
            pairs = cpu_cir_sample()
            cir["cpu_baseline"] = {"value": pairs / args.cir_rows, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                                   "sample": "topk(cdist(Q,G)) on 256 q x 200k items, scaled linearly in nq*N"}
    if "cir3" not in skip and world == 1:
        # configs[2]: the queries are produced by the d_model-1024 encoder INSIDE the timed step
        m1024, sd1024 = make_model(dev, 1024)
        nq3 = 4096
        emb3, mask3, len3 = synth.make_outfits(nq3, "concat", seed=301)
        emb3, mask3 = torch.from_numpy(emb3).to(dev), torch.from_numpy(mask3).to(dev)
        text3 = torch.from_numpy(synth.make_text_prefix(nq3, 512, seed=303)).to(dev)
        k3 = max(3, min(args.steps, 10))
        cir3 = bench_search(ctx, args, 1_000_000, None, k3,
                            "configs[2]: 4096 outfit queries produced by the d_model-1024 CIR forward inside the timed step "
                            "(n ~ U{2..16} items), exact top-10 (L2) over a 1000000-item gallery, 1 GPU", "burst",
                            embed=lambda: m1024.cir_embed(emb3, mask3, text3))
        # BASELINE.md quotes config 3 for the search alone (target 475 k q/s): report it beside the whole step
        cir3["search_only"] = {"value": 4096 / (cir3["roofline"]["ms_search"] * 1e-3), "unit": "queries/s",
                               "ms": cir3["roofline"]["ms_search"],
                               "note": "same queries already embedded; `value` above includes the CIR forward"}
        enc_fl = float(flops_alg(len3, dm=1024, task="cir").sum())
        tot = (enc_fl + cir3["roofline"]["flops_per_launch"]) / (cir3["ms_per_step"] * 1e-3) / 1e12
        cir3["roofline_step"] = {"bound": "tensor", "achieved": tot, "peak": pk["burst"], "unit": "TFLOP/s",
                                 "frac": tot / pk["burst"], "frac_of_sustained_peak": tot / pk["sustained"],
                                 "flops_encoder": enc_fl,
                                 "kernel": "whole step: d_model-1024 CIR forward of 4096 outfits + search sweep + re-rank"}
        if "cpu" not in skip:
            from oracle import torch_port
            torch.set_num_threads(os.cpu_count() or 1)
            port = torch_port.ReferencePort.from_numpy(sd1024)
            n = 128
            t0 = time.perf_counter()
            want_q = port.cir(emb3[:n].cpu(), mask3[:n].cpu(), text3[:n].cpu())
            t_embed = (time.perf_counter() - t0) / n
            pairs = cpu_cir_sample(128, 200_000, reps=1)
            t_search = 1_000_000 / pairs
            got_q = m1024.cir_embed(emb3[:n], mask3[:n], text3[:n]).cpu()
            rel = float((got_q - want_q).abs().max() / want_q.abs().max())
            cir3["cpu_baseline"] = {"value": 1.0 / (t_embed + t_search), "unit": "queries/s", "cores": torch.get_num_threads(),
                                    "kind": "port", "sample": "CIR forward of 128 outfits + topk(cdist) of 128 q x 200k items, "
                                                              "scaled linearly to 1 M items"}
            cir3["verified"] = bool(cir3["verified"] and rel <= 5e-2)
            cir3["verified_how"] += f"; bf16 query embeddings vs the CPU port on 128 outfits: max rel err {rel:.2e} (bar 5e-2)"
        del m1024
        torch.cuda.empty_cache()
    if "large" not in skip and world == 1:
        large = bench_large(ctx, args)
        if args.sweep_out:
            with open(args.sweep_out, "a") as f:
                for e in large["sweep"]:
                    f.write(json.dumps(dict(e, workload="configs[4] large encoder CP")) + "\n")

    if rank == 0:
        ffn_traffic, ffn_src = ncu_traffic("ffn_block_82158")
        line = {
            "metric": "CP outfits/sec", "value": cp_value, "unit": "outfits/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cp_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "configs[1]: CP + FITB(4 candidates) scoring, 8192 outfits per GPU, bf16, "
                                   "mean-aggregation fusion (d_model 512, 6 layers, 16 heads, d_ffn 2024), "
                                   "n ~ U{2..16} items per outfit", "batch_per_gpu": B,
                       "l2": "inputs (805 MB per step) larger than L2", "parallelism": f"dp{world} by outfit, no collective"},
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": dom["tflops"], "peak": pk["burst"], "unit": "TFLOP/s",
                         "frac": dom["tflops"] / pk["burst"], "traffic": ffn_traffic, "traffic_source": ffn_src,
                         "kernel": "ffn_block_kernel (fused LN2 + linear1 + mish + linear2 + residual + norm1 of the "
                                   "next layer; dominant kernel of the step), timed alone with CUDA events",
                         "rows_per_launch": dom["rows"], "us_per_launch": dom["us_per_launch"],
                         "flops_per_launch": dom["flops_per_launch"],
                         "algorithmic_bytes_per_launch": dom["rows"] * 5120,
                         "peak_kind": f"burst bf16, {pk['source']}"},
            "roofline_step": {"bound": "tensor", "achieved": cp_tflops, "peak": pk["burst"], "unit": "TFLOP/s",
                              "frac": cp_tflops / pk["burst"], "frac_of_sustained_peak": cp_tflops / pk["sustained"],
                              "flops_per_step": flops_step,
                              "kernel": "whole step, all launches (flops_alg: minimum exact work, SURVEY 8d)"},
            "e2e": {"value": e2e_value, "unit": "outfits/s", "h2d_bytes_per_step": h2d_packed, "d2h_bytes_per_step": d2h,
                    "api": "outfitx_b200.pipeline.HostScoringPipeline.score_packed: fp32 image + text embeddings of the "
                           "VALID items (sum n_i, 512) + lengths from pinned host memory, chunked H2D overlapped with scoring"},
            "e2e_padded": {"value": e2e_pad_value, "unit": "outfits/s", "h2d_bytes_per_step": h2d_padded, "d2h_bytes_per_step": d2h,
                           "api": "HostScoringPipeline.score: the reference collate's zero-padded (B,16,512) tensors"},
            "e2e_device_collate": {"value": e2e_ids_value, "unit": "outfits/s", "h2d_bytes_per_step": ids_h2d,
                                   "d2h_bytes_per_step": d2h,
                                   "api": "HostScoringPipeline.score_ids: item ids from host, 200k-item embedding "
                                          "tables resident in HBM (SURVEY.md N2)"},
            "gpu_launches": int(launches_cp),
            "cpu_baseline": cpu,
            "verified": verified, "verified_how": vhow,
            "cir": cir, "cir3": cir3, "large": large, "fp32": fp32,
        }
        print(json.dumps(line), file=_RESULT_OUT, flush=True)
    if dist_ok:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
