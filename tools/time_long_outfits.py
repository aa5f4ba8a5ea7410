"""Cost of outfits of up to 64 items on one GPU, its cases alternated in one process.

    python tools/time_long_outfits.py [--rounds 7] [--out profiles/r3_time_long_outfits.json]

Cases, each a CP + FITB(4) step over 8192 outfits, d_model 512, bf16, mean fusion on the fly (bench.py's step):
  a16   n ~ U{2..16}, padded to 16 slots (the bench workload)
  a64   the same outfits padded to 64 slots: the cost of the wider attention launch alone
  c64   n ~ U{2..64}, 64 slots
and large: CP over the c64 outfits with the large encoder (d_model 1024, concat fusion on the fly).
Each is timed with CUDA events `rounds` times in the order a16, a64, c64, large, a16, ...  Reports ms, outfits/s and
valid tokens/s (prefix token + valid items) per case.  A separate torch.profiler run of one a16 and one c64 step
gives the attention kernels' time per layer.  The card's name, power limit and maximum SM clock are read with
nvidia-smi in the same run and written with the results as JSON."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from outfitx_b200 import synth  # noqa: E402

B = 8192
W = 64
CASES = ("a16", "a64", "c64", "large")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def pad_slots(t, width, value):
    pad = torch.full((t.shape[0], width - t.shape[1]) + tuple(t.shape[2:]), value, dtype=t.dtype, device=t.device)
    return torch.cat([t, pad], 1).contiguous()


def make_steps(dev):
    model, _ = bench.make_model(dev)
    large, _ = bench.make_model(dev, 1024)
    img, txt, mask, text, cand, lengths = bench.make_cp_inputs(B, dev, 1000)
    g = torch.Generator(device=dev).manual_seed(2000)
    img_c = torch.randn(B, W, bench.DPM, device=dev, generator=g)
    txt_c = torch.randn(B, W, bench.DPM, device=dev, generator=g)
    len_c = synth.make_lengths(B, 2001, hi=W)
    mask_c = torch.from_numpy(synth.make_mask(len_c, W)).to(dev)
    inputs = {"a16": (img, txt, mask, lengths),
              "a64": (pad_slots(img, W, 0.0), pad_slots(txt, W, 0.0), pad_slots(mask, W, True), lengths),
              "c64": (img_c, txt_c, mask_c, len_c)}
    steps, tokens = {}, {}
    for name, (i, t, m, n) in inputs.items():
        enc = {"image_embeddings": i, "text_embeddings": t}

        def step(enc=enc, m=m):
            model.score_cp(outfit_mask=m, encoder_input_dict=enc)
            model.score_fitb(outfit_mask=m, target_item_text_embedding=text, candidate_item_embedding=cand,
                             encoder_input_dict=enc)
        steps[name], tokens[name] = step, int(B + n.sum())
    enc_c = {"image_embeddings": img_c, "text_embeddings": txt_c, "aggregation_method": "concat"}
    steps["large"] = lambda: large.score_cp(outfit_mask=mask_c, encoder_input_dict=enc_c)
    tokens["large"] = tokens["c64"]
    return steps, tokens


def measure(steps, tokens, rounds, reps=10, warmup=3):
    for name in CASES:
        for _ in range(warmup):
            steps[name]()
    torch.cuda.synchronize()
    ms = {c: [] for c in CASES}
    for _ in range(rounds):
        for c in CASES:
            ms[c].append(event_ms(steps[c], reps))
    out = {}
    for c, v in ms.items():
        s = sorted(v)
        med = s[len(s) // 2]
        out[c] = {"median_ms": med, "min_ms": s[0], "max_ms": s[-1], "ms": v, "valid_tokens": tokens[c],
                  "outfits_per_s": B / med * 1e3, "valid_tokens_per_s": tokens[c] / med * 1e3}
    return out


def attention_profile(steps, names=("a16", "c64")):
    """Attention kernel time per layer: one step = CP + FITB forwards of 6 layers each = 12 attention launches."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name in names:
        steps[name]()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            steps[name]()
            torch.cuda.synchronize()
        attn, total, kernels = 0.0, 0.0, {}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            us = e.device_time if hasattr(e, "device_time") else e.cuda_time
            total += us
            if "attention" in e.name:
                attn += us
                k = kernels.setdefault(e.name.split("(")[0], [0, 0.0])
                k[0] += 1
                k[1] += us
        n_launch = sum(k[0] for k in kernels.values())
        out[name] = {"attention_us_per_layer": attn / max(n_launch, 1), "attention_launches": n_launch,
                     "attention_share_of_kernel_time": attn / max(total, 1e-9), "kernel_time_us": total,
                     "kernels": {k: {"launches": v[0], "mean_us": v[1] / v[0]} for k, v in kernels.items()}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_time_long_outfits.json"))
    args = ap.parse_args()
    if args.rounds < 7:
        raise SystemExit("--rounds must be >= 7")
    assert torch.cuda.is_available(), "tools/time_long_outfits.py needs a B200 (no CPU fallback)"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "rounds": args.rounds, "batch": B,
           "order": "a16, a64, c64, large alternating; CUDA events per round, 10 steps each",
           "cases": {"a16": "CP + FITB(4), d_model 512 bf16, n ~ U{2..16}, 16 slots",
                     "a64": "the a16 outfits padded to 64 slots",
                     "c64": "CP + FITB(4), d_model 512 bf16, n ~ U{2..64}, 64 slots",
                     "large": "CP only, d_model 1024 bf16 (concat), the c64 outfits"}}
    with torch.no_grad():
        steps, tokens = make_steps(dev)
        res["timing"] = measure(steps, tokens, args.rounds)
        res["profile"] = attention_profile(steps)
    for c in CASES:
        r = res["timing"][c]
        print(f"{c:6s} {r['median_ms']:8.3f} ms [{r['min_ms']:.3f}-{r['max_ms']:.3f}]  "
              f"{r['outfits_per_s'] / 1e3:8.1f} k outfits/s  {r['valid_tokens_per_s'] / 1e6:7.2f} M tokens/s")
    for c, p in res["profile"].items():
        print(f"{c}: attention {p['attention_us_per_layer']:.1f} us per layer ({p['attention_launches']} launches), "
              f"{100 * p['attention_share_of_kernel_time']:.1f} % of kernel time; {p['kernels']}")
    print(res["gpu"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
