"""precision="fp16" against "bf16" on one GPU, alternating the two in one process.

    python tools/time_fp16.py [--rounds 7] [--out profiles/r3_time_fp16.json]

Three workloads, each timed with CUDA events, `rounds` times per precision in the order bf16, fp16, bf16, ...:
  cp_fitb  configs[1]: one CP + FITB(4) step over 8192 outfits, d_model 512, mean fusion on the fly (bench.py's step)
  large    the large encoder: CP over 4096 outfits of 16 items, d_model 1024
  ffn      the fused FFN block alone, in the form layers 0-4 launch (it also emits the next layer's norm1):
           82k token rows, d_model 512, d_ffn 2048, inputs rotated over 4 buffers (larger than L2)
Reports the median and range of each (ms per step / per launch) with the card's name, power limit and maximum SM
clock, read with nvidia-smi in the same run, and writes them as JSON."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from outfitx_b200 import _lib  # noqa: E402

PRECISIONS = ("bf16", "fp16")


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


def cp_fitb_steps(dev):
    img, txt, mask, text, cand, _ = bench.make_cp_inputs(8192, dev, 1000)
    enc = {"image_embeddings": img, "text_embeddings": txt}
    steps = {}
    for prec in PRECISIONS:
        model, _ = bench.make_model(dev, precision=prec)

        def step(model=model):
            model.score_cp(outfit_mask=mask, encoder_input_dict=enc)
            model.score_fitb(outfit_mask=mask, target_item_text_embedding=text, candidate_item_embedding=cand,
                             encoder_input_dict=enc)
        steps[prec] = step
    return steps


def large_steps(dev):
    B = 4096
    g = torch.Generator(device=dev).manual_seed(B)
    emb = torch.nn.functional.normalize(torch.randn(B, 16, 2, bench.DPM, device=dev, generator=g),
                                        dim=-1).reshape(B, 16, 1024)
    mask = torch.zeros(B, 16, dtype=torch.bool, device=dev)
    steps = {}
    for prec in PRECISIONS:
        model, _ = bench.make_model(dev, 1024, precision=prec)
        steps[prec] = lambda model=model: model.score_cp(emb, mask)
    return steps


def ffn_steps(dev, rows=82000):
    L = _lib.lib()
    dm, fp, f = bench.D_MODEL, 2048, bench.F_FFN
    g = torch.Generator(device=dev).manual_seed(11)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    ln_w, ln_b = 1.0 + 0.1 * r(dm), 0.1 * r(dm)
    w1 = r(fp, dm) / dm ** 0.5
    w1[f:] = 0
    w2 = r(dm, fp) / fp ** 0.5
    w2[:, f:] = 0
    b1, b2 = 0.1 * r(fp), 0.1 * r(dm)
    b1[f:] = 0
    bufs = [r(rows, dm) for _ in range(4)]
    ws = torch.empty(int(L.ofx_ffn_block_workspace_bytes(rows, dm, fp)), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    steps = {}
    for prec, dt, fn in (("bf16", torch.bfloat16, L.ofx_ffn_block_ln_bf16), ("fp16", torch.float16, L.ofx_ffn_block_f16)):
        w1t, w2t = w1.to(dt).contiguous(), w2.to(dt).contiguous()
        h = torch.empty(rows, dm, device=dev, dtype=dt)
        it = iter(range(1 << 62))

        def step(fn=fn, w1t=w1t, w2t=w2t, h=h, it=it):
            x = bufs[next(it) % 4]
            _lib.check(fn(x.data_ptr(), rows, dm, fp, ln_w.data_ptr(), ln_b.data_ptr(), w1t.data_ptr(), b1.data_ptr(),
                          w2t.data_ptr(), b2.data_ptr(), h.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                          ws.data_ptr(), ws.numel(), st))
        steps[prec] = step
    return steps


def measure(steps, rounds, reps, warmup=3):
    for prec in PRECISIONS:
        for _ in range(warmup):
            steps[prec]()
    torch.cuda.synchronize()
    ms = {p: [] for p in PRECISIONS}
    for _ in range(rounds):
        for prec in PRECISIONS:
            ms[prec].append(event_ms(steps[prec], reps))
    out = {}
    for prec, v in ms.items():
        s = sorted(v)
        out[prec] = {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1], "ms": v}
    out["fp16_over_bf16_median"] = out["fp16"]["median_ms"] / out["bf16"]["median_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_time_fp16.json"))
    args = ap.parse_args()
    if args.rounds < 5:
        raise SystemExit("--rounds must be >= 5")
    assert torch.cuda.is_available(), "tools/time_fp16.py needs a B200 (no CPU fallback)"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "rounds": args.rounds, "order": "bf16, fp16 alternating; CUDA events per round"}
    with torch.no_grad():
        res["cp_fitb"] = dict(measure(cp_fitb_steps(dev), args.rounds, reps=10),
                              workload="configs[1]: CP + FITB(4) step, 8192 outfits, d_model 512, ms per step")
        res["large"] = dict(measure(large_steps(dev), args.rounds, reps=5),
                            workload="CP over 4096 outfits x 16 items, d_model 1024, ms per pass")
        res["ffn"] = dict(measure(ffn_steps(dev), args.rounds, reps=20),
                          workload="fused FFN block emitting the next norm1, 82000 rows, d_ffn 2048, ms per launch")
    for k in ("cp_fitb", "large", "ffn"):
        r = res[k]
        print(f"{k:8s} bf16 {r['bf16']['median_ms']:.3f} ms [{r['bf16']['min_ms']:.3f}-{r['bf16']['max_ms']:.3f}]  "
              f"fp16 {r['fp16']['median_ms']:.3f} ms [{r['fp16']['min_ms']:.3f}-{r['fp16']['max_ms']:.3f}]  "
              f"fp16/bf16 {r['fp16_over_bf16_median']:.4f}")
    print(res["gpu"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
