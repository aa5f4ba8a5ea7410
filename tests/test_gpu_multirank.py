"""GPU, world_size 2 over NCCL: the gallery-sharded search as it really runs (one process per GPU,
torch.distributed all_gather_into_tensor between ofx_topk_search and ofx_topk_merge) must equal the single-GPU
search of the whole gallery bit for bit -- indices AND fp64 scores.  (The reference has no multi-GPU inference to
compare with: complementary_item_retrieval_trainer.py:350-351 refuses world_size > 1 in test mode.)

Skipped with fewer than 2 GPUs; CPU coverage of the same host logic is tests/test_sharded_host.py (gloo).
"""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["OFX_ROOT"])
from outfitx_b200 import synth
from outfitx_b200.search import Gallery, ShardedSearch, cir_search, local_search, shard_rows
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
ok = True
for n, nq, k, metric in ((60_001, 300, 10, "l2"), (9_000, 64, 50, "dot"), (7, 5, 10, "l2")):
    gal = synth.make_items(n, 512, seed=n, dup=min(500, n // 4))
    q = torch.from_numpy(synth.make_queries(nq, 1024, seed=n + 1)).to(dev)
    lo, hi = shard_rows(n, rank, world)
    shard = Gallery.build(torch.from_numpy(gal[lo:hi]).to(dev), id_offset=lo)
    idx, score = cir_search(q, shard, k=k, metric=metric)                  # sharded: the group is initialised
    full_i, full_s = local_search(q, Gallery.build(torch.from_numpy(gal).to(dev)), k, metric)   # whole gallery, this GPU
    same = torch.equal(idx, full_i) and torch.equal(score, full_s)
    flag = torch.tensor([1 if same else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = ok and bool(flag.item())
    if rank == 0:
        print(f"case n={n} nq={nq} k={k} {metric}: sharded == single: {bool(flag.item())}", flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_nccl_sharded_search_equals_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, OFX_ROOT=ROOT, NCCL_DEBUG="WARN")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(script)],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("sharded == single: True") == 3
