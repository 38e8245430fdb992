"""BASELINE cfg-4: 3-D Mehler kernel, greedy mutual-information design of 512 points from |V| = 200 000 candidates,
the |V| x |V| factor and its inverse-transpose sharded by column blocks over the ranks.

    python -m torch.distributed.run --nproc-per-node 8 ... scripts/cfg4_mi.py [--V 200000] [--N 512] [--compare-dense] [--nu]

--nu replaces the scalar noise 1e-2 by the per-point noise nu(x) = 1e-2 (1 + |x|^2 / 3) at every pool point.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--V", type=int, default=200_000)
ap.add_argument("--N", type=int, default=512)
ap.add_argument("--compare-dense", action="store_true", help="rank 0 also runs the single-GPU dense engine (small V only)")
ap.add_argument("--nu", action="store_true", help="per-point noise nu(x) = 1e-2 (1 + |x|^2 / 3) instead of the scalar 1e-2")
args = ap.parse_args()

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

from gpexp_b200 import kernels  # noqa: E402
from gpexp_b200.device import Device  # noqa: E402
from gpexp_b200.engine import GreedyMIEngine, Shard, ShardedMIEngine  # noqa: E402

V, N, noise = args.V, args.N, 1e-2
pool = np.random.default_rng(4).standard_normal((V, 3))
nu = 1e-2 * (1.0 + np.sum(pool * pool, axis=1) / 3.0) if args.nu else None
dev = Device.get(local)
kern = kernels.KernelMehlerND([0.9, 0.9, 0.9], 3)
kern._bind(dev)
shard = Shard() if world > 1 else None


def sync():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()


sync()
t0 = time.perf_counter()
eng = ShardedMIEngine(dev, pool, N, 0.0 if args.nu else noise, shard=shard, pool_noise=nu)
sync()
setup_s = time.perf_counter() - t0
t0 = time.perf_counter()
idx = eng.run(N, start=0)
sync()
design_s = time.perf_counter() - t0
info = int(eng.info.item())
scores = eng.pick_scores[:N].cpu().numpy()
if rank == 0:
    out = {"workload": "cfg-4: 3-D Mehler t=0.9, greedy MI design of %d points from |V|=%d, noise %s"
                       % (N, V, "1e-2 (1 + |x|^2 / 3)" if args.nu else "1e-2"),
           "n_gpus": world, "setup_s": setup_s, "setup_useful_tflops_total": (2.0 * V ** 3 / 3.0) / setup_s / 1e12,
           "setup_tflops_per_gpu": (2.0 * V ** 3 / 3.0 / world) / setup_s / 1e12,
           "design_s": design_s, "ms_per_step": 1e3 * design_s / (N - 1), "candidates_per_s_per_step": (N - 1) * V / design_s,
           "potrf_info": info, "distinct_picks": len(set(int(i) for i in idx)) == N, "first_picks": [int(i) for i in idx[:10]],
           "min_pick_score": float(scores[1:].min()), "max_pick_score": float(scores[1:].max()),
           "hbm_per_gpu_gb": 2 * 8.0 * V * max(eng.ncols_per_rank) / 1e9, "blk": eng.BLK,
           "distribution": "block-cyclic column blocks, structural zeros of Y skipped in-kernel"}
    if args.compare_dense:
        dense = GreedyMIEngine(dev, dev.points(pool), N, 0.0 if args.nu else noise, pool_noise=nu)
        didx = dense.run(N, start=0)
        out["indices_equal_dense_single_gpu_engine"] = [int(i) for i in didx] == [int(i) for i in idx]
    print(json.dumps(out), flush=True)
    os.makedirs("gpurun_out", exist_ok=True)
    json.dump(out, open("gpurun_out/cfg4_V%d_N%d.json" % (V, world), "w"), indent=1)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
