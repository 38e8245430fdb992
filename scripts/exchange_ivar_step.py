"""Cost of the exchange refinement of greedy IVAR designs at cfg-2 size (100 000 candidates x 100 000 integration points,
2-D SE cl = (0.06, 0.09), noise 1e-6, INT8 core, contraction mode as in bench.py).

    python scripts/exchange_ivar_step.py [--reps 50] [--rounds 3] [--steps 5] [--max-sweeps 10] [--out result.json]

1. gpx_design_delete_rows on a 255-row factor of 100 000 columns (j = 0: 16 * 255 * 1e5 = 408 MB read + written, more
   than the 126 MB L2), CUDA events over --reps launches, against the bandwidth of a 1 GB device-to-device copy measured
   in the same run.
2. gpx_design_delete_factor at n = 255 and n = 4096 (j = 0, the exchange's position), each call on a fresh copy of the
   Cholesky factor of a seeded design, CUDA events around the kernel alone.
3. One exchange step (remove position 0 of a 256-point design, score at n = 255, keep-or-swap, append) against one
   greedy step (score at n = 255, append), alternated: --rounds rounds of --steps steps each.
4. refineGreedyIVARExperimentalDesign of bench.py's 256-point greedy design (same seed and inputs): sweeps, swaps, cost
   before and after, wall time.
Prints the device name and power limit (a query only) and one JSON line, which --out also writes to a file."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=50)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--max-sweeps", type=int, default=10)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import bench  # noqa: E402  (the workload's inputs: same seed, same candidates and integration points)
import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import gp as gpmod, kernels  # noqa: E402
from gpexp_b200._lib import check, lib  # noqa: E402
from gpexp_b200.approximation import Space  # noqa: E402
from gpexp_b200.device import Device, ptr  # noqa: E402
from gpexp_b200.engine import DesignFactor  # noqa: E402

ed.VERBOSE = False
CFG = bench.CFG
N = CFG["N"]          # 256
RTOL = 1e-8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


dev = Device.get(0)
cand, mc = bench.make_inputs()
kern = kernels.KernelSquaredExponential(CFG["cl"], CFG["signal"], CFG["d"])
cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, CFG["noise"]), 1, Space(CFG["d"], None, None), mcPoints=mc)
out = {"device": gpu_info(),
       "workload": "cfg-2: 2-D SE cl = (0.06, 0.09), signal 1, noise 1e-6, C = M = 100 000, INT8 core, contraction mode"}

# ---- 1. delete_rows bandwidth ------------------------------------------------------------------------------------------
n, ncols = N - 1, CFG["C"]
ld = (ncols + 127) // 128 * 128
kern._bind(dev)
f255 = DesignFactor(dev, dev.points(cand[np.random.default_rng(0).permutation(ncols)[:n]]), CFG["noise"])
rot = dev.zeros(2 * n)
U = f255.U.clone()
check(lib.gpx_design_delete_factor(dev.h, ptr(U), n, U.shape[1], 0, ptr(rot), None, None, None, dev.stream), "delete_factor")
W = torch.randn(n, ld, dtype=torch.float64, device=dev.torch_device) / np.sqrt(n)
var = dev.zeros(ld)


def rows():
    check(lib.gpx_design_delete_rows(dev.h, ptr(rot), 0, n, ptr(W), ld, ncols, ptr(var), dev.stream), "delete_rows")


for _ in range(3):
    rows()
e0, e1 = events()
e0.record()
for _ in range(args.reps):
    rows()
e1.record()
torch.cuda.synchronize()
rows_ms = e0.elapsed_time(e1) / args.reps
rows_bytes = 16 * n * ncols
src = torch.empty(1 << 27, dtype=torch.float64, device=dev.torch_device).fill_(1.0)
dst = torch.empty_like(src)
for _ in range(3):
    dst.copy_(src)
e0, e1 = events()
e0.record()
for _ in range(args.reps):
    dst.copy_(src)
e1.record()
torch.cuda.synchronize()
copy_gbs = 2 * src.numel() * 8 / (e0.elapsed_time(e1) / args.reps * 1e-3) / 1e9
del src, dst, W
out["delete_rows"] = {"n": n, "j": 0, "ncols": ncols, "us": round(rows_ms * 1e3, 2), "bytes": rows_bytes,
                      "GB_s": round(rows_bytes / (rows_ms * 1e-3) / 1e9, 1), "copy_GB_s": round(copy_gbs, 1),
                      "fraction_of_copy": round(rows_bytes / (rows_ms * 1e-3) / 1e9 / copy_gbs, 3)}

# ---- 2. delete_factor latency ------------------------------------------------------------------------------------------
out["delete_factor_us"] = {}
for nf in (255, 4096):
    fac = f255 if nf == n else DesignFactor(dev, dev.points(cand[np.random.default_rng(1).permutation(ncols)[:nf]]),
                                            CFG["noise"])
    r = dev.zeros(2 * nf)
    times = []
    for rep in range(args.reps + 3):
        Uc = fac.U.clone()
        e0, e1 = events()
        e0.record()
        check(lib.gpx_design_delete_factor(dev.h, ptr(Uc), nf, Uc.shape[1], 0, ptr(r), None, None, None, dev.stream),
              "delete_factor")
        e1.record()
        torch.cuda.synchronize()
        if rep >= 3:
            times.append(e0.elapsed_time(e1) * 1e3)
    out["delete_factor_us"][str(nf)] = {"median": round(float(np.median(times)), 1), "min": round(float(np.min(times)), 1)}
    del fac, Uc

# ---- 3. exchange step vs greedy step, alternated -----------------------------------------------------------------------
base = list(np.random.default_rng(0).permutation(ncols)[:n])
g = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
for i in base:
    g.force(int(i))
snap = g.snapshot()
g.run(N)                                   # the greedy 256th pick, then back to 255 points
x = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
for i in base + [int(g.picks[n].item())]:
    x.force(int(i))
g.restore(snap)


def greedy_step():
    g.run(N)
    g.restore(snap)


def exchange_step():
    x.exchange_step(RTOL)


for fn in (greedy_step, exchange_step):
    fn()
    fn()
torch.cuda.synchronize()
ms = {"greedy": [], "exchange": []}
for _ in range(args.rounds):
    for tag, fn in (("greedy", greedy_step), ("exchange", exchange_step)):
        e0, e1 = events()
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms[tag].append(round(e0.elapsed_time(e1) / args.steps, 3))
out["step_ms"] = ms
out["exchange_over_greedy"] = round(float(np.median(ms["exchange"]) / np.median(ms["greedy"])), 4)
del g, x

# ---- 4. the whole refinement of bench.py's greedy design ---------------------------------------------------------------
torch.cuda.synchronize()
t0 = time.perf_counter()
idx = ed.performGreedyIVARExperimentalDesign(cf, cand, N, returnIndices=True, resident=False)
torch.cuda.synchronize()
greedy_s = time.perf_counter() - t0
greedy_cost = float(cf.lastScores[-1])
t0 = time.perf_counter()
ref = ed.refineGreedyIVARExperimentalDesign(cf, cand, idx, maxSweeps=args.max_sweeps, rtol=RTOL, returnIndices=True,
                                            resident=False)
torch.cuda.synchronize()
refine_s = time.perf_counter() - t0
out["refine"] = {"design": N, "greedy_s": round(greedy_s, 2), "greedy_cost": greedy_cost, "refined_cost": cf.lastCost,
                 "relative_drop": (greedy_cost - cf.lastCost) / greedy_cost, "sweeps": len(cf.lastSwaps),
                 "swaps": cf.lastSwaps, "max_sweeps": args.max_sweeps, "wall_s": round(refine_s, 2),
                 "points_changed": int(len(set(int(i) for i in idx) - set(int(i) for i in ref)))}
line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
