"""Cost and gain of the exchange refinement of greedy MI and maximum-variance designs on one GPU.

    python scripts/exchange_mi_step.py [--reps 20] [--rounds 3] [--steps 10] [--max-sweeps 10] [--out result.json]

MI workload: cfg-4 at its one-GPU size (bench.py's cfg-4 block): 3-D Mehler t = 0.9, noise 1e-2, |V| = 40 000 (pool seed 4),
a 512-point greedy design grown from point 0 by an engine that keeps its factors (keep_factors=True).
1. One exchange step (remove position 0, score, keep-or-swap, take) against one greedy step (score, take at n = 511),
   alternated: --rounds rounds of --steps steps each.  Before each greedy step the last point is removed (untimed).
2. The parts of an exchange step on copies of the engine's state (CUDA events over --reps launches, j = 0):
   the two factor downdates as one launch of two blocks (gpx_design_delete_factors) and as two launches of
   gpx_design_delete_factor; the two row downdates (W / num and Us / pd), which move 16 n |V| bytes each.
3. refineGreedyMIExperimentalDesign of the greedy design (default sweeps): swaps per sweep, I(y_A; y_{V minus A}) before
   and after, wall time (including the O(|V|^3) set-up, timed on its own too).
Variance workload: cfg-3 size (bench.py's cfg-3 block): 5-D Matern 3/2 rho = 1, 1 024 of 250 000 (pool seed 3).
4. A greedy design (the engine loop of performGreedyVarExperimentalDesign), then refineGreedyVarExperimentalDesign: swaps per sweep, log det K_AA before
   and after, wall time.
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
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--max-sweeps", type=int, default=10)
ap.add_argument("--V", type=int, default=40_000)
ap.add_argument("--N", type=int, default=512)
ap.add_argument("--var-C", type=int, default=250_000)
ap.add_argument("--var-N", type=int, default=1024)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import gp as gpmod, kernels  # noqa: E402
from gpexp_b200._lib import check, lib  # noqa: E402
from gpexp_b200.approximation import Space  # noqa: E402
from gpexp_b200.device import Device, ptr  # noqa: E402
from gpexp_b200.engine import GreedyVarEngine  # noqa: E402

ed.VERBOSE = False
RTOL = 1e-8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed(fn, reps, before=None):
    """Mean ms of fn() over reps launches, CUDA events around fn alone (before() runs untimed)."""
    total = 0.0
    for _ in range(reps):
        if before is not None:
            before()
        a, b = events()
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / reps


dev = Device.get(0)
V, N = args.V, args.N
pool = np.random.default_rng(4).standard_normal((V, 3))
kern = kernels.KernelMehlerND([0.9, 0.9, 0.9], 3)
cf = ed.costFunctionGP_MI(gpmod.GP(kern, 1e-2), 1, Space(3, None, None), nmc=V, mcpoints=pool)
out = {"device": gpu_info(),
       "mi_workload": f"cfg-4 one-GPU size: 3-D Mehler t = 0.9, noise 1e-2, |V| = {V}, {N}-point greedy design"}

torch.cuda.synchronize()
t0 = time.perf_counter()
eng = ed._mi_new_engine(cf, N, keep_factors=True)
torch.cuda.synchronize()
out["mi_setup_s"] = time.perf_counter() - t0
t0 = time.perf_counter()
greedy_idx = eng.run(N, start=0)
torch.cuda.synchronize()
out["mi_greedy_s"] = time.perf_counter() - t0
out["mi_greedy"] = eng.mutual_information()

# ---- 1. exchange step against greedy step, alternated ----------------------------------------------------------------
swaps = dev.zeros(1, dtype=torch.int64)
cost = dev.zeros(1)
eng.exchange_step(RTOL, swaps, cost)          # warm-up of every launch of both steps
eng.remove(N - 1)
eng.step()
x_ms, g_ms = [], []
for _ in range(args.rounds):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.exchange_step(RTOL, swaps, cost)
    torch.cuda.synchronize()
    x_ms.append((time.perf_counter() - t0) * 1e3 / args.steps)
    t = 0.0
    for _ in range(args.steps):
        eng.remove(N - 1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.step()
        torch.cuda.synchronize()
        t += time.perf_counter() - t0
    g_ms.append(t * 1e3 / args.steps)
out["exchange_step_ms"] = x_ms
out["greedy_step_ms"] = g_ms
out["exchange_over_greedy"] = float(np.mean(x_ms) / np.mean(g_ms))

# ---- 2. parts of an exchange step (j = 0, n = N) on copies of the state ------------------------------------------------
n, ld, nloc = eng.n, eng.ld, eng.nloc
ldu = eng.UA.shape[1]
UA0, UQ0 = eng.UA.clone(), eng.UQ.clone()
UA, UQ = UA0.clone(), UQ0.clone()
rotA, rotQ = dev.zeros(2 * N), dev.zeros(2 * N)
W, Us, num, pd = eng.W.clone(), eng.Us.clone(), eng.num.clone(), eng.pd.clone()


def fresh():
    UA.copy_(UA0)
    UQ.copy_(UQ0)


def fused():
    check(lib.gpx_design_delete_factors(dev.h, n, 0, ptr(UA), ldu, ptr(rotA), None, None, None, ptr(UQ), ldu, ptr(rotQ),
                                        dev.stream), "gpx_design_delete_factors")


def separate():
    check(lib.gpx_design_delete_factor(dev.h, ptr(UA), n, ldu, 0, ptr(rotA), None, None, None, dev.stream), "delete_factor")
    check(lib.gpx_design_delete_factor(dev.h, ptr(UQ), n, ldu, 0, ptr(rotQ), None, None, None, dev.stream), "delete_factor")


def rows():
    check(lib.gpx_design_delete_rows(dev.h, ptr(rotA), 0, n, ptr(W), ld, nloc, ptr(num), dev.stream), "delete_rows")
    check(lib.gpx_design_delete_rows(dev.h, ptr(rotQ), 0, n, ptr(Us), ld, nloc, ptr(pd), dev.stream), "delete_rows")


fused()
separate()
rows()
out["factor_downdates_fused_ms"] = timed(fused, args.reps, fresh)
out["factor_downdates_two_launches_ms"] = timed(separate, args.reps, fresh)
rows_ms = timed(rows, args.reps)
out["row_downdates_ms"] = rows_ms
row_bytes = 2 * 16.0 * n * nloc
out["row_downdates_bytes"] = row_bytes
out["row_downdates_TBps"] = row_bytes / (rows_ms * 1e-3) / 1e12
step = float(np.mean(x_ms))
out["exchange_step_split_ms"] = {"factor_downdates": out["factor_downdates_fused_ms"], "row_downdates": rows_ms,
                                 "rest": step - out["factor_downdates_fused_ms"] - rows_ms}
out["two_launch_downdates_share_of_step"] = out["factor_downdates_two_launches_ms"] / (
    step - out["factor_downdates_fused_ms"] + out["factor_downdates_two_launches_ms"])
del eng, UA0, UQ0, UA, UQ, W, Us, num, pd
torch.cuda.empty_cache()

# ---- 3. full MI refinement of the greedy design ------------------------------------------------------------------------
torch.cuda.synchronize()
t0 = time.perf_counter()
ref_idx = ed.refineGreedyMIExperimentalDesign(cf, greedy_idx, maxSweeps=args.max_sweeps, rtol=RTOL, returnIndices=True)
torch.cuda.synchronize()
out["mi_refine"] = {"wall_s_including_setup": time.perf_counter() - t0, "swaps_per_sweep": cf.lastSwaps,
                    "mi_before": out["mi_greedy"], "mi_after": cf.lastMI,
                    "changed_points": int(len(set(greedy_idx.tolist()) - set(int(i) for i in ref_idx)))}
torch.cuda.empty_cache()

# ---- 4. variance refinement at cfg-3 size ------------------------------------------------------------------------------
C, NV = args.var_C, args.var_N
vpool = np.random.default_rng(3).uniform(-1, 1, (C, 5))
vk = kernels.KernelIsoMatern(1.0, 1.0, 5)
out["var_workload"] = f"cfg-3 size: 5-D Matern 3/2 rho = 1, {NV} of {C} candidates, nugget 0"
vdev = vk._bind()
torch.cuda.synchronize()
t0 = time.perf_counter()
keep = [int(i) for i in GreedyVarEngine(vdev, vdev.points(vpool), NV).run(NV)]   # performGreedyVarExperimentalDesign's loop
torch.cuda.synchronize()
out["var_greedy_s"] = time.perf_counter() - t0
_, info0 = ed.refineGreedyVarExperimentalDesign(vk, vpool, keep, maxSweeps=0, returnIndices=True, returnInfo=True)
torch.cuda.synchronize()
t0 = time.perf_counter()
vidx, info = ed.refineGreedyVarExperimentalDesign(vk, vpool, keep, maxSweeps=args.max_sweeps, rtol=RTOL,
                                                  returnIndices=True, returnInfo=True)
torch.cuda.synchronize()
out["var_refine"] = {"wall_s": time.perf_counter() - t0, "swaps_per_sweep": info["swaps"],
                     "logdet_before": info0["logdet"], "logdet_after": info["logdet"],
                     "changed_points": int(len(set(keep) - set(int(i) for i in vidx)))}
print(out["device"])
line = json.dumps(out)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
