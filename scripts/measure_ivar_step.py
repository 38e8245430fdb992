"""cfg-2's greedy IVAR step with the integral over U[-1, 1]^2 in closed form (costFunctionGP_IVAR.measure) against the
Monte-Carlo step on the INT8 core: 100 000 candidates, 2-D SE cl = (0.06, 0.09), signal 1, noise 1e-6, n = 255 -> 256.

    python scripts/measure_ivar_step.py [--rounds 3] [--out result.json]

Each round, alternated in one run:
  exact   a fresh MeasureIVAREngine grows the greedy design to 255 points, then the step 255 -> 256 is timed alone
          (CUDA events: scoring pass with the Y update, W and Z row appends, Psi row); then the whole 256-point design
          from an empty state is timed (one engine, 256 steps, synchronised at the end).
  mc      GreedyIVAREngine with cfg-2's 100 000 integration points, a seeded random 255-point design loaded through
          Gram + Cholesky + TRSM, one INT8-core step 255 -> 256 (restore() between repetitions), as
          scripts/matern_ivar_step.py times it.
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
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--mc-steps", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import _lib, gp as gpmod, kernels  # noqa: E402
from gpexp_b200.approximation import Space, UniformMeasure  # noqa: E402
from gpexp_b200.device import Device  # noqa: E402
from gpexp_b200.engine import DesignFactor  # noqa: E402

ed.VERBOSE = False
C = M = 100_000
N, noise = 256, 1e-6
rng = np.random.default_rng(2)
cand = rng.uniform(-1.0, 1.0, (C, 2))
mc = rng.uniform(-1.0, 1.0, (M, 2))
design = cand[np.random.default_rng(0).permutation(C)[: N - 1]]
kern = kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


dev = Device.get(0)
cf_exact = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), measure=UniformMeasure(-1.0, 1.0))
cf_mc = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), mcPoints=mc)
_lib.check(_lib.lib.gpx_set_ivar_core(dev.h, 2), "gpx_set_ivar_core")
mc_eng = ed.beginGreedyIVARExperimentalDesign(cf_mc, cand, N, resident=False)
mc_eng.load_design(DesignFactor(dev, dev.points(design), noise))
mc_snap = mc_eng.snapshot()


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def exact_round():
    eng = ed.beginGreedyIVARExperimentalDesign(cf_exact, cand, N)
    eng.run(N - 1)
    torch.cuda.synchronize()
    e0, e1 = events()
    e0.record()
    eng.step()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1)
    eng2 = ed.beginGreedyIVARExperimentalDesign(cf_exact, cand, N)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng2.run(N)
    torch.cuda.synchronize()
    design_ms = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(eng.indices(), eng2.indices())
    return step_ms, design_ms, eng2


def mc_round():
    kern._bind(dev)
    mc_eng.run(N)
    mc_eng.restore(mc_snap)
    torch.cuda.synchronize()
    e0, e1 = events()
    e0.record()
    for _ in range(args.mc_steps):
        mc_eng.run(N)
        mc_eng.restore(mc_snap)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.mc_steps


exact_round()   # warm-up: modules, allocations
mc_round()
step_ms, design_ms, mc_ms = [], [], []
for _ in range(args.rounds):
    s, d, eng = exact_round()
    step_ms.append(s)
    design_ms.append(d)
    mc_ms.append(mc_round())

# traffic of the exact step at n = 255 (doubles): W and Z appends read n C each, the scoring pass reads 3 n C and writes n C
n = N - 1
step_bytes = 8 * C * (n + n + 3 * n + n)
out = {"device": gpu_info(),
       "workload": "cfg-2 greedy IVAR, C = 100 000 candidates, 2-D SE cl = (0.06, 0.09), signal 1, noise 1e-6, "
                   "exact integral over U[-1, 1]^2 vs M = 100 000 Monte-Carlo points on the INT8 core",
       "exact_step_255_to_256_ms": [round(x, 4) for x in step_ms],
       "exact_design_256_ms": [round(x, 2) for x in design_ms],
       "mc_i8_step_255_to_256_ms": [round(x, 3) for x in mc_ms],
       "step_speedup": round(float(np.median(mc_ms) / np.median(step_ms)), 1),
       "exact_step_bytes": step_bytes,
       "exact_step_GBps": round(step_bytes / (np.median(step_ms) * 1e-3) / 1e9, 1),
       "exact_cost_of_256_point_design": float(eng.pick_scores[N - 1].item())}
line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
