"""cfg-2's final greedy IVAR step (100 000 candidates x 100 000 integration points, 2-D ARD SE cl = (0.06, 0.09),
n = 255 -> 256) with a scalar noise and with a heteroscedastic noise function, on the same design.

    python scripts/hetero_ivar_step.py [--steps 10] [--rounds 3] [--e2e 3] [--out result.json]

Scalar noise 1e-6 against nu(x) = 1e-6 (1 + x0^2).  The design is a seeded random set of 255 candidates loaded through
Gram + Cholesky + TRSM (the state shape of bench.py --quick-design).  Both engines are built once; the two steps are then
timed in turn, `--rounds` times, each as `--steps` C-side steps of 255 -> 256 with restore() in between (CUDA events).
scoreCandidatesIVAR (host buffers in, costs out) is timed end to end both ways as well.  Prints the device name and power
limit (a query only) and one JSON line, which --out also writes to a file."""
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
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--e2e", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import gp as gpmod, kernels  # noqa: E402
from gpexp_b200.approximation import Space  # noqa: E402
from gpexp_b200.device import Device  # noqa: E402
from gpexp_b200.engine import DesignFactor  # noqa: E402

ed.VERBOSE = False
C = M = 100_000
N, noise = 256, 1e-6
rng = np.random.default_rng(2)
cand = rng.uniform(-1.0, 1.0, (C, 2))
mc = rng.uniform(-1.0, 1.0, (M, 2))
design = cand[np.random.default_rng(0).permutation(C)[: N - 1]]


def nu(p):
    return 1e-6 * (1.0 + p[:, 0] ** 2)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


dev = Device.get(0)
kern = kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2)
spaces = {"scalar": Space(2, None, None), "hetero": Space(2, None, None, noise=nu)}
engines, snaps = {}, {}
for tag, space in spaces.items():
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, space, mcPoints=mc)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
    eng.load_design(DesignFactor(dev, dev.points(design), noise if tag == "scalar" else nu(design)))
    engines[tag], snaps[tag] = eng, eng.snapshot()


def step(tag):
    eng = engines[tag]
    eng.run(N)
    eng.restore(snaps[tag])


for tag in engines:   # warm-up: modules, INT8 scratch, prologue operands
    step(tag)
    step(tag)
torch.cuda.synchronize()
ms = {tag: [] for tag in engines}
for _ in range(args.rounds):
    for tag in engines:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(tag)
        e1.record()
        torch.cuda.synchronize()
        ms[tag].append(e0.elapsed_time(e1) / args.steps)
picks = {tag: int(engines[tag].picks[N - 1].item()) for tag in engines}   # restore() keeps the last step's pick

e2e = {tag: [] for tag in engines}
for tag, space in spaces.items():
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, space, mcPoints=mc)
    ed.scoreCandidatesIVAR(cf, design, cand)   # warm-up
    torch.cuda.synchronize()
    for _ in range(args.e2e):
        t0 = time.perf_counter()
        ed.scoreCandidatesIVAR(cf, design, cand)
        torch.cuda.synchronize()
        e2e[tag].append((time.perf_counter() - t0) * 1e3)

out = {"device": gpu_info(), "workload": "cfg-2 greedy IVAR step n = 255 -> 256, C = M = 100 000, random 255-point design",
       "steps_per_round": args.steps,
       "step_ms_scalar": [round(x, 3) for x in ms["scalar"]], "step_ms_hetero": [round(x, 3) for x in ms["hetero"]],
       "e2e_ms_scalar": [round(x, 2) for x in e2e["scalar"]], "e2e_ms_hetero": [round(x, 2) for x in e2e["hetero"]],
       "pick_256": picks}
line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
