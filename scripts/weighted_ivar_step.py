"""cfg-2's final greedy IVAR step (100 000 candidates x 100 000 integration points, 2-D ARD SE cl = (0.06, 0.09),
n = 255 -> 256) with the plain Monte-Carlo mean and with weighted integration points, on the same design, on the INT8
core and on the DMMA core.

    python scripts/weighted_ivar_step.py [--steps 10] [--rounds 3] [--e2e 3] [--out result.json]

Weights w(x) = exp(-|x|^2) / M against none.  The design is a seeded random set of 255 candidates loaded through
Gram + Cholesky + TRSM (the state shape of bench.py --quick-design).  The four engines (core x weighting) are built once;
the steps are then timed in turn, `--rounds` times, each as `--steps` C-side steps of 255 -> 256 with restore() in between
(CUDA events).  scoreCandidatesIVAR (host buffers in, costs out) is timed end to end both ways on the default core.  Prints
the device name and power limit (a query only) and one JSON line, which --out also writes to a file."""
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
from gpexp_b200 import _lib, gp as gpmod, kernels  # noqa: E402
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
weights = np.exp(-np.sum(mc * mc, axis=1)) / M
CORES = {"i8": 2, "dmma": 1}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


dev = Device.get(0)
kern = kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2)
engines, snaps = {}, {}
for wtag, w in (("plain", None), ("weighted", weights)):
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), mcPoints=mc, mcWeights=w)
    for core in CORES:
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
        eng.load_design(DesignFactor(dev, dev.points(design), noise))
        engines[(core, wtag)], snaps[(core, wtag)] = eng, eng.snapshot()


def step(key):
    _lib.check(_lib.lib.gpx_set_ivar_core(dev.h, CORES[key[0]]), "gpx_set_ivar_core")
    eng = engines[key]
    eng.run(N)
    eng.restore(snaps[key])


for key in engines:   # warm-up: modules, INT8 scratch, prologue operands
    step(key)
    step(key)
torch.cuda.synchronize()
ms = {key: [] for key in engines}
for _ in range(args.rounds):
    for key in engines:
        _lib.check(_lib.lib.gpx_set_ivar_core(dev.h, CORES[key[0]]), "gpx_set_ivar_core")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(key)
        e1.record()
        torch.cuda.synchronize()
        ms[key].append(e0.elapsed_time(e1) / args.steps)
_lib.check(_lib.lib.gpx_set_ivar_core(dev.h, CORES["i8"]), "gpx_set_ivar_core")
picks = {f"{c}_{w}": int(engines[(c, w)].picks[N - 1].item()) for c, w in engines}   # restore() keeps the last pick

e2e = {"plain": [], "weighted": []}
for _ in range(args.e2e):
    for wtag, w in (("plain", None), ("weighted", weights)):
        cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), mcPoints=mc, mcWeights=w)
        if not e2e[wtag]:
            ed.scoreCandidatesIVAR(cf, design, cand)   # warm-up on the first round
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ed.scoreCandidatesIVAR(cf, design, cand)
        torch.cuda.synchronize()
        e2e[wtag].append((time.perf_counter() - t0) * 1e3)

out = {"device": gpu_info(), "workload": "cfg-2 greedy IVAR step n = 255 -> 256, C = M = 100 000, random 255-point design, "
                                         "w(x) = exp(-|x|^2) / M",
       "steps_per_round": args.steps}
for (c, w), v in ms.items():
    out[f"step_ms_{c}_{w}"] = [round(x, 3) for x in v]
out["e2e_ms_plain"] = [round(x, 2) for x in e2e["plain"]]
out["e2e_ms_weighted"] = [round(x, 2) for x in e2e["weighted"]]
out["pick_256"] = picks
line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
