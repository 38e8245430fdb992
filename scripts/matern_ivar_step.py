"""cfg-2's final greedy IVAR step (100 000 candidates x 100 000 integration points, 2-D, n = 255 -> 256) for the
squared-exponential kernel of cfg-2 (cl = 0.06, 0.09) against the isotropic Matern kernels nu = 1/2, 3/2 and 5/2, on the
INT8 core and on the DMMA core.

    python scripts/matern_ivar_step.py [--steps 10] [--rounds 3] [--e2e 3] [--out result.json]

One rho = 0.2 for the three Matern kernels: the 255-point design's Gram + 1e-6 I then has cond 1e3 (nu = 1/2), 1e5
(3/2) and 6e5 (5/2), against 1.5e4 for SE; the script computes and reports each.  The design is a seeded random set of
255 candidates loaded through Gram + Cholesky + TRSM (the state shape of bench.py --quick-design).  Every engine
(kernel x core) is built once; the steps are then timed in turn, `--rounds` times, each as `--steps` C-side steps of
255 -> 256 with restore() in between (CUDA events).  The prologue form each kernel's contraction runs (expanded or
difference) is reported: nu = 1/2 always takes the difference form.  scoreCandidatesIVAR (host buffers in, costs out) is
timed end to end per kernel on the default core.  Prints the device name and power limit (a query only) and one JSON
line, which --out also writes to a file."""
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
N, noise, RHO = 256, 1e-6, 0.2
rng = np.random.default_rng(2)
cand = rng.uniform(-1.0, 1.0, (C, 2))
mc = rng.uniform(-1.0, 1.0, (M, 2))
design = cand[np.random.default_rng(0).permutation(C)[: N - 1]]
CORES = {"i8": 2, "dmma": 1}
KERNELS = {"se": kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2),
           "matern12": kernels.KernelIsoMatern(RHO, 1.0, 2, nu=0.5),
           "matern32": kernels.KernelIsoMatern(RHO, 1.0, 2, nu=1.5),
           "matern52": kernels.KernelIsoMatern(RHO, 1.0, 2, nu=2.5)}
FORMS = {_lib.PRO_EXPANDED: "expanded", _lib.PRO_DIFF: "difference"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


def gram_cond(kern):
    """Condition number of the design's Gram + noise, from the device Gram."""
    from gpexp_b200 import gp_kernel_utilities as gku
    return float(np.linalg.cond(gku.calculateCovarianceMatrix(kern, design, noise)))


dev = Device.get(0)
engines, snaps, forms, conds = {}, {}, {}, {}
for ktag, kern in KERNELS.items():
    conds[ktag] = gram_cond(kern)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), mcPoints=mc)
    for core in CORES:
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
        eng.load_design(DesignFactor(dev, dev.points(design), noise))
        engines[(core, ktag)], snaps[(core, ktag)] = eng, eng.snapshot()
        kern._bind(dev)
        forms[ktag] = FORMS[eng.prologue()[0]]


def step(key):
    # the engines share the device handle, which holds one covariance function: bind this engine's (a no-op when it is
    # already bound; a switch re-prepares the expanded-form operands on the next step, so the timed loop warms up first)
    KERNELS[key[1]]._bind(dev)
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
        step(key)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(key)
        e1.record()
        torch.cuda.synchronize()
        ms[key].append(e0.elapsed_time(e1) / args.steps)
_lib.check(_lib.lib.gpx_set_ivar_core(dev.h, CORES["i8"]), "gpx_set_ivar_core")
picks = {f"{c}_{k}": int(engines[(c, k)].picks[N - 1].item()) for c, k in engines}   # restore() keeps the last pick

e2e = {k: [] for k in KERNELS}
for _ in range(args.e2e):
    for ktag, kern in KERNELS.items():
        cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(2, None, None), mcPoints=mc)
        if not e2e[ktag]:
            ed.scoreCandidatesIVAR(cf, design, cand)   # warm-up on the first round
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ed.scoreCandidatesIVAR(cf, design, cand)
        torch.cuda.synchronize()
        e2e[ktag].append((time.perf_counter() - t0) * 1e3)

out = {"device": gpu_info(), "workload": "cfg-2 greedy IVAR step n = 255 -> 256, C = M = 100 000, random 255-point design, "
                                         "SE cl = (0.06, 0.09); Matern rho = 0.2, signal 1, noise 1e-6",
       "steps_per_round": args.steps, "gram_cond": {k: float(f"{v:.3g}") for k, v in conds.items()}, "prologue": forms}
for (c, k), v in ms.items():
    out[f"step_ms_{c}_{k}"] = [round(x, 3) for x in v]
for k, v in e2e.items():
    out[f"e2e_ms_{k}"] = [round(x, 2) for x in v]
out["pick_256"] = picks
line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
