"""Greedy IVAR step with the integral over N(0, I_3) in closed form for a Mehler kernel (cfg-4's kernel family) against the
Monte-Carlo step on the INT8 core, and an A/B of the squared-exponential measure step against a previous build.

    python scripts/mehler_measure_step.py [--rounds 3] [--prev-lib OLD.so] [--out result.json]

Workload: 3-D Mehler t = (0.9, 0.9, 0.9), measure N(0, I_3), noise 1e-2, C = 100 000 candidates drawn from N(0, I_3),
a seeded random 255-point design taken from the candidates.  Each round, alternated in one run:
  exact   MeasureIVAREngine: the 255 design points appended one by one through force() (each a scoring pass and an
          append, as a greedy step), then the step 255 -> 256 timed alone with CUDA events (scoring pass with the Y
          update, W and Z row appends, Psi row).  Then the whole 256-point greedy design from an empty state (one engine, 256 steps,
          synchronised at the end, host clock).
  mc      GreedyIVAREngine with M = 100 000 points drawn from N(0, I_3), the 255-point design loaded, one INT8-core step
          255 -> 256 (restore() between repetitions).  Its estimator of the Mehler IVAR has infinite variance at t = 0.9
          (var_D(x) grows like exp(x^2 t / (1 + t)) under the Gaussian); the step is timed, not trusted.
SE A/B (--prev-lib): the same exact step for a 3-D SE kernel, cl = 0.3, signal 1, at the same shape, run in child
processes alternately against the tree's library and OLD.so (GPX_LIB), each reporting its step times and a SHA-256 of
the 100 000 scores of that step and of the pick.
Reads the device name and power limit (a query only) and prints one JSON line, which --out also writes to a file."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--mc-steps", type=int, default=5)
ap.add_argument("--prev-lib", default=None, help="libgpexp_b200.so of the previous build for the SE A/B")
ap.add_argument("--se-child", action="store_true", help=argparse.SUPPRESS)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import torch  # noqa: E402

import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import _lib, gp as gpmod, kernels  # noqa: E402
from gpexp_b200.approximation import GaussianMeasure, Space  # noqa: E402
from gpexp_b200.device import Device  # noqa: E402
from gpexp_b200.engine import DesignFactor  # noqa: E402

ed.VERBOSE = False
C = M = 100_000
N, D, noise = 256, 3, 1e-2
rng = np.random.default_rng(4)
cand = rng.normal(size=(C, D))
mc = rng.normal(size=(M, D))
perm = np.random.default_rng(0).permutation(C)[: N - 1]
design = cand[perm]
measure = GaussianMeasure(0.0, 1.0)
dev = Device.get(0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (power limit not available)"


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def exact_step(cf):
    """(step ms, scores of the step, pick) for the step 255 -> 256 from the random design."""
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N)
    for p in perm:
        eng.force(int(p))
    torch.cuda.synchronize()
    e0, e1 = events()
    e0.record()
    eng.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), eng.scores[:C].cpu().numpy(), int(eng.indices()[-1])


def se_child():
    kern = kernels.KernelSquaredExponential([0.3], 1.0, D)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(D, None, None), measure=measure)
    exact_step(cf)   # warm-up
    times, digest = [], None
    for _ in range(args.rounds):
        ms, scores, pick = exact_step(cf)
        times.append(ms)
        h = hashlib.sha256(scores.tobytes() + np.int64(pick).tobytes()).hexdigest()
        assert digest in (None, h), "SE measure step scores differ from run to run"
        digest = h
    print(json.dumps({"lib": _lib.LIB_PATH, "se_step_ms": times, "se_scores_sha256": digest}), flush=True)


if args.se_child:
    se_child()
    sys.exit(0)

kern = kernels.KernelMehlerND([0.9] * D, D)
cf_exact = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(D, None, None), measure=measure)
cf_mc = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(D, None, None), mcPoints=mc)
_lib.check(_lib.lib.gpx_set_ivar_core(dev.h, 2), "gpx_set_ivar_core")
mc_eng = ed.beginGreedyIVARExperimentalDesign(cf_mc, cand, N, resident=False)
mc_eng.load_design(DesignFactor(dev, dev.points(design), noise))
mc_snap = mc_eng.snapshot()


def exact_round():
    step_ms, _, _ = exact_step(cf_exact)
    eng = ed.beginGreedyIVARExperimentalDesign(cf_exact, cand, N)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.run(N)
    torch.cuda.synchronize()
    return step_ms, (time.perf_counter() - t0) * 1e3, eng


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

n = N - 1
step_bytes = 8 * C * (n + n + 3 * n + n)   # W and Z appends read n C each; the scoring pass reads 3 n C, writes n C
out = {"device": gpu_info(),
       "workload": "3-D Mehler t = (0.9, 0.9, 0.9), C = 100 000 candidates ~ N(0, I3), noise 1e-2, random 255-point "
                   "design: exact integral over N(0, I3) vs M = 100 000 Monte-Carlo points ~ N(0, I3) on the INT8 core",
       "exact_step_255_to_256_ms": [round(x, 4) for x in step_ms],
       "exact_design_256_ms": [round(x, 2) for x in design_ms],
       "mc_i8_step_255_to_256_ms": [round(x, 3) for x in mc_ms],
       "step_speedup": round(float(np.median(mc_ms) / np.median(step_ms)), 1),
       "exact_step_bytes": step_bytes,
       "exact_step_GBps": round(step_bytes / (np.median(step_ms) * 1e-3) / 1e9, 1),
       "exact_cost_of_256_point_design": float(eng.pick_scores[N - 1].item())}

if args.prev_lib:
    ab = {"new": [], "prev": []}
    for _ in range(args.rounds):
        for name, lib in (("prev", args.prev_lib), ("new", None)):
            env = dict(os.environ)
            env.pop("GPX_LIB", None)
            if lib:
                env["GPX_LIB"] = os.path.abspath(lib)
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--se-child", "--rounds", "3"], env=env,
                                 capture_output=True, text=True, check=True)
            ab[name].append(json.loads(res.stdout.strip().splitlines()[-1]))
    hashes = {name: sorted({r["se_scores_sha256"] for r in runs}) for name, runs in ab.items()}
    out["se_ab"] = {"workload": "3-D SE cl = 0.3, signal 1, same candidates, design, noise and measure; exact step "
                                "255 -> 256, 3 child processes per build, alternated",
                    "new_step_ms": [round(x, 4) for r in ab["new"] for x in r["se_step_ms"]],
                    "prev_step_ms": [round(x, 4) for r in ab["prev"] for x in r["se_step_ms"]],
                    "new_scores_sha256": hashes["new"], "prev_scores_sha256": hashes["prev"],
                    "bit_identical": hashes["new"] == hashes["prev"] and len(hashes["new"]) == 1}

line = json.dumps(out)
print(line, flush=True)
if args.out:
    with open(args.out, "w") as f:
        f.write(line + "\n")
