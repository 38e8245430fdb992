"""A/B of the two IVAR scoring cores (GPX_CORE_DMMA, GPX_CORE_I8) on the same engine state, one GPU.

usage: python scripts/ivar_core_ab.py [--out FILE] [--reps R]

For each shape it loads a seeded random design through DesignFactor (the state shape of a greedy step at design size n),
then times eng.score() -- slicing + contraction kernel + finalisation -- with CUDA events, alternating the cores, and
compares the scores of the two cores.  A separate profiled call gives the device time of the slicing pass and of the
INT8 contraction kernel alone.  Shapes: cfg-2 (d = 2 SE, 100k x 100k) at n = 255 and 1023, and the cfg-5 shape
(d = 10, 125k integration points) with a 25k-candidate slice at n = 4095.
Rates: the FP64-equivalent rate counts 2 M C n flop; the INT8 rate counts 2 M C ldk x 28 integer ops (ldk = n rounded
up to 64: the K extent the tensor cores actually run, 28 slice products each).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import gpexp_b200.experimentalDesign as ed  # noqa: E402
from gpexp_b200 import gp as gpmod, kernels  # noqa: E402
from gpexp_b200._lib import check, lib  # noqa: E402
from gpexp_b200.approximation import Space  # noqa: E402
from gpexp_b200.device import Device  # noqa: E402
from gpexp_b200.engine import DesignFactor  # noqa: E402

CORES = {"dmma": 1, "i8": 2}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def i8_kernel_times(eng):
    """Device time (ms) of the slicing pass (both sides) and of the INT8 contraction in one eng.score(), from a separate
    profiled call."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.score()
        torch.cuda.synchronize()
    out = {"ivar_slice_kernel": 0.0, "ivar_i8_kernel": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        t = ev.cuda_time_total if t is None else t
        for name in out:
            if name in ev.key:
                out[name] += t / 1e3
    return out


def run_shape(name, d, C, M, n, reps, seed=0):
    rng = np.random.default_rng(seed)
    cand = rng.uniform(-1.0, 1.0, (C, d))
    mc = rng.uniform(-1.0, 1.0, (M, d))
    cl = [0.06, 0.09] if d == 2 else [0.5] * d
    kern = kernels.KernelSquaredExponential(cl, 1.0, d)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, 1e-6), 1, Space(d, None, None), mcPoints=mc)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, n + 1, resident=False)
    dev = Device.get()
    pick = rng.permutation(C)[:n]
    eng.load_design(DesignFactor(dev, dev.points(cand[pick]), 1e-6))
    scores, times = {}, {k: [] for k in CORES}
    for core, code in CORES.items():  # warm-up + outputs
        check(lib.gpx_set_ivar_core(dev.h, code), "gpx_set_ivar_core")
        eng.score()
        torch.cuda.synchronize()
        scores[core] = eng.scores[:C].cpu().numpy().copy()
    for _ in range(reps):
        for core, code in CORES.items():
            check(lib.gpx_set_ivar_core(dev.h, code), "gpx_set_ivar_core")
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            eng.score()
            ev[1].record()
            torch.cuda.synchronize()
            times[core].append(ev[0].elapsed_time(ev[1]))
    check(lib.gpx_set_ivar_core(dev.h, CORES["i8"]), "gpx_set_ivar_core")
    kernel_ms = i8_kernel_times(eng)
    a, b = scores["dmma"], scores["i8"]
    rel = float(np.max(np.abs(a - b) / np.abs(a)))
    ldk = (n + 63) // 64 * 64
    out = {"shape": name, "d": d, "C": C, "M": M, "n": n, "ms": {k: v for k, v in times.items()},
           "max_rel_score_diff": rel, "argmin_equal": int(np.argmin(a)) == int(np.argmin(b)), "i8_kernel_ms": kernel_ms}
    for core in CORES:
        t = float(np.median(times[core])) * 1e-3
        out[f"{core}_fp64_equiv_tflops"] = 2.0 * M * C * n / t / 1e12
    out["i8_int_tops"] = 2.0 * M * C * ldk * 28 / (float(np.median(times["i8"])) * 1e-3) / 1e12
    print(json.dumps(out), flush=True)
    del eng
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="cfg2_255,cfg2_1023,cfg5_4095")
    args = ap.parse_args()
    ed.VERBOSE = False
    res = {"card": card(), "runs": []}
    print(json.dumps({"card": res["card"]}), flush=True)
    shapes = {"small": ("small", 2, 3_000, 2_000, 33), "cfg2_255": ("cfg2", 2, 100_000, 100_000, 255),
              "cfg2_1023": ("cfg2", 2, 100_000, 100_000, 1023), "cfg5_4095": ("cfg5-slice", 10, 25_000, 125_000, 4095)}
    for key in args.shapes.split(","):
        res["runs"].append(run_shape(*shapes[key], args.reps))
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
