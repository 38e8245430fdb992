#!/usr/bin/env python
"""bench.py -- candidates scored per second per greedy IVAR step (BASELINE.json metric).

Workload: BASELINE.json configs[1] (cfg-2) -- 2-D ARD squared-exponential, cl=(0.06, 0.09), signal 1, noise 1e-6, greedy
IVAR design of 256 points from C = 100 000 candidates x M = 100 000 Monte-Carlo integration points (SURVEY.md 8d, seed 2).
The whole 256-point design is grown once on the device through the public driver object
(`experimentalDesign.beginGreedyIVARExperimentalDesign(...).run(255)`, reported as `design_total_s`); a timed STEP is the
final, most expensive greedy step of that design: `run(256)` = score all candidates at design size n = 255 with the FP64 DMMA
contraction, arg-min, exchange (N > 1), append the chosen row to W_C / W_M; the state is then restored (two 0.8 MB copies,
inside the timed region).

N > 1 is STRONG scaling: the same 100 000 candidates are split into N contiguous blocks (integration points replicated), one
NCCL all-gather of pivot records per step.  Every N > 1 line also carries a `parity` block (sharded greedy IVAR / greedy
variance / greedy MI on small seeded pools against the CPU oracle, all ranks agreeing) and, at N = 8, `extras.cfg5`: the
north-star step (10-D ARD, n = 4096, 1 000 000 candidates x 100 000 MC points).  The other BASELINE configurations ride in
`extras` of every line: cfg-1 (N = 1), cfg-3 (whole 1 024-point conditional-entropy design from 250 000 candidates) and
cfg-4 (512-point MI design; pool 40 000 / 80 000 / 120 000 / 200 000 on 1 / 2 / 4 / 8 GPUs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned to its caller as float64 .npy files (see dump_step_outputs);
the inputs are seeded, so two builds run with the same arguments can be compared output for output.

--impl reference times the UNMODIFIED reference (baseline/_ref/gpExp, staged by __graft_entry__.build(); the line-by-line
oracle port if it is absent) on the host cores: costFunctionGP_IVAR.evaluate (experimentalDesign.py:79-117 ->
gp.py:156-259) of design + [c], one candidate per worker process per step.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(d=2, cl=[0.06, 0.09], signal=1.0, noise=1e-6, C=100_000, M=100_000, N=256, seed=2)
METRIC = "candidates scored/sec per greedy IVAR step"
UNIT = "candidates/s"
WORKLOAD = ("cfg-2: 2-D ARD squared-exponential cl=(0.06,0.09), IVAR greedy step at design size 255->256, "
            "100k candidates x 100k MC integration points, noise 1e-6, float64")


def config_dict(world):
    """The SAME dictionary for both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "candidates_total": CFG["C"], "mc_points": CFG["M"], "design_size": CFG["N"] - 1,
            "l2": "inputs larger than L2 (W_M + W_C >= 230 MB per GPU vs 126 MB L2)",
            "sharding": f"candidates/{world}, integration points replicated"}


def make_inputs():
    rng = np.random.default_rng(CFG["seed"])
    cand = rng.uniform(-1.0, 1.0, (CFG["C"], CFG["d"]))
    mc = rng.uniform(-1.0, 1.0, (CFG["M"], CFG["d"]))
    return cand, mc


def dump_step_outputs(out_dir, eng, n_points, total_c, torch, dist, world, rank):
    """What a caller of the timed step `eng.run(256)` receives, taken after the last timed step (restore() resets only the
    running variances, so these still hold that step's results): the 256 design indices (exact in float64), the cost of
    each pick, the pivot var_D(p) + noise of each pick, and the cost of every one of the candidates at design size 255.
    0.8 MB in all at cfg-2 size.  With N > 1 the candidate costs of the ranks' contiguous blocks are gathered in global
    order and rank 0 writes."""
    scores = eng.scores[: eng.cand.n]
    if world > 1:
        from gpexp_b200.engine import Shard
        width = -(-total_c // world)
        mine = torch.zeros(width, dtype=torch.float64, device=scores.device)
        mine[: scores.numel()] = scores
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine)
        sizes = [hi - lo for lo, hi in (Shard.split(total_c, world, r) for r in range(world))]
        scores = torch.cat([p[:s] for p, s in zip(parts, sizes)])
    if rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    out = {"indices": eng.picks[:n_points], "pick_scores": eng.pick_scores[:n_points], "pivots": eng.pick_pivots[:n_points],
           "scores": scores}
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


# ---------------------------------------------------------------------------------------------
# reference arm: the unmodified reference on the host cores
# ---------------------------------------------------------------------------------------------
_REF = {}


def _ref_worker_init(path, design, mc):
    import warnings
    warnings.filterwarnings("ignore")
    os.environ["OMP_NUM_THREADS"] = "1"
    kind = "port"
    if path:
        sys.path.insert(0, path)
        try:
            import gpExp.experimentalDesign as red
            import gpExp.gp as rgp
            import gpExp.kernels as rk
            from gpExp.approximation import Space
            kern = rk.KernelSquaredExponential(list(CFG["cl"]), CFG["signal"], CFG["d"])
            gp = rgp.GP(kern, float(CFG["noise"]))
            cf = red.costFunctionGP_IVAR(gp, design.shape[0] + 1, Space(CFG["d"], None, None, noise=None), mcPoints=mc)
            _REF.update(cf=cf)
            kind = "reference"
        except ImportError:
            pass
    if kind == "port":
        from oracle import gpexp_oracle as orc
        _REF.update(orc=orc, kern=orc.KernelSpec.se(CFG["cl"], CFG["signal"], CFG["d"]))
    _REF.update(kind=kind, design=design, mc=mc)
    try:
        from threadpoolctl import threadpool_limits
        _REF["limit"] = threadpool_limits(limits=1)  # one BLAS thread per worker: the workers are the parallelism
    except Exception:
        pass


def _ref_eval(c):
    pts = np.vstack([_REF["design"], c[None, :]])
    if _REF["kind"] == "reference":
        return float(_REF["cf"].evaluate(pts))
    return float(_REF["orc"].ref_ivar_cost(_REF["kern"], pts, _REF["mc"], CFG["noise"]))


def reference_design(n):
    """A deterministic n-point design for the CPU arm: the first n greedy max-variance picks of a 2 000-candidate
    subsample (cheap on the CPU, well conditioned like a greedy design)."""
    from oracle import gpexp_oracle as orc
    cand, mc = make_inputs()
    idx, _ = orc.fast_greedy_var(orc.KernelSpec.se(CFG["cl"], CFG["signal"], CFG["d"]), cand[:2000], n)
    return cand, mc, cand[idx]


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import multiprocessing as mp
    cand, mc, design = reference_design(CFG["N"] - 1)
    path = os.path.join(ROOT, "baseline", "_ref")
    path = path if os.path.isdir(os.path.join(path, "gpExp")) else ""
    cores = max(1, min(os.cpu_count() or 1, args.ref_procs))
    # a fresh spawn pool: no CUDA state is inherited, every worker imports the reference itself
    with mp.get_context("spawn").Pool(cores, initializer=_ref_worker_init, initargs=(path, design, mc)) as pool:
        kind = pool.apply(_ref_kind)
        step = 0

        def one_step():
            nonlocal step
            chunk = cand[5000 + step * cores: 5000 + (step + 1) * cores]
            step += 1
            t0 = time.perf_counter()
            pool.map(_ref_eval, list(chunk), chunksize=1)
            return time.perf_counter() - t0
        for _ in range(args.warmup):
            one_step()
        t = sum(one_step() for _ in range(args.steps))
    value = args.steps * cores / t
    sample = (f"{cores} candidates per step (one per worker process) at n=255, M=100000 through "
              f"{'the unmodified reference costFunctionGP_IVAR.evaluate (baseline/_ref)' if kind == 'reference' else 'the oracle port of costFunctionGP_IVAR.evaluate'}"
              " = pinv + per-point python loop; scores are independent per candidate, so the rate extrapolates linearly in C")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "timing": "host wall clock, CPU only",
    }
    print(json.dumps(line))


def _ref_kind():
    return _REF["kind"]


def run_reference_configs():
    """CPU legs of BASELINE configs[0], [2] and [3] (SURVEY.md 8d, plan items i, iii and iv): the UNMODIFIED reference on
    bounded samples -- costFunctionGP_IVAR.evaluate on 40 cfg-1 candidates, performGreedyVarExperimentalDesign on 20 000 of the cfg-3 candidates for 16 points, and
    costFunctionGP_MI.evaluate at |V| = 400 of the cfg-4 pool.  One JSON line; baselines, not targets."""
    import contextlib
    import io
    import warnings
    warnings.filterwarnings("ignore")
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        print(json.dumps({"unavailable": "baseline/_ref is not staged"}))
        return
    sys.path.insert(0, path)
    import gpExp.experimentalDesign as red
    import gpExp.gp as rgp
    import gpExp.kernels as rk
    from gpExp.approximation import Space
    out = {"cores": os.cpu_count(), "kind": "reference"}
    rng = np.random.default_rng(1)
    cand1, mc1 = rng.uniform(-1, 1, (1000, 1)), rng.uniform(-1, 1, (10000, 1))
    cf1 = red.costFunctionGP_IVAR(rgp.GP(rk.KernelSquaredExponential([0.05], 1.0, 1), 1e-6), 2, Space(1, None, None, noise=None),
                                  mcPoints=mc1)
    t0 = time.perf_counter()
    for c in range(1, 41):
        cf1.evaluate(np.vstack([cand1[:1], cand1[c:c + 1]]))
    t = time.perf_counter() - t0
    out["cfg1"] = {"candidates_per_s_per_step": 40 / t, "seconds": t,
                   "sample": "costFunctionGP_IVAR.evaluate, 1-D SE cl=0.05, 40 of the 1 000 candidates of the second greedy step "
                             "(10 000 integration points; the full 20-point design is 20 000 such evaluations)"}
    rng = np.random.default_rng(3)
    pool = rng.uniform(-1, 1, (20_000, 5))
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        red.performGreedyVarExperimentalDesign(rk.KernelIsoMatern(1.0, 1.0, 5), pool, 16, 5)
    t = time.perf_counter() - t0
    out["cfg3"] = {"candidates_per_s_per_step": 20_000 * 16 / t, "seconds": t,
                   "sample": "performGreedyVarExperimentalDesign, 5-D Matern rho=1, 16 points from 20 000 candidates "
                             "(cost per step grows with the design size; cfg-3 runs to 1 024 points from 250 000)"}
    rng = np.random.default_rng(4)
    V = 400
    pts = rng.standard_normal((V, 3))
    gp = rgp.GP(rk.KernelMehlerND([0.9, 0.9, 0.9], 3), 1e-2)
    cf = red.costFunctionGP_MI(gp, 8, Space(3, None, None, noise=None), nmc=V, mcpoints=pts)
    t0 = time.perf_counter()
    for i in range(1, 31):
        cf.evaluate(i, [0])
    t = time.perf_counter() - t0
    out["cfg4"] = {"candidates_per_s_per_step": 30 / t, "seconds": t, "V": V,
                   "sample": "costFunctionGP_MI.evaluate, 3-D Mehler t=0.9, |V| = 400, 30 candidates of one greedy step "
                             "(two pinv of O(|V|^3) per candidate; cfg-4 has |V| = 200 000)"}
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 6]
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[0]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any("Active" in r[3 + i] and "Not" not in r[3 + i] for r in rows)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows),
                "samples": len(rows), "reasons": reasons}


# ---------------------------------------------------------------------------------------------
# checker-only block (N > 1): sharded engines against the CPU oracle on small seeded pools
# ---------------------------------------------------------------------------------------------
def parity_block(ed, gpmod, kernels, Space, ShardedMIEngine, Device, shard, dist, torch, rank, world):
    """Every rank runs the sharded drivers; rank 0 compares with the oracle (checker only: nothing here is timed)."""
    rng = np.random.default_rng(42)
    out = {}
    dev = Device.get()
    # greedy IVAR, candidates sharded; 4001 candidates do not divide evenly
    cand, mc = rng.uniform(-1, 1, (4001, 2)), rng.uniform(-1, 1, (3000, 2))
    kern = kernels.KernelSquaredExponential([0.2, 0.3], 1.0, 2)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, 1e-6), 1, Space(2, None, None), mcPoints=mc)
    picks = {}
    for resident in (False, True):
        picks[resident] = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True,
                                                                                   shard=shard, resident=resident)]
    ivar_scores = cf.lastScores.copy()
    # greedy max variance, pool sharded
    pool = rng.uniform(-1, 1, (10007, 5))
    mk = kernels.KernelIsoMatern(1.0, 1.0, 5)
    vpts = ed.performGreedyVarExperimentalDesign(mk, pool, 25, 5, shard=shard)
    vidx = [int(np.where(np.all(pool == p, axis=1))[0][0]) for p in vpts]
    # greedy mutual information, |V| x |V| factor sharded by column blocks; the 100-point pool is ONE elimination block,
    # so every rank but the first holds no columns (the case a 4-rank run tripped over in round 1)
    hk = kernels.KernelMehlerND([0.9, 0.9, 0.9], 3)
    hk._bind(dev)
    mi = {}
    for tag, V, n in (("mi_1500", 1500, 14), ("mi_100_empty_ranks", 100, 6)):
        vpool = np.random.default_rng(43).standard_normal((V, 3))
        eng = ShardedMIEngine(dev, vpool, n, 1e-2, shard=shard)
        mi[tag] = ([int(i) for i in eng.run(n, start=0)], int(eng.info.item()), vpool, n,
                   int(sum(1 for c in eng.ncols_per_rank if c == 0)))
    torch.cuda.synchronize()
    flat = picks[False] + picks[True] + vidx + mi["mi_1500"][0] + mi["mi_100_empty_ranks"][0]
    t = torch.tensor(flat, device="cuda")
    g = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(g, t)
    out["all_ranks_agree"] = all(bool((x == t).all()) for x in g)
    if rank == 0:
        from oracle import gpexp_oracle as orc
        ref, costs = orc.fast_greedy_ivar(orc.KernelSpec.se([0.2, 0.3], 1.0, 2), cand, mc, 12, 1e-6)
        want = np.array([c[i] for c, i in zip(costs, ref)])
        out["greedy_ivar_contraction"] = picks[False] == ref
        out["greedy_ivar_resident"] = picks[True] == ref
        out["greedy_ivar_max_rel_err_scores"] = float(np.max(np.abs(ivar_scores - want) / np.abs(want)))
        vref, _ = orc.fast_greedy_var(orc.KernelSpec.matern32(1.0, 1.0, 5), pool, 25)
        out["greedy_var"] = vidx == vref
        for tag, (got, info, vpool, n, empty) in mi.items():
            mref, _ = orc.fast_greedy_mi(orc.KernelSpec.mehler([0.9, 0.9, 0.9], 3), vpool, 1e-2, n, start=0)
            out[tag] = (got == mref) and info == 0
            out[tag + "_ranks_without_columns"] = empty
        out["ok"] = bool(out["all_ranks_agree"] and out["greedy_ivar_contraction"] and out["greedy_ivar_resident"] and
                         out["greedy_var"] and out["mi_1500"] and out["mi_100_empty_ranks"] and
                         out["greedy_ivar_max_rel_err_scores"] <= 1e-9)
        out["note"] = "checker: oracle.fast_* on rank 0; picks must be identical, all ranks must hold the same picks"
    return out


def cfg5_block(ed, gpmod, kernels, Space, shard, dist, torch, rank, world, local, dgemm_tflops):
    """BASELINE configs[4], the north-star target: ONE greedy IVAR step at n = 4096 over 1 000 000 candidates x 100 000
    integration points, 10-D ARD SE, candidates sharded over the ranks -- through the public design object."""
    from gpexp_b200.engine import DesignFactor
    d, n, C, M, noise = 10, 4096, 1_000_000, 100_000, 1e-6
    rng = np.random.default_rng(5)
    cl = list(np.linspace(0.5, 1.5, d))
    cand_h = rng.uniform(-1, 1, (C, d))
    mc_h = rng.uniform(-1, 1, (M, d))
    design_h = cand_h[np.sort(rng.permutation(C)[:n])]
    kern = kernels.KernelSquaredExponential(cl, 1.0, d)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, noise), 1, Space(d, None, None), mcPoints=mc_h)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand_h, n + 1, shard=shard, resident=False)
    dev = eng.dev

    def sync():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
    sync()
    t0 = time.perf_counter()
    eng.load_design(DesignFactor(dev, dev.points(design_h), noise))
    sync()
    setup_s = time.perf_counter() - t0
    snap = eng.snapshot()
    eng.run(n + 1)          # warm-up step
    eng.restore(snap)
    sync()
    clocks = Clocks(local) if rank == 0 else None
    steps = 2
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        eng.run(n + 1)      # the whole step through gpx_ivar_greedy_run: score, arg-min, NCCL exchange, append
        if s + 1 < steps:
            eng.restore(snap)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1) / steps
    eng.restore(snap)
    ks = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):  # the contraction alone, for the roofline figure
        ks[s][0].record()
        eng.score()
        ks[s][1].record()
    sync()
    score_ms = float(np.mean([a.elapsed_time(b) for a, b in ks]))
    eng.run(n + 1)
    t = torch.tensor([ms, score_ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, score_ms = float(t[0]), float(t[1])
    clk = clocks.stop() if clocks else None
    winner = int(eng.picks[n].item())
    wscore = float(eng.pick_scores[n].item())
    lo, hi = eng.index_offset, eng.index_offset + eng.cand.n
    out = None
    if rank == 0:
        flops_gpu = 2.0 * M * n * (hi - lo)
        tf = flops_gpu / score_ms / 1e9
        out = {"workload": "cfg-5: 10-D ARD SE, one greedy IVAR step at n=4096, 1 000 000 candidates x 100 000 MC points, "
                           f"candidates/{world}", "n_gpus": world, "s_per_step": ms / 1e3, "score_s": score_ms / 1e3,
               "candidates_per_s": C / ms * 1e3, "tflops_per_gpu": tf, "frac_of_in_run_dgemm": tf / dgemm_tflops,
               "frac_of_dmma_pipe_peak_37.2": tf / 37.2, "in_run_dgemm_tflops": dgemm_tflops,
               "target": ">= 0.60 of the FP64 tensor roofline (BASELINE.json north_star)", "meets_target": bool(tf / 37.2 >= 0.6),
               "design": "4096 seeded-random candidates loaded through Gram + Cholesky + fused Gram/TRSM",
               "setup_from_scratch_s": setup_s, "winner_global_index": winner, "winner_cost": wscore,
               "total_flop_per_step": 2.0 * M * n * C, "clocks": clk}
        # checker: the winner's cost and 255 random candidates against the oracle (rank 0's block + the winner)
        from oracle import gpexp_oracle as orc
        okern = orc.KernelSpec.se(cl, 1.0, d)
        sub = np.unique(np.concatenate([[winner], rng.permutation(C)[:255]]))
        w_m, var_m = orc.fast_design_state(okern, design_h, mc_h, noise)
        w_c, var_c = orc.fast_design_state(okern, design_h, cand_h[sub], noise)
        ref = orc.fast_ivar_scores(okern, cand_h[sub], mc_h, w_m, var_m, w_c, var_c, noise)
        wi = int(np.where(sub == winner)[0][0])
        out["oracle_winner_cost_rel_err"] = float(abs(ref[wi] - wscore) / abs(ref[wi]))
        out["oracle_winner_is_min_of_sample"] = bool(ref[wi] == ref.min())
        mine = (sub >= lo) & (sub < hi)
        got = eng.scores[: eng.cand.n].cpu().numpy()[sub[mine] - lo]
        out["oracle_max_rel_err_local_sample"] = float(np.max(np.abs(got - ref[mine]) / np.abs(ref[mine])))
    del eng
    torch.cuda.empty_cache()
    return out


def cfg3_block(ed, kernels, shard, dist, torch, rank, world):
    """BASELINE configs[2]: 5-D Matern, conditional-entropy greedy design of 1 024 points from 250 000 candidates (the pool
    sharded over the ranks), through performGreedyVarExperimentalDesign -> gpx_var_greedy_run."""
    rng = np.random.default_rng(3)
    C, N = 250_000, 1024
    pool = rng.uniform(-1, 1, (C, 5))
    kern = kernels.KernelIsoMatern(1.0, 1.0, 5)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    ed.performGreedyVarExperimentalDesign(kern, pool[:5000], 16, 5, shard=shard)     # warm-up (allocator, communicator)
    sync()
    t0 = time.perf_counter()
    pts = ed.performGreedyVarExperimentalDesign(kern, pool, N, 5, shard=shard)
    sync()
    t = time.perf_counter() - t0
    if rank != 0:
        return None
    bytes_alg = sum(8.0 * (n + 2) * C for n in range(N))
    out = {"workload": f"cfg-3: 5-D Matern rho=1, greedy max posterior variance, 1 024 of 250 000 candidates, candidates/{world}",
           "design_s": t, "candidates_per_s_per_step": N * C / t, "append_gbs_aggregate": bytes_alg / t / 1e9,
           "call": "performGreedyVarExperimentalDesign(kernel, pool, 1024, 5, shard) from host arrays (upload included)"}
    # checker: first 150 picks against the oracle, all picks distinct
    from oracle import gpexp_oracle as orc
    ref, _ = orc.fast_greedy_var(orc.KernelSpec.matern32(1.0, 1.0, 5), pool, 150)
    out["first_150_picks_match_oracle"] = bool(np.array_equal(pts[:150], pool[ref]))
    out["distinct_points"] = bool(len(np.unique(pts, axis=0)) == N)
    return out


def cfg4_block(ed, gpmod, kernels, Space, shard, dist, torch, rank, world):
    """BASELINE configs[3]: 3-D Mehler, greedy mutual-information design of 512 points; the |V| x |V| factor and its
    inverse-transpose are sharded block-cyclically, so the pool size follows the memory of the job:
    |V| = 40 000 / 80 000 / 120 000 / 200 000 (the full cfg-4 size) on 1 / 2 / 4 / 8 GPUs."""
    V = {1: 40_000, 2: 80_000, 4: 120_000}.get(world, 200_000 if world >= 8 else 40_000 * world)
    N, noise = 512, 1e-2
    pool = np.random.default_rng(4).standard_normal((V, 3))
    kern = kernels.KernelMehlerND([0.9, 0.9, 0.9], 3)
    from gpexp_b200.engine import ShardedMIEngine
    from gpexp_b200.device import Device
    dev = Device.get()
    kern._bind(dev)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    sync()
    t0 = time.perf_counter()
    eng = ShardedMIEngine(dev, pool, N, noise, shard=shard)
    sync()
    setup_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    idx = eng.run(N, start=0)
    sync()
    design_s = time.perf_counter() - t0
    info = int(eng.info.item())
    out = None
    if rank == 0:
        out = {"workload": f"cfg-4: 3-D Mehler t=0.9, greedy MI design of 512 points from |V|={V}, noise 1e-2, "
                           f"block-cyclic column blocks over {world} GPU(s)" + ("" if V == 200_000 else " (full cfg-4 size is 200 000 on 8 GPUs)"),
               "V": V, "setup_s": setup_s, "setup_tflops_per_gpu": (2.0 * V ** 3 / 3.0 / world) / setup_s / 1e12,
               "design_s": design_s, "ms_per_step": 1e3 * design_s / (N - 1), "candidates_per_s_per_step": (N - 1) * V / design_s,
               "potrf_info": info, "distinct_picks": len(set(int(i) for i in idx)) == N, "first_picks": [int(i) for i in idx[:8]],
               "hbm_per_gpu_gb": 2 * 8.0 * V * max(eng.ncols_per_rank) / 1e9, "blk": eng.BLK}
    del eng
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod, kernels
    from gpexp_b200._lib import check, lib
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device, ptr
    from gpexp_b200.engine import DesignFactor, Shard, ShardedMIEngine

    ed.VERBOSE = False
    shard = Shard() if world > 1 else None
    dev = Device.get(local)
    cand_all, mc_h = make_inputs()
    lo, hi = Shard.split(cand_all.shape[0], world, rank)
    kern = kernels.KernelSquaredExponential(CFG["cl"], CFG["signal"], CFG["d"])
    N = CFG["N"]
    n = N - 1
    cf = ed.costFunctionGP_IVAR(gpmod.GP(kern, CFG["noise"]), 1, Space(CFG["d"], None, None), mcPoints=mc_h)
    # the public design object: contraction mode (the DMMA path the headline metric is about)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand_all, N, shard=shard, resident=False)
    cand, mc = eng.cand, eng.mc

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- the whole design once: n = 0 .. 254 (also the warm state for the timed step) -------------
    sync_all()
    t0 = time.perf_counter()
    if args.quick_design:
        # profiling aid: same state shape, design = 255 seeded-random candidates loaded through Gram+Cholesky+TRSM
        assert world == 1, "--quick-design is a single-GPU profiling aid"
        pick = np.random.default_rng(0).permutation(cand_all.shape[0])[:n]
        eng.load_design(DesignFactor(dev, dev.points(cand_all[pick]), CFG["noise"]))
    else:
        eng.run(n)
    sync_all()
    design_255_s = time.perf_counter() - t0
    snap = eng.snapshot()

    def step():
        eng.run(N)            # ONE greedy step through the C-side loop: score, arg-min, exchange, append
        eng.restore(snap)

    for _ in range(args.warmup):
        step()
    sync_all()
    clocks = Clocks(local) if rank == 0 else None
    launches0 = dev.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for s in range(args.steps):
        step()
    ev[1].record()
    sync_all()
    launches = dev.launches - launches0
    ms = ev[0].elapsed_time(ev[1])
    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        dump_step_outputs(args.dump_outputs, eng, N, cand_all.shape[0], torch, dist, world, rank)
    # the dominant kernel alone, on the same state (its CUDA-event time is what the roofline is computed from)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s in range(args.steps):
        kev[s][0].record()
        eng.score()
        kev[s][1].record()
    sync_all()
    score_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    if world > 1:
        t = torch.tensor([ms, score_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, score_ms = float(t[0]), float(t[1])
    ms_per_step = ms / args.steps
    total_c = cand_all.shape[0]
    value = total_c / (ms_per_step * 1e-3)

    # finish the design (step 256) so that design_total_s covers all N steps
    sync_all()
    t0 = time.perf_counter()
    eng.run(N)
    sync_all()
    design_total_s = design_255_s + (time.perf_counter() - t0)
    picks = eng.indices()
    if args.quick_design:
        picks = np.concatenate([pick, picks[-1:]])
    prologue_mode = int(eng.prologue()[0])

    # ---- end to end through the public API with HOST (pinned) buffers: every rank scores its own shard -------------
    design_h = cand_all[picks[:n]]
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    cand_p, mc_p, des_p = pin(cand_all), pin(mc_h), pin(design_h)
    cf_e2e = ed.costFunctionGP_IVAR(gpmod.GP(kern, CFG["noise"]), 1, Space(CFG["d"], None, None), mcPoints=mc_p)
    e2e_steps = max(2, min(args.steps, 5))
    costs, gbest = ed.scoreCandidatesIVAR(cf_e2e, des_p, cand_p, shard=shard)  # warm-up
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        costs, gbest = ed.scoreCandidatesIVAR(cf_e2e, des_p, cand_p, shard=shard)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())

    # ---- in-run FP64 yard-stick: cuBLAS DGEMM 8192^3 (MEASURED_PEAKS.json has no FP64 entry) -----------------------
    A = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    torch.matmul(A, A)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        torch.matmul(A, A)
    e1.record()
    torch.cuda.synchronize()
    dgemm_tflops = 3 * 2 * 8192.0 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12
    del A

    # ---- N > 1: parity of the sharded engines (checker only), and at N = 8 the north-star step -----------------------
    parity = cfg5 = None
    del eng
    torch.cuda.empty_cache()

    def guarded(fn, *a):
        """The side blocks must not cost the headline line: a failure is reported in place of the block's result."""
        try:
            return fn(*a)
        except Exception as e:  # noqa: BLE001
            torch.cuda.empty_cache()
            return {"error": f"{type(e).__name__}: {e}"[:400]} if rank == 0 else None
    if world > 1 and not args.no_parity:
        parity = guarded(parity_block, ed, gpmod, kernels, Space, ShardedMIEngine, Device, shard, dist, torch, rank, world)
    if world >= 8 and not args.no_cfg5:
        cfg5 = guarded(cfg5_block, ed, gpmod, kernels, Space, shard, dist, torch, rank, world, local, dgemm_tflops)
    cfg3 = cfg4 = None
    if not args.no_configs:
        cfg3 = guarded(cfg3_block, ed, kernels, shard, dist, torch, rank, world)
        cfg4 = guarded(cfg4_block, ed, gpmod, kernels, Space, shard, dist, torch, rank, world)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (DMMA contraction, K5) ------------------------------------
    flops = 2.0 * CFG["M"] * n * cand.n                     # algorithmic: 2*M*n flop per candidate per step
    achieved = flops / (score_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "ivar_core_traffic.json")
    if world == 1 and os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    ring = {0: "32-row chunks x 3 stages, per-row cp.async.bulk", 1: "32-row chunks x 3 stages, 2-D tensor-map TMA (UTMALDG)",
            2: "24-row chunks x 4 stages, 2-D tensor-map TMA"}.get(int(os.environ.get("GPX_IVAR_RING", "1")), "?")
    roofline = {"bound": "tensor",
                "kernel": f"ivar_ws_kernel<SE, {'EXPANDED' if prologue_mode == 1 else 'DIFF'} prologue> (FP64 DMMA.8x8x4 "
                          f"contraction + covariance prologue on the tensor pipe; {ring})",
                "achieved": achieved, "peak": dgemm_tflops, "unit": "TFLOP/s", "frac": achieved / dgemm_tflops,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry); "
                               "theoretical DMMA peak 148 SM x 128 flop/clk x 1.965 GHz = 37.2 TFLOP/s",
                "frac_of_dmma_pipe_peak": achieved / 37.2, "flops_per_launch": flops, "launch_ms": score_ms,
                "launch_timing": "CUDA events around gpx_score_ivar on the launching stream, mean of the timed steps, max over ranks"}

    e2e = {"value": total_c / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": int(total_c * CFG["d"] * 8 + world * (CFG["M"] + n) * CFG["d"] * 8),
           "d2h_bytes_per_step": int(total_c * 8 + world * 8), "ms_per_step": e2e_s * 1e3,
           "call": "gpexp_b200.experimentalDesign.scoreCandidatesIVAR(costFunc, design[255,2], candidates[100000,2], shard) "
                   "from pinned host arrays: H2D + Gram + Cholesky + fused Gram/TRSM for W_C, W_M + DMMA scoring + D2H of all "
                   "costs + global arg-min; max over ranks",
           "argmin_matches_greedy_step": bool(gbest == int(picks[n]))}

    # ---- CPU baseline: the reference arm in a fresh process (no CUDA state), bounded sample --------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                               capture_output=True, text=True, timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
            ref_line = json.loads(r.stdout.strip().splitlines()[-1])
            cpu = ref_line["cpu_baseline"]
        except Exception as e:  # the baseline is a reported number, not a gate
            cpu = {"value": None, "unit": UNIT, "cores": None, "kind": "unavailable", "sample": f"reference arm failed: {e}"}
        # the same-algorithm CPU line (vectorised Cholesky/Schur oracle) and the parity of this run's costs against it
        from oracle import gpexp_oracle as orc
        okern = orc.KernelSpec.se(CFG["cl"], CFG["signal"], CFG["d"])
        t1 = time.perf_counter()
        w_m, var_m = orc.fast_design_state(okern, design_h, mc_h, CFG["noise"])
        w_c, var_c = orc.fast_design_state(okern, design_h, cand_all[:2000], CFG["noise"])
        ref_scores = orc.fast_ivar_scores(okern, cand_all[:2000], mc_h, w_m, var_m, w_c, var_c, CFG["noise"])
        tfast = time.perf_counter() - t1
        cpu["vectorised_port_value"] = 2000 / tfast
        cpu["vectorised_port_sample"] = f"2000 candidates, numpy Cholesky/Schur restatement, {tfast:.1f} s"
        cpu["gpu_vs_oracle_max_rel_err_2000_candidates"] = float(np.max(np.abs(costs[:2000] - ref_scores) / np.abs(ref_scores)))

    # ---- the other figures of the BASELINE metric and the small configurations ---------------------------------------
    extras = {}
    if world == 1:
        hbm, hbm_src = 6650.0, "B200_PROFILING.md fallback"
        try:
            hbm, hbm_src = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json"
        except Exception:
            pass

        def ev_ms(fn, reps=3):
            fn()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(reps):
                fn()
            a1.record()
            torch.cuda.synchronize()
            return a0.elapsed_time(a1) / reps
        kern._bind(dev)
        nx = 4096
        G = dev.empty(nx, cand.ld)
        t_gram = ev_ms(lambda: check(lib.gpx_gram(dev.h, ptr(cand.X), nx, cand.ld, ptr(cand.X), cand.n, cand.ld, ptr(G),
                                                  cand.ld, 0, None, 0.0, dev.stream)))
        gram_gbs = 8.0 * nx * cand.n / (t_gram * 1e-3) / 1e9
        del G
        # HBM-bound row append (K3+K4) at n = 255 on a fresh factor of the same shape (reads 8*n*C bytes)
        Wt, vt, rec = dev.zeros(N, cand.ld), dev.zeros(cand.ld), dev.zeros(19 + N)
        rec[2] = 1.0
        t_app = ev_ms(lambda: check(lib.gpx_append_row(dev.h, 0, ptr(rec), None, ptr(cand.X), cand.n, cand.ld, ptr(Wt),
                                                       cand.ld, n, ptr(vt), dev.stream)), reps=10)
        app_gbs = 8.0 * (n + 2) * cand.n / (t_app * 1e-3) / 1e9
        del Wt, vt
        # 8(f): the analytic IVAR gradient the SLSQP polish calls (experimentalDesign.py:148-179)
        cf_e2e.numInputs = n
        cf_e2e.derivative(des_p)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        grad = cf_e2e.derivative(des_p)
        torch.cuda.synchronize()
        grad_ms = (time.perf_counter() - t0) * 1e3
        # a7: posterior variance of 100k points given the 255-point design, from host arrays (GP.evaluateVariance)
        g_pv = gpmod.GP(kern, CFG["noise"])
        g_pv.addNodesAndComputeCovariance(des_p)
        g_pv.evaluateVariance(mc_p)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pv = g_pv.evaluateVariance(mc_p)
        torch.cuda.synchronize()
        pv_ms = (time.perf_counter() - t0) * 1e3
        # f4: matrix-free Gram x vector over the 100k integration points (covTimesV)
        from gpexp_b200 import gp_kernel_utilities as gku
        op = gku._GramOperator(kern, mc_p)
        v = np.random.default_rng(0).standard_normal(CFG["M"])
        op(v)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        op(v)
        torch.cuda.synchronize()
        mv_ms = (time.perf_counter() - t0) * 1e3
        # cfg-1 (configs[0], the reference's own CPU-runnable case): the whole 20-point design, C-side loop
        rng1 = np.random.default_rng(1)
        c1, m1 = rng1.uniform(-1, 1, (1000, 1)), rng1.uniform(-1, 1, (10000, 1))
        k1 = kernels.KernelSquaredExponential([0.05], 1.0, 1)
        cf1 = ed.costFunctionGP_IVAR(gpmod.GP(k1, 1e-6), 1, Space(1, None, None), mcPoints=m1)
        cfg1 = {}
        for resident in (False, True):
            e1_ = ed.beginGreedyIVARExperimentalDesign(cf1, c1, 20, resident=resident)
            e1_.run(20)
            torch.cuda.synchronize()
            e1_ = ed.beginGreedyIVARExperimentalDesign(cf1, c1, 20, resident=resident)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e1_.run(20)
            torch.cuda.synchronize()
            cfg1["resident_ms" if resident else "contraction_ms"] = (time.perf_counter() - t0) * 1e3
            cfg1["picks"] = [int(i) for i in e1_.indices()[:6]]
        cfg1["note"] = ("whole 20-point design of configs[0] (1 000 candidates x 10 000 MC points), wall clock of one run() call: "
                        "contraction = 20 x 5 launches from the C-side loop, resident = " +
                        ("ONE cooperative kernel (gpx_ivar_greedy_small)" if type(e1_).ONE_KERNEL_PAIRS >= 10_000_000
                         else "20 x 4 launches from the C-side loop"))
        # resident-covariance mode of the same greedy loop (HBM-bound, 16*M*C bytes per step)
        kern._bind(dev)
        torch.cuda.empty_cache()
        res = None
        free, _ = torch.cuda.mem_get_info()
        if 8.0 * mc.n * cand.ld < 0.8 * free and not args.quick_design:
            reng = ed.beginGreedyIVARExperimentalDesign(cf, cand_all, N, resident=True)
            reng.run(4)
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            reng.run(24)
            r1.record()
            torch.cuda.synchronize()
            rms = r0.elapsed_time(r1) / 20.0
            torch.cuda.synchronize()
            tr0 = time.perf_counter()
            reng.run(N)
            torch.cuda.synchronize()
            rest_s = time.perf_counter() - tr0
            rfull = reng.indices()
            res = {"ms_per_step": rms, "design_total_s_extrapolated_from_steps_24_to_256": rest_s * N / (N - 24.0),
                   "all_256_picks_equal_dmma_path": [int(i) for i in rfull] == [int(i) for i in picks[:N]],
                   "candidates_per_s": cand.n / rms * 1e3, "hbm_gbs": 16.0 * mc.n * cand.n / (rms * 1e-3) / 1e9,
                   "frac_of_measured_hbm": 16.0 * mc.n * cand.n / (rms * 1e-3) / 1e9 / hbm, "resident_gb": 8.0 * mc.n * cand.ld / 1e9,
                   "note": "same greedy loop with the M x C posterior covariance resident in HBM and one rank-1 update pass "
                           "per step; cost independent of n; the DMMA contraction stays the path for scoring a given design"}
            del reng
            torch.cuda.empty_cache()
        extras = {"resident_covariance_mode": res, "cfg1_whole_design": cfg1, "posterior_variance_ms": pv_ms,
                  "posterior_variance_points_per_s": mc_p.shape[0] / pv_ms * 1e3, "posterior_variance_min": float(pv.min()),
                  "ivar_gradient_ms": grad_ms, "ivar_gradient_shape": [int(grad.size)],
                  "gram_matvec_100k_ms": mv_ms, "gram_matvec_pairs_per_s": CFG["M"] ** 2 / mv_ms * 1e3,
                  "gram_gbs": gram_gbs, "gram_frac_of_measured_hbm": gram_gbs / hbm, "gram_block": [nx, cand.n],
                  "append_row_gbs": app_gbs, "append_row_frac_of_measured_hbm": app_gbs / hbm, "hbm_peak_gbs": hbm,
                  "hbm_peak_source": hbm_src}
    if world == 1 and not args.no_cpu and not args.no_configs:
        try:  # CPU legs of cfg-3 / cfg-4 (the unmodified reference, bounded samples) in a fresh process
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-configs"], capture_output=True,
                               text=True, timeout=300, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
            extras["cpu_reference_other_configs"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            extras["cpu_reference_other_configs"] = {"unavailable": str(e)}
    if cfg5 is not None:
        extras["cfg5"] = cfg5
    if cfg3 is not None:
        extras["cfg3"] = cfg3
    if cfg4 is not None:
        extras["cfg4"] = cfg4

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_dict(world),
        "clocks": clk, "e2e": e2e, "gpu_launches": int(launches),
        "gpu_launches_note": "kernel launches counted inside libgpexp_b200.so (gpx_launch_count) over the timed region, this rank",
        "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
        "step_call": "beginGreedyIVARExperimentalDesign(costFunc, candidates, 256, shard, resident=False).run(256) from n=255 "
                     "(gpx_ivar_greedy_run: one C call per step), then restore of the two running-variance vectors",
        "design_total_s": design_total_s, "design_points": N,
        "design_candidates_per_s": N * total_c / design_total_s,
        "design_first_picks": [int(i) for i in picks[:8]],
        "extras": extras,
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # Only the JSON line may reach stdout: NCCL prints its version banner there during the first collective.
    # Everything else written to fd 1 while the benchmark runs is sent to stderr; the JSON line goes to the real stdout.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-configs"])
    ap.add_argument("--ref-procs", type=int, default=32, help="worker processes of the reference arm (capped at the core count)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the N>1 parity block")
    ap.add_argument("--no-cfg5", action="store_true", help="skip extras.cfg5 at N=8")
    ap.add_argument("--no-configs", action="store_true", help="skip extras.cfg3 / extras.cfg4 (the other BASELINE configurations)")
    ap.add_argument("--quick-design", action="store_true",
                    help="profiling aid: load a random 255-point design instead of running the 255 greedy steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64) for output-for-output comparison")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-configs":
        run_reference_configs()
    else:
        run_ours(args)
    real_stdout.flush()


if __name__ == "__main__":
    main()
