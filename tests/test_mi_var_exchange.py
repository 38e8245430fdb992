"""Exchange refinement of discrete MI and maximum-variance designs (refineGreedyMIExperimentalDesign,
refineGreedyVarExperimentalDesign) and the engine deletions under them.

The oracles are tests/mi_var_exchange_oracle.py (brute-force passes that refactor from scratch at every step, the MI pass
again through the reference's pinv loop, and the two objectives) and tests/ivar_exchange_oracle.py (fast_design_delete).
CPU: the two MI oracles agree; a Givens downdate of U_Q / Us gives the precision-side state of A minus j built from
scratch; with zero noise every accepted MI swap raises I(y_A; y_{V minus A}) by 1/2 log(score ratio); the variance
objective never decreases.
GPU: remove(j) against an engine forced with the remaining points (MI over several block-cyclic blocks, and variance);
both refinements against the oracles over every kernel family, scalar and per-point noise, weights and fixed seeds; the
reported objectives; argument checks; greedy runs unchanged by factor storage; a 2-rank NCCL run when two GPUs are
visible."""
import functools
import os
import socket

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests import ivar_exchange_oracle as xo
from tests import mi_var_exchange_oracle as mx

RTOL = 1e-8


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b))) if a.size else 0.0


KERN_X = {"se_ard": ("se", [0.25, 0.35], 1.0), "matern12": (0.5, 0.5, 1.0), "matern32": (1.5, 0.4, 1.0),
          "matern52": (2.5, 0.4, 1.0), "mehler": ("mehler", [0.7, 0.6], None)}


def _spec(name):
    a, b, c = KERN_X[name]
    if a == "se":
        return orc.KernelSpec.se(b, c, 2)
    if a == "mehler":
        return orc.KernelSpec.mehler(b, 2)
    return {0.5: orc.KernelSpec.matern12, 1.5: orc.KernelSpec.matern32, 2.5: orc.KernelSpec.matern52}[a](b, c, 2)


def _kernel(name):
    from gpexp_b200 import kernels as K
    a, b, c = KERN_X[name]
    if a == "se":
        return K.KernelSquaredExponential(b, c, 2)
    if a == "mehler":
        return K.KernelMehlerND(b, 2)
    return K.KernelIsoMatern(b, c, 2, nu=a)


def _sample(rng, name, shape):
    return rng.standard_normal(shape) if name == "mehler" else rng.uniform(-1, 1, shape)


def _mi_noise(name, variant, pool):
    noise = 1e-2 if name == "mehler" else 1e-4
    if variant == "nu":
        noise = noise * (1.0 + 20.0 * np.minimum(pool[:, 0] ** 2, 4.0))
    return noise


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
MI_CPU = [(k, v) for k in ("se_ard", "matern12", "mehler") for v in ("scalar", "nu")]


@pytest.mark.parametrize("kname,variant", MI_CPU, ids=[f"{k}-{v}" for k, v in MI_CPU])
def test_fast_mi_exchange_equals_reference_loop(kname, variant):
    rng = np.random.default_rng(11)
    spec = _spec(kname)
    pool = _sample(rng, kname, (60, 2))
    noise = _mi_noise(kname, variant, pool)
    start = [int(i) for i in rng.choice(60, 6, replace=False)]
    d_ref, s_ref, w_ref, _, _ = mx.ref_exchange_mi(spec, pool, start, noise, RTOL, 10)
    d, s, w, margins, _ = mx.fast_exchange_mi(spec, pool, start, noise, RTOL, 10)
    assert min(margins) > 1e-6
    assert d == d_ref and w == w_ref
    assert _rel(s, s_ref) <= 1e-8
    assert w[-1] == 0 and sum(w) > 0


DELETE_CASES = [(n, j) for n in (1, 2, 9) for j in sorted({0, n // 2, n - 1})]


@pytest.mark.parametrize("n,j", DELETE_CASES, ids=[f"n{n}-j{j}" for n, j in DELETE_CASES])
def test_precision_downdate_equals_refactoring(n, j):
    rng = np.random.default_rng(300 + n)
    spec = _spec("se_ard")
    pool = rng.uniform(-1, 1, (80, 2))
    nu = 1e-3 * (1.0 + pool[:, 1] ** 2)
    a = [int(i) for i in rng.choice(80, n, replace=False)]
    uq, us, pd = mx.precision_state(spec, pool, a, nu)
    uq1, us1, r, pd1 = xo.fast_design_delete(uq, us, pd, j)
    rest = a[:j] + a[j + 1:]
    if rest:
        uq0, us0, pd0 = mx.precision_state(spec, pool, rest, nu)
        assert np.max(np.abs(uq1 - uq0)) <= 1e-11 * np.max(np.abs(uq0))
        assert np.max(np.abs(us1 - us0)) <= 1e-11 * np.max(np.abs(us0))
    else:
        pd0 = np.diag(np.linalg.inv(spec.gram(pool, pool) + np.diag(nu)))
    assert np.max(np.abs(pd1 - pd0)) <= 1e-11 * np.max(np.abs(pd0))
    # the downdated state scores like a fresh one
    s_state = np.full(80, -np.inf)
    s_free = np.setdiff1d(np.arange(80), rest)
    num = spec.prior(pool) - (np.sum(np.linalg.solve(np.linalg.cholesky(spec.gram(pool[rest], pool[rest]) + np.diag(nu[rest])),
                                                     spec.gram(pool[rest], pool)) ** 2, axis=0) if rest else 0.0)
    s_state[s_free] = num[s_free] / (1.0 / pd1[s_free] - nu[s_free])
    assert _rel(s_state[s_free], mx.mi_scores(spec, pool, rest, nu)[s_free]) <= 1e-9


def test_noise_free_mi_swaps_raise_the_mutual_information():
    rng = np.random.default_rng(5)
    spec = orc.KernelSpec.matern12(0.5, 1.0, 2)    # a well-conditioned Gram without a nugget
    pool = rng.uniform(-1, 1, (70, 2))
    start = [int(i) for i in rng.choice(70, 8, replace=False)]
    d, _, swaps, _, moves = mx.fast_exchange_mi(spec, pool, start, 0.0, RTOL, 10)
    assert sum(swaps) > 0
    design = list(start)
    prev = mx.mi_objective(spec, pool, design, 0.0)
    for inc, win, s_inc, s_win in moves:
        design = design[1:] + [win]
        cur = mx.mi_objective(spec, pool, design, 0.0)
        assert abs((cur - prev) - 0.5 * np.log(s_win / s_inc)) <= 1e-9 * max(1.0, abs(cur))
        if win != inc:
            assert cur > prev
        prev = cur
    assert design == d


@pytest.mark.parametrize("weighted", [False, True], ids=["plain", "weights"])
def test_variance_objective_never_decreases(weighted):
    rng = np.random.default_rng(8)
    spec = _spec("matern32")
    pool = rng.uniform(-1, 1, (300, 2))
    w = rng.uniform(0.5, 2.0, 300) if weighted else None
    start = [int(i) for i in rng.choice(300, 10, replace=False)]
    d, _, swaps, _, moves = mx.fast_exchange_var(spec, pool, start, RTOL, 10, weights=w, n_fixed=2)
    assert sum(swaps) > 0 and d[:2] == start[:2]
    design = list(start)
    prev = mx.var_objective(spec, pool, design, w)
    for inc, win, s_inc, s_win in moves:
        design = design[:2] + design[3:] + [win]
        cur = mx.var_objective(spec, pool, design, w)
        assert cur >= prev - 1e-10 * abs(prev)
        assert abs((cur - prev) - np.log(s_win / s_inc)) <= 1e-8 * max(1.0, abs(cur))
        prev = cur


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    ed.VERBOSE = False

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ed, ns.gp, ns.Space = torch, ed, gpmod, Space
    ns.dev = Device.get(0)
    return ns


def _mi_cost_function(env, kname, pool, noise):
    return env.ed.costFunctionGP_MI(env.gp.GP(_kernel(kname), noise), 1, env.Space(2, None, None), nmc=pool.shape[0],
                                    mcpoints=pool)


def _host(t, rows, cols):
    return t[:rows, :cols].cpu().numpy().copy()


def _close(got, want, tol, scale=None):
    scale = np.max(np.abs(want)) if scale is None else scale
    assert np.max(np.abs(got - want), initial=0.0) <= tol * scale, (np.max(np.abs(got - want)), scale)


@pytest.mark.gpu
@pytest.mark.parametrize("position", ["first", "middle", "last"])
def test_mi_remove_matches_forced_engine(env, monkeypatch, position):
    monkeypatch.setenv("GPX_MI_BLK", "256")       # |V| = 3 001 spans 12 cyclic blocks on the one rank
    rng = np.random.default_rng(21)
    pool = rng.uniform(-1, 1, (3001, 2))
    nu = 1e-3 * (1.0 + pool[:, 0] ** 2)
    cf = _mi_cost_function(env, "se_ard", pool, nu)
    n = 40
    j = {"first": 0, "middle": n // 2, "last": n - 1}[position]
    picks = [int(i) for i in rng.choice(3001, n, replace=False)]
    eng = env.ed._mi_new_engine(cf, n, keep_factors=True)
    assert eng.BLK == 256
    for p in picks:
        eng.force(p)
    eng.remove(j)
    assert eng.n == n - 1
    rest = picks[:j] + picks[j + 1:]
    ref = env.ed._mi_new_engine(cf, n, keep_factors=True)
    for p in rest:
        ref.force(p)
    m, L = n - 1, eng.nloc
    assert [int(i) for i in eng.indices()] == rest
    for a, b in ((eng.W, ref.W), (eng.Us, ref.Us)):
        want = _host(b, m, L)
        _close(_host(a, m, L), want, 1e-12, np.max(np.linalg.norm(want, axis=0)))
    for a, b in ((eng.UA, ref.UA), (eng.UQ, ref.UQ)):
        want = _host(b, m, m)
        _close(_host(a, m, m), want, 1e-12)
        assert np.all(_host(a, n, n)[m] == 0.0) and np.all(_host(a, n, n)[:, m] == 0.0)
    _close(eng.num[:L].cpu().numpy(), ref.num[:L].cpu().numpy(), 1e-12, 1.0)
    pd = ref.pd[:L].cpu().numpy()
    _close(eng.pd[:L].cpu().numpy(), pd, 1e-12)
    assert np.array_equal(eng.mask[:L].cpu().numpy(), ref.mask[:L].cpu().numpy())
    assert _rel(eng.pivots(), ref.pivots()) <= 1e-11
    # the reduced state has the forced design's objective and scores every pool point as it does
    mi_ref = ref.mutual_information()
    assert abs(eng.mutual_information() - mi_ref) <= 1e-10 * abs(mi_ref)
    eng.score()
    ref.score()
    free = ref.mask[:L].cpu().numpy() == 0
    assert _rel(eng.scores[:L].cpu().numpy()[free], ref.scores[:L].cpu().numpy()[free]) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("position", ["first", "middle", "last"])
def test_var_remove_matches_forced_engine(env, position):
    from gpexp_b200.engine import GreedyVarEngine
    rng = np.random.default_rng(22)
    pool_h = rng.uniform(-1, 1, (3001, 2))
    w = rng.uniform(0.5, 2.0, 3001)
    dev = _kernel("matern52")._bind()
    pool = dev.points(pool_h)
    n = 40
    j = {"first": 0, "middle": n // 2, "last": n - 1}[position]
    picks = [int(i) for i in rng.choice(3001, n, replace=False)]
    eng = GreedyVarEngine(dev, pool, n, weights=w, keep_factors=True)
    for p in picks:
        eng.force(p)
    eng.remove(j)
    rest = picks[:j] + picks[j + 1:]
    ref = GreedyVarEngine(dev, pool, n, weights=w, keep_factors=True)
    for p in rest:
        ref.force(p)
    m = n - 1
    assert [int(i) for i in eng.indices()] == rest
    want = _host(ref.W, m, 3001)
    _close(_host(eng.W, m, 3001), want, 1e-12, np.max(np.linalg.norm(want, axis=0)))
    _close(_host(eng.U, m, m), _host(ref.U, m, m), 1e-12)
    _close(eng.var[:3001].cpu().numpy(), ref.var[:3001].cpu().numpy(), 1e-12, 1.0)
    assert _rel(eng.pivots(), ref.pivots()) <= 1e-11


@functools.lru_cache(maxsize=None)
def _mi_problem(kname, variant):
    """|V| = 400, a random 12-point start; the brute-force oracle's run of the exchange."""
    rng = np.random.default_rng(0)
    pool = _sample(rng, kname, (400, 2))
    start = tuple(int(i) for i in rng.choice(400, 12, replace=False))
    noise = _mi_noise(kname, variant, pool)
    return pool, start, noise, mx.fast_exchange_mi(_spec(kname), pool, list(start), noise, RTOL, 10)


MI_X = [(k, v) for k in KERN_X for v in ("scalar", "nu")]


@pytest.mark.gpu
@pytest.mark.parametrize("kname,variant", MI_X, ids=[f"{k}-{v}" for k, v in MI_X])
def test_mi_refinement_matches_oracle(env, kname, variant):
    pool, start, noise, (d_ref, s_ref, w_ref, margins, _) = _mi_problem(kname, variant)
    # no decision of the oracle lies within 1e-6 of flipping, so rounding cannot change a decision
    assert min(margins) > 1e-6, min(margins)
    assert sum(w_ref) > 0
    cf = _mi_cost_function(env, kname, pool, noise)
    idx = env.ed.refineGreedyMIExperimentalDesign(cf, list(start), maxSweeps=10, rtol=RTOL, returnIndices=True)
    assert [int(i) for i in idx] == d_ref
    assert cf.lastSwaps == w_ref
    assert _rel(cf.lastScores, s_ref) <= 1e-8
    assert abs(cf.lastMI - mx.mi_objective(_spec(kname), pool, d_ref, noise)) <= 1e-9 * max(1.0, abs(cf.lastMI))


@functools.lru_cache(maxsize=None)
def _var_problem(kname, weighted):
    rng = np.random.default_rng(0)
    pool = _sample(rng, kname, (1500, 2))
    start = tuple(int(i) for i in rng.choice(1500, 16, replace=False))
    w = rng.uniform(0.5, 2.0, 1500) if weighted else None
    return pool, start, w, mx.fast_exchange_var(_spec(kname), pool, list(start), RTOL, 10, weights=w, n_fixed=3)


VAR_X = [(k, False) for k in KERN_X] + [("se_ard", True), ("matern12", True), ("mehler", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("kname,weighted", VAR_X, ids=[f"{k}-{'weights' if w else 'plain'}" for k, w in VAR_X])
def test_var_refinement_matches_oracle(env, kname, weighted):
    pool, start, w, (d_ref, s_ref, w_ref, margins, _) = _var_problem(kname, weighted)
    assert min(margins) > 1e-6, min(margins)
    assert sum(w_ref) > 0
    out, info = env.ed.refineGreedyVarExperimentalDesign(_kernel(kname), pool, list(start), weights=w, nFixed=3,
                                                          rtol=RTOL, returnIndices=True, returnInfo=True)
    assert [int(i) for i in out] == d_ref and [int(i) for i in info["indices"]] == d_ref
    assert list(out[:3]) == list(start[:3])          # the seeds never move
    assert info["swaps"] == w_ref
    assert _rel(info["scores"], s_ref) <= 1e-9
    ld = mx.var_objective(_spec(kname), pool, d_ref, w)
    assert abs(info["logdet"] - ld) <= 1e-9 * max(1.0, abs(ld))


@pytest.mark.gpu
def test_refinements_check_arguments(env):
    ed = env.ed
    pool, start, noise, (d_ref, _, _, _, _) = _mi_problem("se_ard", "scalar")
    cf = _mi_cost_function(env, "se_ard", pool, noise)
    same = ed.refineGreedyMIExperimentalDesign(cf, list(start), maxSweeps=0, returnIndices=True)
    assert [int(i) for i in same] == list(start) and cf.lastSwaps == [] and cf.lastScores.size == 0
    assert abs(cf.lastMI - mx.mi_objective(_spec("se_ard"), pool, list(start), noise)) <= 1e-9 * abs(cf.lastMI)
    pts = ed.refineGreedyMIExperimentalDesign(cf, d_ref)
    assert cf.lastSwaps == [0] and np.array_equal(pts, pool[d_ref])
    for bad in ([0, 400], [-1, 3], [0.0, 1.0], [], np.array([[1, 2]]), [4, 9, 4]):
        with pytest.raises(ValueError):
            ed.refineGreedyMIExperimentalDesign(cf, bad)
    for kw in ({"rtol": -1e-3}, {"maxSweeps": -1}, {"maxSweeps": 1.5}):
        with pytest.raises(ValueError):
            ed.refineGreedyMIExperimentalDesign(cf, [1, 2], **kw)
    vpool, vstart, _, _ = _var_problem("se_ard", False)
    k = _kernel("se_ard")
    same = ed.refineGreedyVarExperimentalDesign(k, vpool, list(vstart), maxSweeps=0, returnIndices=True)
    assert [int(i) for i in same] == list(vstart)
    out, info = ed.refineGreedyVarExperimentalDesign(k, vpool, list(vstart), nFixed=len(vstart), returnIndices=True,
                                                     returnInfo=True)
    assert [int(i) for i in out] == list(vstart) and info["swaps"] == [] and info["scores"].size == 0
    assert abs(info["logdet"] - mx.var_objective(_spec("se_ard"), vpool, list(vstart))) <= 1e-9 * abs(info["logdet"])
    for bad in ([0, 1500], [-1, 3], [0.5], []):
        with pytest.raises(ValueError):
            ed.refineGreedyVarExperimentalDesign(k, vpool, bad)
    for kw in ({"nFixed": 17}, {"nFixed": -1}, {"rtol": -1.0}, {"maxSweeps": -2}, {"weights": np.zeros(1500)},
               {"weights": np.ones(7)}):
        with pytest.raises(ValueError):
            ed.refineGreedyVarExperimentalDesign(k, vpool, list(vstart), **kw)
    with pytest.raises(ValueError):              # a repeated point: the Gram without a nugget is singular
        ed.refineGreedyVarExperimentalDesign(k, vpool, [5, 5, 7])


@pytest.mark.gpu
def test_greedy_runs_unchanged_by_factor_storage(env):
    from gpexp_b200.engine import GreedyVarEngine
    ed = env.ed
    rng = np.random.default_rng(4)
    pool = rng.uniform(-1, 1, (2500, 2))
    cf = _mi_cost_function(env, "matern32", pool, 1e-4)
    ed.performGreedyMIExperimentalDesign(cf, 30, start=7)
    plain = cf.lastEngine
    kept = ed._mi_new_engine(cf, 30, keep_factors=True)
    kept.run(30, start=7)
    assert plain.UA is None and plain.UQ is None
    for a, b in ((plain.picks, kept.picks), (plain.pick_scores, kept.pick_scores), (plain.pick_pivots, kept.pick_pivots),
                 (plain.W, kept.W), (plain.Us, kept.Us), (plain.num, kept.num), (plain.pd, kept.pd)):
        assert env.torch.equal(a, b)
    w = rng.uniform(0.5, 2.0, 2500)
    design = ed.performGreedyVarExperimentalDesign(_kernel("matern32"), pool, 30, 2, weights=w)
    dev = _kernel("matern32")._bind()
    engs = [GreedyVarEngine(dev, dev.points(pool), 30, weights=w, keep_factors=k) for k in (False, True)]
    for e in engs:
        e.run(30)
    assert engs[0].U is None
    assert np.array_equal(design, pool[engs[0].indices()])
    for a, b in ((engs[0].picks, engs[1].picks), (engs[0].pick_scores, engs[1].pick_scores),
                 (engs[0].pick_pivots, engs[1].pick_pivots), (engs[0].W, engs[1].W), (engs[0].var, engs[1].var)):
        assert env.torch.equal(a, b)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, mi_args, var_args, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["GPX_MI_BLK"] = "256"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        import gpexp_b200.experimentalDesign as ed
        from gpexp_b200 import gp
        from gpexp_b200.approximation import Space
        from gpexp_b200.engine import Shard
        ed.VERBOSE = False
        pool, start, noise = mi_args
        cf = ed.costFunctionGP_MI(gp.GP(_kernel("se_ard"), noise), 1, Space(2, None, None), nmc=pool.shape[0], mcpoints=pool)
        idx = ed.refineGreedyMIExperimentalDesign(cf, list(start), returnIndices=True, shard=Shard())
        vpool, vstart, w = var_args
        vout, info = ed.refineGreedyVarExperimentalDesign(_kernel("se_ard"), vpool, list(vstart), weights=w, nFixed=3,
                                                          returnIndices=True, returnInfo=True, shard=Shard())
        q.put((rank, ([int(i) for i in idx], list(cf.lastSwaps), cf.lastScores.tolist(), cf.lastMI),
               ([int(i) for i in vout], info["swaps"], info["scores"].tolist(), info["logdet"])))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_refinements_match_single_gpu(env):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("a 2-rank NCCL run needs two visible GPUs")
    import torch.multiprocessing as mp
    pool, start, noise, (d_ref, s_ref, w_ref, _, _) = _mi_problem("se_ard", "nu")
    vpool, vstart, w, (vd_ref, vs_ref, vw_ref, _, _) = _var_problem("se_ard", True)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    mp.spawn(_sharded_worker, args=(2, _free_port(), (pool, start, noise), (vpool, vstart, w), q), nprocs=2, join=True)
    for _ in range(2):
        rank, mi, var = q.get()
        assert mi[0] == d_ref and mi[1] == w_ref, rank
        assert _rel(mi[2], s_ref) <= 1e-8
        assert var[0] == vd_ref and var[1] == vw_ref, rank
        assert _rel(var[2], vs_ref) <= 1e-9
