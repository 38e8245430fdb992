"""Exchange refinement of discrete IVAR designs (refineGreedyIVARExperimentalDesign) and the design-point deletion under it.

The oracles are tests/ivar_exchange_oracle.py: fast_design_delete (the Givens downdate in numpy, any float dtype),
fast_exchange_ivar (the queue-ordered pass with D minus the removed point refactored from scratch at every step) and
ref_exchange_ivar (the same decisions from the reference's pinv cost loop).
CPU: the downdate against a fresh Cholesky factor and a longdouble restatement; the fast exchange oracle against the
reference loop (SE, Matern 3/2, Mehler; a noise vector; weights), monotone cost and 1-swap optimality of the result.
GPU: gpx_design_delete_factor / gpx_design_delete_rows against the oracle (ragged column counts, n from 1 to 1000);
delete + re-append restores the cost; the exchange pass against the oracle over every kernel family, a noise function,
mcWeights, both contraction cores and both scoring modes; idempotence and argument checks; a mid-size cfg-2 problem; a
2-rank NCCL run when two GPUs are visible."""
import functools
import os
import socket

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests import ivar_exchange_oracle as xo

EPS = float(np.finfo(np.float64).eps)
DMMA, I8 = 1, 2
RTOL = 1e-8


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b))) if a.size else 0.0


def _factor_state(kern, design, x, noise):
    """U (upper, K_DD + noise I = U^T U), W = U^-T K(D, x), var."""
    from scipy.linalg import solve_triangular
    K = kern.gram(design, design) + noise * np.eye(design.shape[0])
    U = np.linalg.cholesky(K).T
    W = solve_triangular(U, kern.gram(design, x), trans="T", lower=False)
    return U, W, kern.prior(x) - np.sum(W * W, axis=0)


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
DELETE_CASES = [(n, j) for n in (1, 2, 7, 40) for j in sorted({0, n // 2, n - 1})]


@pytest.mark.parametrize("n,j", DELETE_CASES, ids=[f"n{n}-j{j}" for n, j in DELETE_CASES])
def test_fast_design_delete_equals_refactoring(n, j):
    rng = np.random.default_rng(100 + n)
    kern = orc.KernelSpec.se([0.3, 0.45], 1.7, 2)
    design, x = rng.uniform(-1, 1, (n, 2)), rng.uniform(-1, 1, (60, 2))
    noise = 1e-3
    U, W, var = _factor_state(kern, design, x, noise)
    U1, W1, r, var1 = xo.fast_design_delete(U, W, var, j)
    # a fresh factorisation of the design without point j
    keep = np.delete(np.arange(n), j)
    if n > 1:
        U0, W0, var0 = _factor_state(kern, design[keep], x, noise)
        assert np.max(np.abs(U1 - U0)) <= 1e-12 * np.max(np.abs(U0))
        assert np.max(np.abs(W1 - W0)) <= 1e-11
    else:
        var0 = kern.prior(x)
    assert np.max(np.abs(var1 - var0)) <= 1e-12 * kern.signal
    assert np.array_equal(W1[:j], W[:j])
    # against the same algorithm in long double: 8 (n - j) eps |W[:, x]|_2 per column; var' = var + r^2 within two
    # roundings of k(x,x) (the square and the sum) plus what the residual's own error contributes
    L = np.longdouble
    U2, W2, r2, var2 = xo.fast_design_delete(U.astype(L), W.astype(L), var.astype(L), j)
    bound = 8 * (n - j) * EPS * np.linalg.norm(W, axis=0)
    assert np.all(np.abs(W1 - W2.astype(np.float64)) <= bound[None, :])
    assert np.all(np.abs(r - r2.astype(np.float64)) <= bound)
    assert np.all(np.abs(var1 - var2.astype(np.float64)) <= 2.0 * EPS * kern.prior(x) + 2.0 * np.abs(r) * bound)
    ubound = 8 * (n - j) * EPS * np.linalg.norm(U, axis=0)
    assert np.all(np.abs(U1 - U2.astype(np.float64)) <= np.max(ubound))
    assert np.all(np.diag(U1) >= 0.0) and np.allclose(np.tril(U1, -1), 0.0)


def _cpu_kernel(name):
    return {"se": orc.KernelSpec.se([0.3, 0.45], 1.7, 2), "matern32": orc.KernelSpec.matern32(0.5, 1.3, 2),
            "mehler": orc.KernelSpec.mehler([0.6, 0.5], 2)}[name]


CPU_X_CASES = [(k, v) for k in ("se", "matern32", "mehler") for v in ("scalar", "noise_vector", "weights")]


@pytest.mark.parametrize("kname,variant", CPU_X_CASES, ids=[f"{k}-{v}" for k, v in CPU_X_CASES])
def test_fast_exchange_equals_reference_loop(kname, variant):
    rng = np.random.default_rng(7)
    kern = _cpu_kernel(kname)
    sample = rng.standard_normal if kname == "mehler" else (lambda s: rng.uniform(-1, 1, s))
    cand, mc = sample((40, 2)), sample((300, 2))
    noise = 1e-2 if kname == "mehler" else 1e-4
    w = None
    if variant == "noise_vector":
        noise = noise * (1.0 + 10.0 * cand[:, 0] ** 2)
    elif variant == "weights":
        w = rng.uniform(0.1, 2.0, 300) / 300
    start = [int(i) for i in rng.choice(40, 6, replace=False)]
    d_ref, c_ref, s_ref, _ = xo.ref_exchange_ivar(kern, cand, mc, start, noise, RTOL, 10, mc_weights=w)
    d, c, s, margins = xo.fast_exchange_ivar(kern, cand, mc, start, noise, RTOL, 10, mc_weights=w)
    assert d == d_ref and s == s_ref
    assert _rel(c, c_ref) <= 1e-9
    assert s[-1] == 0 and sum(s) > 0                  # it stopped by itself, after swapping
    # the cost never increases
    prev = xo.design_cost(kern, cand, mc, start, noise, mc_weights=w)
    for v in c:
        assert v <= prev * (1.0 + 1e-12)
        prev = v
    # 1-swap optimal up to rtol: no exchange of one design point for one candidate is better by more than rtol
    base = xo.design_cost(kern, cand, mc, d, noise, mc_weights=w)
    for j in range(len(d)):
        for cidx in range(40):
            trial = d[:j] + [cidx] + d[j + 1:]
            assert xo.design_cost(kern, cand, mc, trial, noise, mc_weights=w) >= (1.0 - RTOL) * base * (1.0 - 1e-12)


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import _lib, kernels
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    ed.VERBOSE = False

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ed, ns.lib, ns.check, ns.gp, ns.Space, ns.kernels = torch, ed, _lib.lib, _lib.check, gpmod, Space, kernels
    ns.dev = Device.get(0)
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")


def _host(t, rows, cols):
    return t[:rows, :cols].cpu().numpy().copy()


DELETE_GPU = [(n, j) for n in (1, 2, 17, 255, 1000) for j in sorted({0, n // 2, n - 1})]


@pytest.mark.gpu
@pytest.mark.parametrize("n,j", DELETE_GPU, ids=[f"n{n}-j{j}" for n, j in DELETE_GPU])
def test_delete_kernels_match_oracle(env, n, j):
    ed = env.ed
    rng = np.random.default_rng(200 + n)
    C, M = 2001, 1501      # odd, not multiples of the 256-column block
    cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
    noise = 1e-3
    cf = ed.costFunctionGP_IVAR(env.gp.GP(env.kernels.KernelSquaredExponential([0.2, 0.3], 1.0, 2), noise), 1,
                                env.Space(2, None, None), mcPoints=mc)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, n, resident=False)
    picks = rng.choice(C, n, replace=False)
    for p in picks:
        eng.force(int(p))
    U = _host(eng.U, n, n)
    Wm, Wc = _host(eng.Wm, n, M), _host(eng.Wc, n, C)
    vM, vC = eng.varM[:M].cpu().numpy().copy(), eng.varC[:C].cpu().numpy().copy()
    pads = (eng.Wc[:n, C:].clone(), eng.Wm[:n, M:].clone())
    cost0 = float(eng.varM[:M].sum().item()) / M
    eng.remove(j)
    assert eng.n == n - 1
    for W, Wd, v, vd, cols in ((Wm, eng.Wm, vM, eng.varM, M), (Wc, eng.Wc, vC, eng.varC, C)):
        _, W1, r, v1 = xo.fast_design_delete(U, W, v, j)
        got = _host(Wd, n, cols)
        bound = 8 * (n - j) * EPS * np.linalg.norm(W, axis=0)
        assert np.array_equal(got[:j], W[:j])                                  # rows 0..j-1 untouched, bit for bit
        assert np.all(np.abs(got[: n - 1] - W1) <= bound[None, :])
        assert np.all(np.abs(got[n - 1] - r) <= bound)                         # the residual row stays in row n-1
        prior = np.ones(cols)
        assert np.all(np.abs(vd[:cols].cpu().numpy() - v1) <= 2.0 * EPS * prior + 2.0 * np.abs(r) * bound)
    assert bool((eng.Wc[:n, C:] == pads[0]).all()) and bool((eng.Wm[:n, M:] == pads[1]).all())
    U1, _, _, _ = xo.fast_design_delete(U, Wm, vM, j)
    got_u = _host(eng.U, n, n)
    ubound = 8 * (n - j) * EPS * np.max(np.linalg.norm(U, axis=0))
    assert np.all(np.abs(got_u[: n - 1, : n - 1] - np.triu(U1)) <= ubound)
    assert np.all(got_u[n - 1] == 0.0) and np.all(got_u[:, n - 1] == 0.0)
    assert np.all(np.tril(got_u[: n - 1, : n - 1], -1) == 0.0)
    keep = [int(p) for p in np.delete(picks, j)]
    assert [int(i) for i in eng.picks[: n - 1].cpu().numpy()] == keep
    piv = eng.pick_pivots[: n - 1].cpu().numpy()
    assert np.array_equal(piv[j:], np.diag(got_u)[j: n - 1] ** 2)
    # putting the removed point back restores the design's cost
    eng.force(int(picks[j]))
    cost1 = float(eng.varM[:M].sum().item()) / M
    assert abs(cost1 - cost0) <= 1e-12 * cost0


KERN_X = {"se_ard": ("se", [0.25, 0.35], 1.0), "matern12": (0.5, 0.5, 1.0), "matern32": (1.5, 0.4, 1.0),
          "matern52": (2.5, 0.4, 1.0), "mehler": ("mehler", [0.7, 0.6], None)}


def _kernels(name):
    a, b, c = KERN_X[name]
    from gpexp_b200 import kernels as K
    if a == "se":
        return orc.KernelSpec.se(b, c, 2), K.KernelSquaredExponential(b, c, 2)
    if a == "mehler":
        return orc.KernelSpec.mehler(b, 2), K.KernelMehlerND(b, 2)
    spec = {0.5: orc.KernelSpec.matern12, 1.5: orc.KernelSpec.matern32, 2.5: orc.KernelSpec.matern52}[a](b, c, 2)
    return spec, K.KernelIsoMatern(b, c, 2, nu=a)


def nu_x(p):
    return 1e-4 * (1.0 + 20.0 * p[:, 0] ** 2)


# seeds whose oracle runs swap and keep every decision more than 1e-6 (relative) away from flipping
PROBLEM_SEEDS = {("matern12", "scalar"): 4, ("matern32", "scalar"): 4, ("se_ard", "noise_func"): 5}


@functools.lru_cache(maxsize=None)
def _problem(kname, variant):
    """C = 2 000 candidates, M = 3 000 integration points, a random 20-point start; the oracle's run of the exchange."""
    rng = np.random.default_rng(PROBLEM_SEEDS.get((kname, variant), 3))
    spec, _ = _kernels(kname)
    sample = rng.standard_normal if kname == "mehler" else (lambda s: rng.uniform(-1, 1, s))
    cand, mc = sample((2000, 2)), sample((3000, 2))
    start = tuple(int(i) for i in rng.choice(2000, 20, replace=False))
    noise = 1e-2 if kname == "mehler" else 1e-4
    w = None
    if variant == "noise_func":
        noise = nu_x(cand)
    elif variant == "weights":
        w = rng.uniform(0.1, 2.0, 3000) / 3000
    out = xo.fast_exchange_ivar(spec, cand, mc, list(start), noise, RTOL, 10, mc_weights=w)
    return cand, mc, start, noise, w, out


X_CASES = ([(k, "scalar", "i8", "contraction") for k in KERN_X] +
           [("se_ard", v, core, mode) for v in ("noise_func", "weights") for core in ("i8", "dmma")
            for mode in ("contraction", "resident")] +
           [("matern32", "scalar", "dmma", "contraction"), ("mehler", "scalar", "i8", "resident")])


def _cost_function(env, kname, variant, cand, mc, noise, w):
    _, k = _kernels(kname)
    if variant == "noise_func":
        space = env.Space(2, None, None, noise=nu_x)
        gp_noise = 0.5       # not used once the space has a noise function
    else:
        space, gp_noise = env.Space(2, None, None), float(noise)
    return env.ed.costFunctionGP_IVAR(env.gp.GP(k, gp_noise), 1, space, mcPoints=mc, mcWeights=w)


@pytest.mark.gpu
@pytest.mark.parametrize("kname,variant,core,mode", X_CASES, ids=["-".join(c) for c in X_CASES])
def test_exchange_matches_oracle(env, kname, variant, core, mode):
    cand, mc, start, noise, w, (d_ref, c_ref, s_ref, margins) = _problem(kname, variant)
    # no decision of the oracle lies within 1e-6 of flipping, so rounding cannot change a decision
    assert min(margins) > 1e-6, min(margins)
    assert sum(s_ref) > 0
    cf = _cost_function(env, kname, variant, cand, mc, noise, w)
    env.check(env.lib.gpx_set_ivar_core(env.dev.h, DMMA if core == "dmma" else I8), "gpx_set_ivar_core")
    try:
        idx = env.ed.refineGreedyIVARExperimentalDesign(cf, cand, list(start), maxSweeps=10, rtol=RTOL, returnIndices=True,
                                                        resident=(mode == "resident"))
    finally:
        env.check(env.lib.gpx_set_ivar_core(env.dev.h, I8), "gpx_set_ivar_core")
    assert [int(i) for i in idx] == d_ref
    assert cf.lastSwaps == s_ref
    assert _rel(cf.lastScores, c_ref) <= 1e-9
    assert _rel(cf.lastCost, c_ref[-1]) <= 1e-9
    spec, _ = _kernels(kname)
    assert _rel(cf.lastCost, xo.design_cost(spec, cand, mc, d_ref, noise, mc_weights=w)) <= 1e-9


@pytest.mark.gpu
def test_refine_is_idempotent_and_checks_arguments(env):
    ed = env.ed
    cand, mc, start, noise, w, (d_ref, _, _, _) = _problem("se_ard", "scalar")
    cf = _cost_function(env, "se_ard", "scalar", cand, mc, noise, None)
    once = ed.refineGreedyIVARExperimentalDesign(cf, cand, list(start), returnIndices=True)
    assert [int(i) for i in once] == d_ref
    twice = ed.refineGreedyIVARExperimentalDesign(cf, cand, once, returnIndices=True)
    assert cf.lastSwaps == [0] and [int(i) for i in twice] == [int(i) for i in once]
    pts = ed.refineGreedyIVARExperimentalDesign(cf, cand, once)
    assert np.array_equal(pts, cand[once])
    same = ed.refineGreedyIVARExperimentalDesign(cf, cand, list(start), maxSweeps=0, returnIndices=True)
    assert [int(i) for i in same] == list(start) and cf.lastSwaps == [] and cf.lastScores.size == 0
    assert _rel(cf.lastCost, xo.design_cost(_kernels("se_ard")[0], cand, mc, list(start), noise)) <= 1e-9
    for bad in ([0, 2000], [-1, 3], [0.0, 1.0], [], np.array([[1, 2]])):
        with pytest.raises(ValueError):
            ed.refineGreedyIVARExperimentalDesign(cf, cand, bad)
    with pytest.raises(ValueError):
        ed.refineGreedyIVARExperimentalDesign(cf, cand, [1, 2], rtol=-1e-3)
    with pytest.raises(ValueError):
        ed.refineGreedyIVARExperimentalDesign(cf, cand, [1, 2], maxSweeps=-1)
    # a repeated point without noise: the factor has a non-finite (or zero) pivot and cannot be refined
    cf0 = ed.costFunctionGP_IVAR(env.gp.GP(env.kernels.KernelSquaredExponential([0.25, 0.35], 1.0, 2), 0.0), 1,
                                 env.Space(2, None, None), mcPoints=mc)
    dup = ed.beginGreedyIVARExperimentalDesign(cf0, cand, 3, resident=False)
    for i in (5, 5, 7):
        dup.force(i)
    if not bool(env.torch.isfinite(dup.U[:3, :3]).all()):
        with pytest.raises(ValueError):
            ed.refineGreedyIVARExperimentalDesign(cf0, cand, [5, 5, 7])
    # snapshots do not survive a remove()
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, 4, resident=False)
    for i in start[:4]:
        eng.force(i)
    snap = eng.snapshot()
    eng.remove(1)
    with pytest.raises(ValueError):
        eng.restore(snap)


@functools.lru_cache(maxsize=None)
def _cfg2_problem():
    rng = np.random.default_rng(2)
    cand, mc = rng.uniform(0, 1, (5000, 2)), rng.uniform(0, 1, (5000, 2))
    spec = orc.KernelSpec.se([0.06, 0.09], 1.0, 2)
    idx, costs = orc.fast_greedy_ivar(spec, cand, mc, 32, 1e-6)
    out = xo.fast_exchange_ivar(spec, cand, mc, idx, 1e-6, RTOL, 10)
    return cand, mc, idx, costs[-1][idx[-1]], out


@pytest.mark.gpu
def test_mid_size_cfg2_kernel(env):
    ed = env.ed
    cand, mc, idx, greedy_cost, (d_ref, c_ref, s_ref, margins) = _cfg2_problem()
    # every decision lies beyond 10x the 1e-9 agreement of the scores (the closest is 5e-7 from flipping)
    assert min(margins) > 1e-8
    cf = ed.costFunctionGP_IVAR(env.gp.GP(env.kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2), 1e-6), 1,
                                env.Space(2, None, None), mcPoints=mc)
    g = ed.performGreedyIVARExperimentalDesign(cf, cand, 32, returnIndices=True)
    assert [int(i) for i in g] == idx
    out = ed.refineGreedyIVARExperimentalDesign(cf, cand, g, returnIndices=True)
    assert [int(i) for i in out] == d_ref and cf.lastSwaps == s_ref
    assert _rel(cf.lastScores, c_ref) <= 1e-9
    assert cf.lastCost <= greedy_cost


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, cand, mc, start, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        import gpexp_b200.experimentalDesign as ed
        from gpexp_b200 import gp, kernels
        from gpexp_b200.approximation import Space
        from gpexp_b200.engine import Shard
        ed.VERBOSE = False
        cf = ed.costFunctionGP_IVAR(gp.GP(kernels.KernelSquaredExponential([0.25, 0.35], 1.0, 2), 1e-4), 1,
                                    Space(2, None, None), mcPoints=mc)
        out = {}
        for resident in (False, True):
            idx = ed.refineGreedyIVARExperimentalDesign(cf, cand, list(start), returnIndices=True, shard=Shard(),
                                                        resident=resident)
            out[resident] = ([int(i) for i in idx], list(cf.lastSwaps), cf.lastScores.tolist())
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_exchange_matches_single_gpu(env):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("a 2-rank NCCL run needs two visible GPUs")
    import torch.multiprocessing as mp
    cand, mc, start, noise, _, (d_ref, c_ref, s_ref, _) = _problem("se_ard", "scalar")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    mp.spawn(_sharded_worker, args=(2, _free_port(), cand, mc, start, q), nprocs=2, join=True)
    results = dict(q.get() for _ in range(2))
    for rank in (0, 1):
        for resident in (False, True):
            idx, swaps, scores = results[rank][resident]
            assert idx == d_ref and swaps == s_ref, (rank, resident)
            assert _rel(scores, c_ref) <= 1e-9
