"""Greedy IVAR with weighted integration points (costFunctionGP_IVAR.mcWeights): cost_w(D) = |sum_m w_m var_D(x_m)|.

The oracles are oracle/gpexp_oracle.py's ref_greedy_ivar and fast_greedy_ivar with mc_weights.
CPU: the vectorised weighted oracle against the reference's pinv loop (SE, Matern, Mehler; random, half-zero and
Gauss-Legendre weights; with and without a noise function); w = 1/M (M = 2^k) reproduces the unweighted oracles bit for bit;
integer weights equal replicated points; rejected weights.
GPU: the weighted epilogues exactly (INT8 core bit for bit, DMMA cores within the FP64 bound); the weighted sum, row sum and
covariance update exactly; w = 1/M bit-identical to the unweighted design in every loop mode; non-uniform weights against the
oracles; zero weights as dropped points; the reference's own optimiser loop; cfg-2-size scoring."""
import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests.cases import product_kernel, spec
from tests.test_ivar_contraction_exact import gx  # noqa: F401  (the exact-contraction harness's device fixture)

DMMA, I8 = 1, 2


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.abs(np.asarray(b))))


def _sample(name, rng, *shapes):
    d = spec(name).dim
    if name.startswith("mehler"):
        return [rng.standard_normal((n, d)) for n in shapes]
    return [rng.uniform(-1, 1, (n, d)) for n in shapes]


def nu_smooth(p):
    return 1e-4 + 1e-3 * p[:, 0] ** 2


def gauss_legendre_grid(n, d, lo=-1.0, hi=1.0):
    """Tensor Gauss-Legendre rule of n^d nodes on [lo, hi]^d: (points (n^d, d), weights summing to the box volume)."""
    x, w = np.polynomial.legendre.leggauss(n)
    x = lo + (x + 1.0) * (hi - lo) / 2.0
    w = w * (hi - lo) / 2.0
    grids = np.meshgrid(*([x] * d), indexing="ij")
    wgrid = np.meshgrid(*([w] * d), indexing="ij")
    pts = np.stack([g.ravel() for g in grids], axis=1)
    return pts, np.prod(np.stack([g.ravel() for g in wgrid], axis=1), axis=1)


def _weights(profile, mc, rng):
    if profile == "random":
        return rng.uniform(0.1, 2.0, mc.shape[0]) / mc.shape[0]
    if profile == "half_zero":
        return np.where(mc[:, 0] < 0.0, 0.0, 2.0 / mc.shape[0])
    return np.exp(-np.sum(mc ** 2, axis=1)) / mc.shape[0]   # smooth positive


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
CPU_CASES = [(k, p, nf) for k in ("se_ard_2d_wide", "matern_5d", "mehler_3d") for p in ("random", "half_zero", "gauss")
             for nf in (False, True)]


@pytest.mark.parametrize("name,profile,with_nf", CPU_CASES, ids=[f"{k}-{p}-{'nf' if n else 'scalar'}" for k, p, n in CPU_CASES])
def test_fast_weighted_oracle_equals_reference_loop(name, profile, with_nf):
    rng = np.random.default_rng(51)
    ks = spec(name)
    cand, = _sample(name, rng, 40)
    if profile == "gauss":
        mc, w = gauss_legendre_grid(3 if ks.dim > 2 else 8, ks.dim, -2.0 if name.startswith("mehler") else -1.0,
                                    2.0 if name.startswith("mehler") else 1.0)
    else:
        mc, = _sample(name, rng, 150)
        w = _weights(profile, mc, rng)
    noise = 1e-2 if name.startswith("mehler") else 1e-5
    nf = (lambda p: 10.0 * noise * (1.0 + p[:, 0] ** 2)) if with_nf else None
    ref_idx, ref_costs = orc.ref_greedy_ivar(ks, cand, mc, 6, noise, mc_weights=w, noise_func=nf)
    idx, costs = orc.fast_greedy_ivar(ks, cand, mc, 6, noise if nf is None else nf(cand), mc_weights=w)
    assert idx == ref_idx
    for s in range(6):
        assert _rel(costs[s], ref_costs[s]) <= 1e-9, s


def test_uniform_power_of_two_weights_are_the_unweighted_oracles():
    """M = 256, w = 1/M: the weighted forms of ref_greedy_ivar and fast_greedy_ivar reproduce their unweighted forms bit
    for bit."""
    rng = np.random.default_rng(52)
    cand, mc = rng.uniform(-1, 1, (30, 2)), rng.uniform(-1, 1, (256, 2))
    ks, s2, w = spec("se_ard_2d_wide"), 1e-4, np.full(256, 1.0 / 256)
    a_idx, a_costs = orc.ref_greedy_ivar(ks, cand, mc, 5, s2)
    b_idx, b_costs = orc.ref_greedy_ivar(ks, cand, mc, 5, s2, mc_weights=w)
    assert a_idx == b_idx and all(np.array_equal(x, y) for x, y in zip(a_costs, b_costs))
    f_idx, f_costs = orc.fast_greedy_ivar(ks, cand, mc, 5, s2)
    g_idx, g_costs = orc.fast_greedy_ivar(ks, cand, mc, 5, s2, mc_weights=w)
    assert f_idx == g_idx == a_idx and all(np.array_equal(x, y) for x, y in zip(f_costs, g_costs))


def test_integer_weights_equal_replicated_points():
    rng = np.random.default_rng(53)
    cand, mc = rng.uniform(-1, 1, (80, 2)), rng.uniform(-1, 1, (120, 2))
    ks, s2 = spec("se_ard_2d_wide"), 1e-5
    k = rng.integers(1, 5, mc.shape[0])
    rep = np.repeat(mc, k, axis=0)
    a_idx, a_costs = orc.fast_greedy_ivar(ks, cand, mc, 10, s2, mc_weights=k.astype(np.float64))
    b_idx, b_costs = orc.fast_greedy_ivar(ks, cand, rep, 10, s2, mc_weights=np.ones(rep.shape[0]))
    assert a_idx == b_idx == orc.fast_greedy_ivar(ks, cand, rep, 10, s2)[0]
    for s in range(10):
        assert _rel(a_costs[s], b_costs[s]) <= 1e-12, s


BAD = [(lambda n: np.full(n + 1, 1.0), "values for"), (lambda n: np.where(np.arange(n) == 3, np.nan, 1.0), "not finite"),
       (lambda n: np.where(np.arange(n) == 3, np.inf, 1.0), "not finite"),
       (lambda n: np.where(np.arange(n) == 3, -1e-3, 1.0), "negative"), (lambda n: np.zeros(n), "no positive")]


@pytest.mark.parametrize("bad,what", BAD, ids=["length", "nan", "inf", "negative", "zeros"])
def test_bad_weights_are_rejected_before_any_device_call(bad, what):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    rng = np.random.default_rng(54)
    cand, mc = rng.uniform(-1, 1, (50, 2)), rng.uniform(-1, 1, (80, 2))
    cf = ed.costFunctionGP_IVAR(gpmod.GP(product_kernel("se_ard_2d_wide"), 1e-6), 3, Space(2, None, None), mcPoints=mc,
                                mcWeights=bad(80))
    for call in (lambda: ed.performGreedyIVARExperimentalDesign(cf, cand, 4),
                 lambda: ed.beginGreedyIVARExperimentalDesign(cf, cand, 4),
                 lambda: ed.scoreCandidatesIVAR(cf, cand[:3], cand),
                 lambda: cf.evaluate(cand[:3]),
                 lambda: cf.derivative(cand[:3])):
        with pytest.raises(ValueError, match=what):
            call()


def test_weights_sized_for_other_points_are_rejected_with_default_mc_points():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    rng = np.random.default_rng(56)
    space = Space(2, lambda s: rng.uniform(-1, 1, s), None)
    cf = ed.costFunctionGP_IVAR(gpmod.GP(product_kernel("se_ard_2d_wide"), 1e-6), 1, space)
    assert cf.mcWeights is None and cf.nMC == 10000
    cf.mcWeights = np.ones(64)
    with pytest.raises(ValueError, match="64 values for 10000 points"):
        ed.performGreedyIVARExperimentalDesign(cf, np.zeros((5, 2)), 2)


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import _lib, engine
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device, ptr

    class NS:
        pass
    ns = NS()
    ns.ed, ns.lib, ns.check, ns.engine, ns.gp, ns.Space, ns.ptr = ed, _lib.lib, _lib.check, engine, gpmod, Space, ptr
    ns.dev = Device.get(0)
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")
    ns.dev.force_diff_form = False


def _weighted_score(P, core, w):
    """gpx_score_ivar_w on a Problem of tests/test_ivar_contraction_exact.py: the scores of every candidate."""
    dev = P.dev
    wd = dev.upload(w)
    P.gx.check(P.lib.gpx_set_ivar_core(dev.h, core), "gpx_set_ivar_core")
    try:
        P.gx.check(P.lib.gpx_score_ivar_w(
            dev.h, P.mode, P.ptr(P.Wm), P.ldm, P.ptr(P.vM), P.ptr(P.ra), P.M, P.ptr(P.Wc), P.ldc, P.ptr(P.vC), P.ptr(P.rb),
            P.C, P.n, 0.0, 0.0, P.ptr(wd), None, P.ptr(P.ws), P.ptr(P.out), P.ptr(P.best), P.ptr(P.idx), dev.stream),
            "gpx_score_ivar_w")
    finally:
        P.gx.check(P.lib.gpx_set_ivar_core(dev.h, I8), "gpx_set_ivar_core")
    dev.sync()
    return P.out[: P.C].cpu().numpy().copy()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 255])
@pytest.mark.parametrize("family", ["se", "matern", "mehler"])
@pytest.mark.parametrize("expanded", [False, True])
def test_weighted_epilogue_exact(gx, family, expanded, n):
    """k = 0, varM = 0, varC = 1, one non-zero W_M column m* at a tile edge, w_m = 2^((m mod 9) - 4): the INT8 core gives
    fl((w_m* S_model) S_model) = w_m* fl(S_model^2) bit for bit; the tensor-map and generic DMMA cores stay within the
    FP64 bound scaled by w_m*."""
    from tests.test_ivar_contraction_exact import (C_DEF, FAMILIES, M_DEF, M_STAR, Problem, _cycle, dmma_score_ok,
                                                   pair_table, patterns)
    model, exact, absdot = pair_table(n)
    pm, _ = patterns(n)
    w = 2.0 ** ((np.arange(M_DEF) % 9) - 4)
    rot = list(FAMILIES).index(family) + 2 * expanded
    problems = {"i8": Problem(gx, family, expanded, M_DEF, C_DEF, n), "generic": Problem(gx, family, expanded, M_DEF, C_DEF,
                                                                                         n, padded=False)}
    for i, (_, x) in enumerate(pm):
        cols, which = _cycle(n, i + rot, C_DEF)
        m = M_STAR[(i + rot) % 4] % M_DEF
        for P in problems.values():
            P.set_wc(cols)
            P.set_wm_column(m, x)
        got = _weighted_score(problems["i8"], I8, w)
        with np.errstate(over="ignore", under="ignore"):
            want = np.abs((w[m] * model[i, which]) * model[i, which])
        bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
        assert bad.size == 0, (family, expanded, n, i, m, got[bad[:3]], want[bad[:3]])
        # away from the overflow / underflow edge of S^2, where a scaled square and a square round differently
        safe = (absdot[i, which] < 2.0 ** 500) & (absdot[i, which] > 2.0 ** -400)
        for core, P in (("tensor-map", problems["i8"]), ("generic", problems["generic"])):
            got = _weighted_score(P, DMMA, w)
            ok = dmma_score_ok(got / w[m] / M_DEF, exact[i, which], absdot[i, which], n, M_DEF)
            assert np.all(ok | ~safe), (core, family, expanded, n, i, m)


@pytest.mark.gpu
def test_weighted_sum_rowsum_and_cov_update_exact(env):
    """Integer data, power-of-two weights: every product and partial sum is exact, so the results are exact integers
    scaled by powers of two, across the 256-thread, 4096-element block and row-segment edges."""
    dev, lib, ptr = env.dev, env.lib, env.ptr
    rng = np.random.default_rng(55)
    for n in (1, 255, 256, 4097, 70_001):
        v = rng.integers(-1000, 1000, n).astype(np.float64)
        w = 2.0 ** rng.integers(-6, 3, n)
        out, vd, wd = dev.zeros(1), dev.upload(v), dev.upload(w)   # held: a freed upload's block could be reused
        env.check(lib.gpx_sum_w(dev.h, ptr(vd), ptr(wd), n, ptr(out), dev.stream), "gpx_sum_w")
        assert float(out.item()) == float(np.sum(v * w)), n   # |sum| < 2^53 in units of 2^-6: exact either way
    rows, cols, ld = 7, 5003, 5008
    A = rng.integers(-500, 500, (rows, ld)).astype(np.float64)
    w = 2.0 ** rng.integers(-5, 2, cols)
    out, Ad, wd = dev.zeros(rows), dev.upload(A), dev.upload(w)
    env.check(lib.gpx_rowsum_w(dev.h, ptr(Ad), rows, cols, ld, ptr(wd), ptr(out), dev.stream), "gpx_rowsum_w")
    assert np.array_equal(out.cpu().numpy(), A[:, :cols] @ w)
    for M, C in ((1000, 999), (5003, 1536)):
        ldc = C + (C & 1)
        cov = rng.integers(-300, 300, (M, ldc)).astype(np.float64)
        w = 2.0 ** rng.integers(-4, 3, M)
        seg = int(lib.gpx_cov_segments(M, C))
        ldp = ldc
        part = dev.zeros(seg * ldp)
        cd, wd = dev.upload(cov), dev.upload(w)
        env.check(lib.gpx_cov_update_w(dev.h, ptr(cd), ldc, M, C, None, None, ptr(wd), ptr(part), ldp, dev.stream),
                  "gpx_cov_update_w")
        got = part.cpu().numpy().reshape(seg, ldp)[:, :C].sum(axis=0)
        assert np.array_equal(got, (w[:, None] * cov[:, :C] ** 2).sum(axis=0)), (M, C)
        assert np.array_equal(cd.cpu().numpy(), cov)   # a = b = NULL only reduces


LOOP_MODES = ["trace_i8", "trace_dmma", "trace_resident", "loop_i8", "loop_dmma", "resident", "one_kernel"]


def _run_mode(env, cf, cand, N, mode):
    ed = env.ed
    env.check(env.lib.gpx_set_ivar_core(env.dev.h, DMMA if mode.endswith("dmma") else I8), "gpx_set_ivar_core")
    try:
        resident = mode in ("trace_resident", "resident", "one_kernel")
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=resident)
        if mode.startswith("trace"):
            eng.score_trace = []
        if resident:
            eng.ONE_KERNEL_PAIRS = cand.shape[0] * cf.mcPoints.shape[0] if mode == "one_kernel" else 0
        idx = [int(i) for i in eng.run(N)]
    finally:
        env.check(env.lib.gpx_set_ivar_core(env.dev.h, I8), "gpx_set_ivar_core")
    return idx, eng.pick_scores[:N].cpu().numpy(), eng.pivots(), eng.score_trace


PLUMB = [("se_ard_2d_wide", False), ("matern_5d", False), ("mehler_3d", False), ("se_ard_2d_wide", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,diff", PLUMB, ids=[f"{n}-{'diff' if d else 'auto'}" for n, d in PLUMB])
def test_uniform_weights_are_bit_identical_in_every_loop_mode(env, name, diff):
    """M = 2048, w = 1/M: picks, pick scores, pivots and every traced score vector equal the unweighted run bit for bit;
    w = 1 gives M x the unweighted scores bit for bit."""
    ed = env.ed
    cand, mc = _sample(name, np.random.default_rng(56), 700, 2048)
    k, N = product_kernel(name), 12
    noise = 1e-2 if name.startswith("mehler") else 1e-6
    cf0 = ed.costFunctionGP_IVAR(env.gp.GP(k, noise), 1, env.Space(spec(name).dim, None, None), mcPoints=mc)
    cf1 = ed.costFunctionGP_IVAR(env.gp.GP(k, noise), 1, env.Space(spec(name).dim, None, None), mcPoints=mc,
                                 mcWeights=np.full(2048, 1.0 / 2048))
    cfm = ed.costFunctionGP_IVAR(env.gp.GP(k, noise), 1, env.Space(spec(name).dim, None, None), mcPoints=mc,
                                 mcWeights=np.ones(2048))
    env.dev.force_diff_form = diff
    try:
        for mode in LOOP_MODES:
            a = _run_mode(env, cf0, cand, N, mode)
            b = _run_mode(env, cf1, cand, N, mode)
            c = _run_mode(env, cfm, cand, N, mode)
            assert a[0] == b[0] == c[0], (name, mode)
            assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]), (name, mode)
            assert np.array_equal(a[1] * 2048, c[1]), (name, mode)
            if a[3] is not None:
                for s, (x, y, z) in enumerate(zip(a[3], b[3], c[3])):
                    assert np.array_equal(x, y) and np.array_equal(x * 2048, z), (name, mode, s)
    finally:
        env.dev.force_diff_form = False


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["se_ard_2d_wide", "matern_5d", "mehler_3d"])
def test_nonuniform_weights_match_reference_loop(env, name):
    ed = env.ed
    rng = np.random.default_rng(57)
    cand, mc = _sample(name, rng, 120, 600)
    w = _weights("smooth", mc, rng)
    k, ks, N = product_kernel(name), spec(name), 8
    noise = 1e-2 if name.startswith("mehler") else 1e-5
    for nf in (None, lambda p: 10.0 * noise * (1.0 + p[:, 0] ** 2)):
        ref_idx, ref_costs = orc.ref_greedy_ivar(ks, cand, mc, N, noise, mc_weights=w, noise_func=nf)
        want = np.array([c[i] for c, i in zip(ref_costs, ref_idx)])
        cf = ed.costFunctionGP_IVAR(env.gp.GP(k, noise), 1, env.Space(ks.dim, None, None, noise=nf), mcPoints=mc,
                                    mcWeights=w)
        for mode in LOOP_MODES:
            idx, scores, _, trace = _run_mode(env, cf, cand, N, mode)
            assert idx == ref_idx, (name, mode, nf is None)
            assert _rel(scores, want) <= 1e-9, (name, mode)
            if trace is not None:
                for s, c in enumerate(trace):
                    assert _rel(c, ref_costs[s]) <= 1e-9, (name, mode, s)
        for i in range(N):
            one = ed.costFunctionGP_IVAR(env.gp.GP(k, noise), i + 1, env.Space(ks.dim, None, None, noise=nf), mcPoints=mc,
                                         mcWeights=w).evaluate(cand[ref_idx[: i + 1]])
            assert abs(one - want[i]) <= 1e-9 * want[i], (name, i)


@pytest.mark.gpu
def test_nonuniform_weights_mid_size_every_loop_mode(env):
    """3 000 candidates x 20 000 integration points, 16 steps, cfg-2's kernel, smooth weights, with and without a noise
    function: the picks of the vectorised weighted oracle."""
    ed = env.ed
    rng = np.random.default_rng(58)
    cand, mc = rng.uniform(-1, 1, (3000, 2)), rng.uniform(-1, 1, (20_000, 2))
    w = _weights("smooth", mc, rng)
    ks, k, N = spec("se_ard_2d"), product_kernel("se_ard_2d"), 16
    for nf in (None, nu_smooth):
        ref, costs = orc.fast_greedy_ivar(ks, cand, mc, N, 1e-6 if nf is None else nf(cand), mc_weights=w)
        want = np.array([c[i] for c, i in zip(costs, ref)])
        cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 1, env.Space(2, None, None, noise=nf), mcPoints=mc, mcWeights=w)
        for mode in LOOP_MODES:
            idx, scores, _, _ = _run_mode(env, cf, cand, N, mode)
            assert idx == ref, (mode, nf is None)
            assert _rel(scores, want) <= 1e-9, mode


@pytest.mark.gpu
def test_score_candidates_evaluate_and_derivative(env):
    ed = env.ed
    rng = np.random.default_rng(59)
    ks, k = spec("se_ard_2d_wide"), product_kernel("se_ard_2d_wide")
    cand, mc, design = rng.uniform(-1, 1, (3000, 2)), rng.uniform(-1, 1, (2000, 2)), rng.uniform(-1, 1, (20, 2))
    w = _weights("smooth", mc, rng)
    for nf in (None, nu_smooth):
        cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-5), 20, env.Space(2, None, None, noise=nf), mcPoints=mc, mcWeights=w)
        costs, best = ed.scoreCandidatesIVAR(cf, design, cand)
        from scipy.linalg import solve_triangular
        nug = 1e-5 if nf is None else nf(design)
        low = np.linalg.cholesky(ks.gram(design, design) + np.diag(np.broadcast_to(nug, (20,))))
        w_m, w_c = solve_triangular(low, ks.gram(design, mc), lower=True), solve_triangular(low, ks.gram(design, cand), lower=True)
        var_m, var_c = ks.prior(mc) - np.sum(w_m ** 2, axis=0), ks.prior(cand) - np.sum(w_c ** 2, axis=0)
        fast = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, 1e-5 if nf is None else nf(cand), mc_weights=w)
        assert best == int(np.argmin(fast)) and _rel(costs, fast) <= 1e-9
        var = orc.fast_posterior_variance(ks, design, mc, nug)
        assert abs(cf.evaluate(design) - abs(np.sum(w * var))) <= 1e-9 * abs(np.sum(w * var))
    cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-5), 20, env.Space(2, None, None), mcPoints=mc, mcWeights=w)
    want = orc.fast_variance_derivative(ks, design, mc, 1e-5) @ w
    got = cf.derivative(design)
    assert np.max(np.abs(got - want)) <= 1e-9 * np.max(np.abs(want))


@pytest.mark.gpu
def test_zero_weights_drop_points(env):
    ed = env.ed
    rng = np.random.default_rng(60)
    cand, mc = rng.uniform(-1, 1, (1500, 2)), rng.uniform(-1, 1, (3000, 2))
    k, N = product_kernel("se_ard_2d_wide"), 16
    keep = mc[:, 1] > 0.2
    w = keep.astype(np.float64)
    cf_w = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 1, env.Space(2, None, None), mcPoints=mc, mcWeights=w)
    cf_s = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 1, env.Space(2, None, None), mcPoints=mc[keep],
                                  mcWeights=np.ones(int(keep.sum())))
    for resident in (False, True):
        a = ed.performGreedyIVARExperimentalDesign(cf_w, cand, N, returnIndices=True, resident=resident)
        b = ed.performGreedyIVARExperimentalDesign(cf_s, cand, N, returnIndices=True, resident=resident)
        assert np.array_equal(a, b), resident
        assert _rel(cf_w.lastScores, cf_s.lastScores) <= 1e-12, resident


@pytest.mark.gpu
def test_reference_optimiser_loop_reads_mc_weights(env):
    """With the reference staged: mcWeights set on the reference's own costFunctionGP_IVAR changes evaluate and the end
    design of its SLSQP loop (ExperimentalDesignDerivative.begin)."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(root, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        pytest.skip("no reference package available (set GPEXP_REFERENCE and run __graft_entry__.build() to stage it)")
    import contextlib
    import io
    import gpexp_b200
    gpexp_b200.install_as_gpExp(path)
    try:
        import gpExp.approximation as rap
        import gpExp.experimentalDesign as red
        import gpExp.gp as rgp
        import gpExp.kernels as rk
        red.VERBOSE = False
        rng = np.random.default_rng(61)
        mc = rng.uniform(-1, 1, (2000, 2))
        k = rk.KernelSquaredExponential([0.3, 0.45], 1.7, 2)
        dens = lambda p: np.all(np.abs(p) <= 1.0, axis=1).astype(float)  # noqa: E731
        space = rap.Space(2, None, dens, noise=None)
        start = red.performGreedyVarExperimentalDesign(k, mc, 4, 2)
        ends = []
        for w in (None, np.where(mc[:, 0] > 0.3, 1.0 / 2000, 0.0)):
            cf = red.costFunctionGP_IVAR(rgp.GP(k, 1e-6), 4, space, mcPoints=mc)
            if w is not None:
                cf.mcWeights = w
            val = cf.evaluate(start)
            exp = red.ExperimentalDesignDerivative(cf, 4, 2)
            with contextlib.redirect_stdout(io.StringIO()):
                end = exp.begin([start], list(-np.ones(8)), list(np.ones(8)))
            ends.append((val, np.asarray(end)))
        assert ends[0][0] != ends[1][0]
        assert np.max(np.abs(ends[0][1] - ends[1][1])) > 1e-3
    finally:
        for name in [m for m in list(sys.modules) if m == "gpExp" or m.startswith("gpExp.")]:
            del sys.modules[name]


@pytest.mark.gpu
def test_cfg2_size_additivity_and_uniform_weights(env):
    """100 000 candidates, n = 255 through scoreCandidatesIVAR: the weighted cost is additive over a ragged split of the
    100 000 integration points (each part with its own weights); with M = 2^17 points, w = 1/M reproduces the unweighted
    costs bit for bit."""
    ed = env.ed
    rng = np.random.default_rng(62)
    k = product_kernel("se_ard_2d")
    cand, design = rng.uniform(-1, 1, (100_000, 2)), rng.uniform(-1, 1, (255, 2))
    mc = rng.uniform(-1, 1, (100_000, 2))
    w = _weights("smooth", mc, rng)

    def costs(points, weights):
        cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 255, env.Space(2, None, None), mcPoints=points, mcWeights=weights)
        return ed.scoreCandidatesIVAR(cf, design, cand)[0]

    whole = costs(mc, w)
    cut = [0, 31_337, 77_000, 100_000]
    # |base - red| with base > red: the cost is additive in base - red over the parts
    parts = sum(costs(mc[a:b], w[a:b]) for a, b in zip(cut[:-1], cut[1:]))
    assert _rel(parts, whole) <= 1e-11
    mc2 = rng.uniform(-1, 1, (2 ** 17, 2))
    u = costs(mc2, None)
    v = costs(mc2, np.full(2 ** 17, 2.0 ** -17))
    assert np.array_equal(u, v)
