"""Greedy mutual information under a per-point noise nu (gp.noise as an ndarray, one value per pool point): each subset's
Gram takes diag(nu) on that subset, so the numerator is var(y | A) with K_AA + diag nu_A and the denominator is
1/[(K_SS + diag nu_S)^-1]_yy - nu_y.  The engines factor K_VV + diag nu, divide the append by sqrt(num_p + nu_p) and
score with 1/pd_j - nu_j.

The oracles are oracle/gpexp_oracle.py's ref_greedy_mi, ref_mi_cost and fast_greedy_mi with a nu vector.
CPU: the vectorised oracle against the reference's pinv loop with nu on each subset; both oracles with a constant nu
against the float-noise oracles, bit for bit; rejected noise vectors.
GPU: a constant nu reproduces the scalar run bit for bit on the golden cases; a varying nu against the reference's loop
(picks, scores, evaluate, pivots); the cfg-4 kernel at |V| = 700 and 3 000 against the vectorised oracle; a noise profile
changes the design; changing gp.noise rebuilds the cached factorisation; the dense and the one-rank sharded engines agree.

Score tolerance: 2e-8 relative, the bound test_greedy_mi_golden uses for the reference's pinv round-off and the
1/P_yy - nu_y cancellation.  The profiles below keep nu_y below about ten times the denominator, so the cancellation
costs at most one decimal digit of the 1e-13-level accuracy of 1/P_yy (measured: at most 1e-9 on the CPU cases)."""
import functools

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests.cases import product_kernel, spec

SCORE_RTOL = 2e-8
SE_CL, SE_SIGNAL = [0.15, 0.2], 1.0   # the noise-free half of a 100-point pool has cond(K) ~ 3e4 (DESIGN section 2: <~ 1e6)


def kernel_spec(name):
    return orc.KernelSpec.se(SE_CL, SE_SIGNAL, 2) if name == "se_mid" else spec(name)


def kernel_obj(name):
    if name == "se_mid":
        from gpexp_b200 import kernels
        return kernels.KernelSquaredExponential(list(SE_CL), SE_SIGNAL, 2)
    return product_kernel(name)


# ---- noise profiles: one value per pool point ----------------------------------------------------------------------------
def nu_span(p):
    """1e-6 at x0 = -1 to 1e-3 at x0 = 1: three orders of magnitude."""
    return 1e-6 * 1e3 ** np.clip((p[:, 0] + 1.0) / 2.0, 0.0, 1.0)


def nu_half_zero(p):
    """Exactly 0 for x0 < 0."""
    return np.where(p[:, 0] < 0.0, 0.0, 1e-4 + 1e-3 * p[:, 0] ** 2)


def nu_const(p):
    return np.full(p.shape[0], 1e-3)


def nu_mehler_span(p):
    """1e-2 at x0 <= -2 to 10 at x0 >= 2 (a noise-free Mehler Gram is singular: no zero profile here)."""
    return 1e-2 * 1e3 ** np.clip((p[:, 0] + 2.0) / 4.0, 0.0, 1.0)


def nu_mehler_const(p):
    return np.full(p.shape[0], 1e-2)


def nu_cfg4(p):
    """cfg-4's noise level 1e-2 at the origin, growing with the distance from it."""
    return 1e-2 * (1.0 + np.sum(p * p, axis=1) / 3.0)


def nu_steep(p):
    """Large enough at |x0| ~ 1 to move the SE design away from the scalar-noise one."""
    return 1e-3 + 0.3 * p[:, 0] ** 2


def _pool(name, rng, v):
    d = kernel_spec(name).dim
    return rng.standard_normal((v, d)) if name.startswith("mehler") else rng.uniform(-1, 1, (v, d))


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.abs(np.asarray(b))))


CPU_CASES = [("se_mid", nu_span), ("se_mid", nu_half_zero), ("se_mid", nu_const),
             ("matern_5d", nu_span), ("matern_5d", nu_half_zero), ("matern_5d", nu_const),
             ("mehler_3d", nu_mehler_span), ("mehler_3d", nu_mehler_const)]
V_REF, N_REF, START = 100, 8, 3


@functools.lru_cache(maxsize=None)
def _reference_run(name, nu):
    """|V| = 100, 8 picks of the reference's pinv loop (a few seconds each)."""
    pool = _pool(name, np.random.default_rng(41), V_REF)
    idx, scores, opts = orc.ref_greedy_mi(kernel_spec(name), pool, nu(pool), N_REF, start=START)
    return pool, idx, scores, opts


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,nu", CPU_CASES, ids=[f"{n}-{f.__name__}" for n, f in CPU_CASES])
def test_fast_oracle_with_noise_vector_equals_reference_loop(name, nu):
    pool, ref_idx, ref_scores, opts = _reference_run(name, nu)
    idx, scores, pivots = orc.fast_greedy_mi(kernel_spec(name), pool, nu(pool), N_REF, start=START, with_pivots=True)
    assert idx == ref_idx
    for s in range(N_REF - 1):
        assert _rel(scores[s][opts[s]], ref_scores[s]) <= SCORE_RTOL, s
    assert np.isinf(scores[0][START]) and len(pivots) == N_REF


def test_constant_noise_oracles_are_the_float_oracles():
    """With nu = s2 everywhere, the noise-vector forms of both MI oracles reproduce their float-noise forms bit for bit."""
    ks, s2 = spec("matern_5d"), 1e-3
    pool = np.random.default_rng(42).uniform(-1, 1, (60, 5))
    nu = np.full(60, s2)
    a_idx, a_scores, a_opts = orc.ref_greedy_mi(ks, pool, s2, 6, start=2)
    b_idx, b_scores, b_opts = orc.ref_greedy_mi(ks, pool, nu, 6, start=2)
    assert a_idx == b_idx and all(np.array_equal(a, b) for a, b in zip(a_scores, b_scores))
    assert all(np.array_equal(a, b) for a, b in zip(a_opts, b_opts))
    f_idx, f_scores = orc.fast_greedy_mi(ks, pool, s2, 6, start=2)
    g_idx, g_scores = orc.fast_greedy_mi(ks, pool, nu, 6, start=2)
    assert f_idx == g_idx == a_idx and all(np.array_equal(a, b) for a, b in zip(f_scores, g_scores))


BAD = [(lambda v: np.full(v + 1, 1e-3), "values for"),
       (lambda v: np.where(np.arange(v) == 7, np.nan, 1e-3), "not finite"),
       (lambda v: np.where(np.arange(v) == 7, -1e-8, 1e-3), "negative")]


@pytest.mark.parametrize("bad,what", BAD, ids=["length", "nan", "negative"])
def test_bad_pool_noise_is_rejected(bad, what):
    """The checks run before any device work.  The cost function is assembled by hand because its constructor factors
    the pool's Gram on the device."""
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    pool = np.random.default_rng(43).uniform(-1, 1, (50, 2))
    cf = ed.costFunctionGP_MI.__new__(ed.costFunctionGP_MI)
    cf.gaussianProcess, cf.mcPoints, cf.nMC = gpmod.GP(kernel_obj("se_mid"), bad(50)), pool, 50
    with pytest.raises(ValueError, match=what):
        ed.performGreedyMIExperimentalDesign(cf, 4)
    with pytest.raises(ValueError, match=what):
        ed.performGreedyMIExperimentalDesign(cf, 4, shard=object())
    with pytest.raises(ValueError, match=what):
        cf.evaluate(0, [1, 2])


def test_engine_noise_vector_contract():
    """pool_noise replaces the scalar noise and has one value per pool point (checked before any device work)."""
    from gpexp_b200.engine import ShardedMIEngine
    pool = np.random.default_rng(44).uniform(-1, 1, (50, 2))
    with pytest.raises(ValueError, match="replaces the scalar noise"):
        ShardedMIEngine(None, pool, 4, 1e-3, pool_noise=np.full(50, 1e-3))
    with pytest.raises(ValueError, match="49 values for 50 pool points"):
        ShardedMIEngine(None, pool, 4, 0.0, pool_noise=np.full(49, 1e-3))


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import engine
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    ed.VERBOSE = False

    class NS:
        pass
    ns = NS()
    ns.ed, ns.engine, ns.gp, ns.Space = ed, engine, gpmod, Space
    ns.dev = Device.get(0)
    return ns


def _cost_function(env, name, pool, noise):
    k = kernel_obj(name)
    return env.ed.costFunctionGP_MI(env.gp.GP(k, noise), 1, env.Space(k.dimension, None, None), nmc=len(pool),
                                    mcpoints=pool)


def _trace(eng, n, start):
    eng.score_trace = []
    idx = eng.run(n, start=start)
    return [int(i) for i in idx], eng.score_trace


@pytest.mark.gpu
def test_constant_noise_vector_is_the_scalar_run_bit_for_bit(env, golden):
    """nu = s2 * 1 on the golden greedy_mi cases: picks, score traces, pivots and evaluate values of the scalar run, through
    the public driver and both engines (the same addition in the same place)."""
    z = golden("greedy_mi")
    cases = sorted({k.split("/")[1] for k in z.files if k.startswith("gmi/")})
    for ci in cases:
        name = str(z[f"gmi/{ci}/name"])
        pool, noise, start = z[f"gmi/{ci}/pool"], float(z[f"gmi/{ci}/noise"]), int(z[f"gmi/{ci}/start"])
        idx = [int(i) for i in z[f"gmi/{ci}/idx"]]
        n, nu = len(idx), np.full(len(pool), noise)
        cf_s, cf_v = _cost_function(env, name, pool, noise), _cost_function(env, name, pool, nu)
        pts = env.ed.performGreedyMIExperimentalDesign(cf_v, n, start=start)
        env.ed.performGreedyMIExperimentalDesign(cf_s, n, start=start)
        assert [int(i) for i in cf_v.lastIndices] == [int(i) for i in cf_s.lastIndices] == idx, (ci, name)
        assert np.array_equal(pts, pool[idx])
        assert np.array_equal(cf_v.lastEngine.pivots(), cf_s.lastEngine.pivots())
        # the sharded engine behind the driver, and the dense engine
        a_idx, a_tr = _trace(env.ed._mi_new_engine(cf_s, n), n, start)
        b_idx, b_tr = _trace(env.ed._mi_new_engine(cf_v, n), n, start)
        kernel_obj(name)._bind(env.dev)
        pts_dev = env.dev.points(pool)
        c_idx, c_tr = _trace(env.engine.GreedyMIEngine(env.dev, pts_dev, n, noise), n, start)
        d_eng = env.engine.GreedyMIEngine(env.dev, pts_dev, n, 0.0, pool_noise=nu)
        d_idx, d_tr = _trace(d_eng, n, start)
        assert a_idx == b_idx == c_idx == d_idx == idx
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(a_tr, b_tr)), (ci, name)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(c_tr, d_tr)), (ci, name)
        for j in np.flatnonzero(np.isfinite(z[f"gmi/{ci}/scores"][2]))[:5]:
            assert np.array_equal(cf_v.evaluate(int(j), idx[:2]), cf_s.evaluate(int(j), idx[:2])), (ci, j)


GPU_CASES = [("se_mid", nu_span), ("se_mid", nu_half_zero), ("matern_5d", nu_span), ("matern_5d", nu_half_zero),
             ("mehler_3d", nu_mehler_span)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,nu", GPU_CASES, ids=[f"{n}-{f.__name__}" for n, f in GPU_CASES])
def test_varying_noise_matches_reference_loop(env, name, nu):
    pool, ref_idx, ref_scores, opts = _reference_run(name, nu)
    ks, nuv = kernel_spec(name), nu(pool)
    cf = _cost_function(env, name, pool, nuv)
    pts = env.ed.performGreedyMIExperimentalDesign(cf, N_REF, start=START)
    assert [int(i) for i in cf.lastIndices] == ref_idx
    assert np.array_equal(pts, pool[ref_idx])
    # pivots: num_p + nu_p, the prior variance given the picks before p plus nu_p
    piv = cf.lastEngine.pivots()
    for s, p in enumerate(ref_idx):
        var = ks.prior(pool[p:p + 1])[0] if s == 0 else \
            orc.fast_posterior_variance(ks, pool[ref_idx[:s]], pool[p:p + 1], nuv[ref_idx[:s]])[0]
        assert abs(piv[s] - (var + nuv[p])) <= 1e-12 * orc.kern_scale(ks), s
    # every step's scores
    got_idx, trace = _trace(env.ed._mi_new_engine(cf, N_REF), N_REF, START)
    assert got_idx == ref_idx
    for s, sc in enumerate(trace):
        assert _rel(sc[opts[s]], ref_scores[s]) <= SCORE_RTOL, s
    # the single-candidate call against the restated reference cost
    for j in opts[3][::17]:
        want = orc.ref_mi_cost(ks, pool, nuv, int(j), ref_idx[:3])[0]
        got = cf.evaluate(int(j), ref_idx[:3])
        assert got.shape == (1,) and abs(got[0] - want) <= SCORE_RTOL * abs(want), j


@pytest.mark.gpu
@pytest.mark.parametrize("v,n", [(700, 12), (3000, 24)])
def test_cfg4_kernel_matches_fast_oracle(env, v, n):
    """cfg-4's kernel (3-D Mehler t = 0.9, N(0, I) pool) with nu(x) = 1e-2 (1 + |x|^2 / 3)."""
    pool = np.random.default_rng(4).standard_normal((v, 3))
    nu = nu_cfg4(pool)
    ref, _, ref_piv = orc.fast_greedy_mi(spec("mehler_3d"), pool, nu, n, start=0, with_pivots=True)
    cf = _cost_function(env, "mehler_3d", pool, nu)
    env.ed.performGreedyMIExperimentalDesign(cf, n, start=0)
    assert [int(i) for i in cf.lastIndices] == ref
    assert int(cf.lastEngine.info.item()) == 0
    assert np.max(np.abs(cf.lastEngine.pivots() - ref_piv)) <= 1e-12 * max(ref_piv)


@pytest.mark.gpu
def test_noise_profile_changes_the_design(env):
    pool = _pool("se_mid", np.random.default_rng(41), V_REF)
    nu = nu_steep(pool)
    ref, _ = orc.fast_greedy_mi(kernel_spec("se_mid"), pool, nu, N_REF, start=START)
    scalar = _cost_function(env, "se_mid", pool, 1e-3)
    hetero = _cost_function(env, "se_mid", pool, nu)
    env.ed.performGreedyMIExperimentalDesign(scalar, N_REF, start=START)
    env.ed.performGreedyMIExperimentalDesign(hetero, N_REF, start=START)
    assert [int(i) for i in hetero.lastIndices] == ref
    assert [int(i) for i in hetero.lastIndices] != [int(i) for i in scalar.lastIndices]


@pytest.mark.gpu
def test_changing_noise_rebuilds_the_factorisation(env):
    """The evaluate cache is keyed on the bytes of nu: a new array and an in-place change both rebuild."""
    name = "matern_5d"
    pool = _pool(name, np.random.default_rng(45), 80)
    ks = kernel_spec(name)
    added, js = [5, 17], [0, 33, 79]
    cf = _cost_function(env, name, pool, nu_span(pool))

    def check(nu):
        got = np.array([cf.evaluate(j, added)[0] for j in js])
        want = np.array([orc.ref_mi_cost(ks, pool, nu, j, added)[0] for j in js])
        assert _rel(got, want) <= SCORE_RTOL
        return got, cf._mi_cache["engine"]   # the object, not its id(): a freed engine's id can be reused

    a, ea = check(nu_span(pool))
    cf.gaussianProcess.noise = nu_steep(pool)
    b, eb = check(nu_steep(pool))
    cf.gaussianProcess.noise[:] = nu_half_zero(pool)
    c, ec = check(nu_half_zero(pool))
    assert ea is not eb and eb is not ec
    assert np.all(a != b) and np.all(b != c)


@pytest.mark.gpu
@pytest.mark.parametrize("v,blk", [(700, None), (1100, 256)])
def test_dense_and_sharded_engines_agree(env, monkeypatch, v, blk):
    """As test_sharded_mi_engine_single_rank_equals_dense_engine for scalar noise; |V| = 1 100 with GPX_MI_BLK = 256 ends in
    a partial distribution block."""
    if blk is not None:
        monkeypatch.setenv("GPX_MI_BLK", str(blk))
    name, n = "mehler_3d", 10
    pool = _pool(name, np.random.default_rng(46), v)
    nu = nu_mehler_span(pool)
    ref, ref_scores, ref_piv = orc.fast_greedy_mi(spec(name), pool, nu, n, start=2, with_pivots=True)
    kernel_obj(name)._bind(env.dev)
    sharded = env.engine.ShardedMIEngine(env.dev, pool, n, 0.0, pool_noise=nu)
    dense = env.engine.GreedyMIEngine(env.dev, env.dev.points(pool), n, 0.0, pool_noise=nu)
    if blk is not None:
        assert sharded.BLK == blk and v % blk != 0
    for eng in (sharded, dense):
        idx, trace = _trace(eng, n, 2)
        assert int(eng.info.item()) == 0
        assert idx == ref, type(eng).__name__
        for s, sc in enumerate(trace):
            ok = np.isfinite(ref_scores[s])
            assert _rel(sc[ok], ref_scores[s][ok]) <= 1e-8, (type(eng).__name__, s)
        assert np.max(np.abs(eng.pivots() - ref_piv)) <= 1e-12 * max(ref_piv)
