"""GPU parity tests: the CUDA path (through the Python API -> ctypes -> C ABI) against
(1) golden vectors produced by the unmodified reference (tests/golden/*.npz),
(2) the CPU oracle (oracle/gpexp_oracle.py) at sizes the reference cannot reach,
(3) size-independent properties (factor reconstruction, round trips, tie-breaking).

Tolerances: indices identical; scores / variances within 1e-9 relative (north star), widened only
where the reference's own pinv round-off is larger (cond * eps, SURVEY.md section 7) -- written at each use.
"""
import ctypes as C

import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from oracle import gpexp_oracle as orc
from tests.cases import KERNEL_NAMES, product_kernel, spec

pytestmark = pytest.mark.gpu

EPS = 2.220446049250313e-16
# relative accuracy of one covariance value: exp(-x) carries |x| * eps of argument round-off and the test
# inputs reach |x| ~ 800 (cl = 0.06 on [-1,1]^2), so a few 1e-13; FMA contraction differs from numpy too
RTOL_K = 2e-12


def keys(z, prefix):
    return sorted({k.split("/")[1] for k in z.files if k.startswith(prefix + "/")})


@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    ed.VERBOSE = False
    from gpexp_b200 import _lib, device, engine
    from gpexp_b200 import gp as gpmod
    from gpexp_b200 import gp_kernel_utilities as gku
    from gpexp_b200.approximation import Space

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ed, ns.lib, ns._lib, ns.device, ns.engine, ns.gp, ns.gku, ns.Space = \
        torch, ed, _lib.lib, _lib, device, engine, gpmod, gku, Space
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    return ns


def bind(gx, name):
    k = product_kernel(name)
    k._bind(gx.dev)
    return k


# ------------------------------------------------------------------------------------------------
# golden vectors of the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", KERNEL_NAMES)
def test_kernel_pairwise_golden(gx, golden, name):
    z = golden("kernels")
    k = product_kernel(name)
    x1, x2, one = z[f"kern/{name}/x1"], z[f"kern/{name}/x2"], z[f"kern/{name}/one"]
    np.testing.assert_allclose(k.evaluate(x1, x2), z[f"kern/{name}/pair"], rtol=RTOL_K, atol=1e-300)
    np.testing.assert_allclose(k.evaluate(x1, one), z[f"kern/{name}/bcast_right"], rtol=RTOL_K, atol=1e-300)
    np.testing.assert_allclose(k.evaluate(one, x2), z[f"kern/{name}/bcast_left"], rtol=RTOL_K, atol=1e-300)
    np.testing.assert_allclose(k.evaluate(x1, x1), z[f"kern/{name}/prior"], rtol=RTOL_K)
    with pytest.raises(AssertionError):
        k.evaluate(x1[:, :0], x2)
    with pytest.raises(AssertionError):
        k.evaluate(x1[:5], x2[:7])


def test_gram_golden(gx, golden):
    z = golden("gram")
    for name in keys(z, "gram"):
        k = product_kernel(name)
        pts, nug = z[f"gram/{name}/pts"], z[f"gram/{name}/nugvec"]
        np.testing.assert_allclose(gx.gku.calculateCovarianceMatrix(k, pts), z[f"gram/{name}/K0"], rtol=RTOL_K, atol=1e-300)
        np.testing.assert_allclose(gx.gku.calculateCovarianceMatrix(k, pts, 1e-3), z[f"gram/{name}/Kscalar"], rtol=RTOL_K, atol=1e-300)
        np.testing.assert_allclose(gx.gku.calculateCovarianceMatrix(k, pts, nug), z[f"gram/{name}/Kvec"], rtol=RTOL_K, atol=1e-300)
        with pytest.raises(NameError):
            gx.gku.calculateCovarianceMatrix(k, pts, 1)


def test_gp_golden(gx, golden):
    z = golden("gp")
    for name in [n for n in keys(z, "gp") if n != "hetero"]:
        k = product_kernel(name)
        nodes, query = z[f"gp/{name}/nodes"], z[f"gp/{name}/query"]
        noise, cond = float(z[f"gp/{name}/noise"]), float(z[f"gp/{name}/cond"])
        # Cholesky vs the reference's pinv agree to ~cond*eps (SURVEY.md section 7); never tighter than 1e-9
        tol = max(1e-9, 50 * cond * EPS)
        g = gx.gp.GP(k, noise)
        g.train(nodes, z[f"gp/{name}/fvals"])
        scale = float(np.max(np.abs(z[f"gp/{name}/absvar"])) + np.max(np.abs(z[f"gp/{name}/cov"])))
        np.testing.assert_allclose(g.covarianceMatrix, z[f"gp/{name}/cov"], rtol=RTOL_K, atol=1e-300)
        var = g.evaluateVariance(query, parallel=0)
        assert np.max(np.abs(var - z[f"gp/{name}/var"])) <= tol * scale, name
        mean, absvar = g.evaluate(query, compvar=1)
        assert np.max(np.abs(absvar - z[f"gp/{name}/absvar"])) <= tol * scale
        mscale = np.max(np.abs(z[f"gp/{name}/mean"]))
        assert np.max(np.abs(mean - z[f"gp/{name}/mean"])) <= tol * mscale * 10
        mean2, cov = g.evaluate(query[:25], compvar=2)
        assert np.max(np.abs(cov - z[f"gp/{name}/cov25"])) <= tol * scale
        np.testing.assert_allclose(mean2, mean[:25], rtol=1e-12, atol=1e-12 * mscale)
        cscale = np.max(np.abs(z[f"gp/{name}/coeff"]))
        assert np.max(np.abs(g.coeff - z[f"gp/{name}/coeff"])) <= tol * cscale * 10
        prec = g.precisionMatrix
        assert np.max(np.abs(prec - z[f"gp/{name}/prec"])) <= tol * np.max(np.abs(z[f"gp/{name}/prec"])) * 10
        space = gx.Space(k.dimension, None, None, noise=None)
        cf = gx.ed.costFunctionGP_IVAR(g, nodes.shape[0], space, mcPoints=z[f"gp/{name}/mc"])
        ref_cost = float(z[f"gp/{name}/ivar_cost"])
        assert abs(cf.evaluate(nodes) - ref_cost) <= tol * max(ref_cost, 1e-3), name
        with pytest.raises(AssertionError):
            cf.evaluate(nodes[:-1])
    # heteroscedastic branch (experimentalDesign.py:110-114)
    k = product_kernel("se_ard_2d_wide")
    nodes, mc = z["gp/hetero/nodes"], z["gp/hetero/mc"]
    space = gx.Space(2, None, None, noise=lambda p: 1e-4 + 1e-3 * (p[:, 0] ** 2))
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 25, space, mcPoints=mc)
    got = cf.evaluate(nodes)
    assert abs(got - float(z["gp/hetero/ivar_cost"])) <= 1e-9 * got


def _trace_var(gx, name, pool, n, weights, seeds):
    k = bind(gx, name)
    p = gx.dev.points(pool)
    eng = gx.engine.GreedyVarEngine(gx.dev, p, n, weights=weights)
    eng.score_trace = []
    for s in seeds:
        eng.force(int(s))
    idx = eng.run(n)
    return idx, eng.score_trace


def test_greedy_var_golden(gx, golden):
    z = golden("greedy_var")
    for ci in keys(z, "gvar"):
        name = str(z[f"gvar/{ci}/name"])
        pool, idx, ref_scores = z[f"gvar/{ci}/pool"], z[f"gvar/{ci}/idx"], z[f"gvar/{ci}/scores"]
        w = z[f"gvar/{ci}/weights"]
        w = w if w.size else None
        seeds = [int(s) for s in z[f"gvar/{ci}/seeds"]]
        # public API: returns points, mutates the seed list in place (experimentalDesign.py:808,845)
        keep = list(seeds)
        pts = gx.ed.performGreedyVarExperimentalDesign(product_kernel(name), pool, len(idx), pool.shape[1], weights=w,
                                                       indKeepStart=keep)
        assert np.array_equal(pts, pool[idx]), (ci, name)
        if seeds:
            assert keep == [int(i) for i in idx]
        got_idx, trace = _trace_var(gx, name, pool, len(idx), w, seeds)
        assert [int(i) for i in got_idx] == [int(i) for i in idx]
        for s, sc in enumerate(trace):
            ref = ref_scores[len(seeds) + s]
            # 1e-9 of the score scale: entries at already-selected points are +-1e-16 round-off in the reference
            assert np.max(np.abs(sc - ref)) <= 1e-9 * np.max(np.abs(ref)), (ci, s)


def test_greedy_ivar_golden(gx, golden):
    z = golden("greedy_ivar")
    for ci in keys(z, "givar"):
        name = str(z[f"givar/{ci}/name"])
        k = product_kernel(name)
        cand, mc, noise = z[f"givar/{ci}/cand"], z[f"givar/{ci}/mc"], float(z[f"givar/{ci}/noise"])
        idx, ref_costs = z[f"givar/{ci}/idx"], z[f"givar/{ci}/costs"]
        space = gx.Space(k.dimension, None, None, noise=None)
        cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, space, mcPoints=mc)
        pts = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, len(idx))
        assert [int(i) for i in cf.lastIndices] == [int(i) for i in idx], (ci, name)
        assert np.array_equal(pts, cand[idx])
        # per-step cost vectors
        fam, d, params = k._gpx_spec()
        eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), len(idx), noise,
                                         gx.engine.prior_scale(fam, params))
        eng.score_trace = []
        eng.run(len(idx))
        for s, c in enumerate(eng.score_trace):
            err = np.max(np.abs(c - ref_costs[s]) / np.abs(ref_costs[s]))
            assert err <= 1e-9, (ci, name, s, err)   # north-star tolerance
        # stateless scoring from host buffers reproduces the same step
        costs, best = gx.ed.scoreCandidatesIVAR(cf, cand[idx[:3]], cand)
        assert best == int(idx[3])
        assert np.max(np.abs(costs - ref_costs[3]) / np.abs(ref_costs[3])) <= 1e-9


def test_greedy_mi_golden(gx, golden):
    z = golden("greedy_mi")
    for ci in keys(z, "gmi"):
        name = str(z[f"gmi/{ci}/name"])
        k = product_kernel(name)
        pool, noise, start = z[f"gmi/{ci}/pool"], float(z[f"gmi/{ci}/noise"]), int(z[f"gmi/{ci}/start"])
        idx, ref_scores = z[f"gmi/{ci}/idx"], z[f"gmi/{ci}/scores"]
        space = gx.Space(k.dimension, None, None, noise=None)
        cf = gx.ed.costFunctionGP_MI(gx.gp.GP(k, noise), len(idx), space, nmc=len(pool), mcpoints=pool)
        pts = gx.ed.performGreedyMIExperimentalDesign(cf, len(idx), start=start)
        assert [int(i) for i in cf.lastIndices] == [int(i) for i in idx], (ci, name)
        assert np.array_equal(pts, pool[idx])
        eng = gx.ed._mi_new_engine(cf, len(idx))
        eng.score_trace = []
        eng.run(len(idx), start=start)
        for s, sc in enumerate(eng.score_trace):
            ref = ref_scores[s + 1]
            ok = np.isfinite(ref)
            assert np.array_equal(ok, np.isfinite(sc))
            err = np.max(np.abs(sc[ok] - ref[ok]) / np.abs(ref[ok]))
            # the reference's own 1/P_yy - noise cancellation + pinv round-off (SURVEY.md 3.3): 2e-8
            assert err <= 2e-8, (ci, s, err)
        # single-candidate API, shape (1,) like the reference
        j = int(np.flatnonzero(np.isfinite(ref_scores[2]))[3])
        one = cf.evaluate(j, [int(i) for i in idx[:2]])
        assert one.shape == (1,)
        assert abs(one[0] - ref_scores[2][j]) <= 2e-8 * abs(ref_scores[2][j])
        np.testing.assert_allclose(cf.cov, z[f"gmi/{ci}/cov"], rtol=RTOL_K)


# ------------------------------------------------------------------------------------------------
# linear algebra building blocks against numpy / scipy
# ------------------------------------------------------------------------------------------------
def _spd(rng, n):
    a = rng.standard_normal((n, n + 5))
    return a @ a.T / (n + 5) + 0.5 * np.eye(n)


@pytest.mark.parametrize("n", [1, 5, 32, 45, 128, 129, 300, 515])
def test_potrf_trsm_blocks(gx, n):
    from scipy.linalg import solve_triangular
    rng = np.random.default_rng(n)
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    A = _spd(rng, n)
    ld = gx.device.roundup(n)
    Ad = dev.zeros(n, ld)
    Ad[:, :n] = dev.upload(A)
    info = dev.zeros(1, dtype=gx.torch.int32)
    gx.check(lib.gpx_potrf(dev.h, ptr(Ad), n, ld, ptr(info), dev.stream))
    assert int(info.item()) == 0
    U = np.triu(Ad[:, :n].cpu().numpy())
    Uref = np.linalg.cholesky(A).T
    np.testing.assert_allclose(U, Uref, rtol=1e-11, atol=1e-12)
    # forward solve with a materialised right-hand side, ragged column count
    m = 77
    B = rng.standard_normal((n, m))
    ldb = gx.device.roundup(m)
    Bd = dev.zeros(n, ldb)
    Bd[:, :m] = dev.upload(B)
    gx.check(lib.gpx_trsm(dev.h, ptr(Ad), n, ld, ptr(Bd), m, ldb, dev.stream))
    X = solve_triangular(Uref, B, trans='T', lower=False)
    np.testing.assert_allclose(Bd[:, :m].cpu().numpy(), X, rtol=1e-9, atol=1e-10)
    # back solve needs U^T
    Ut = dev.zeros(n, ld)
    gx.check(lib.gpx_transpose(dev.h, ptr(Ad), n, n, ld, ptr(Ut), ld, dev.stream))
    gx.check(lib.gpx_trsm_back(dev.h, ptr(Ut), n, ld, ptr(Bd), m, ldb, dev.stream))
    np.testing.assert_allclose(Bd[:, :m].cpu().numpy(), np.linalg.solve(A, B), rtol=1e-8, atol=1e-9)
    # explicit U^-T, lower triangular with exact zeros above the diagonal
    Y = dev.zeros(n, ld)
    gx.check(lib.gpx_trtri_t(dev.h, ptr(Ad), n, ld, ptr(Y), ld, dev.stream))
    Yh = Y[:, :n].cpu().numpy()
    assert np.all(np.triu(Yh, 1) == 0.0)
    np.testing.assert_allclose(Yh, np.linalg.inv(Uref).T, rtol=1e-8, atol=1e-9)
    # a column of the precision from Y
    p = dev.upload(np.array([n // 2], dtype=np.int64), dtype=gx.torch.int64)
    col = dev.zeros(ld)
    ws = dev.zeros(max(int(lib.gpx_mi_prec_column_workspace(n, ld)), 1))
    gx.check(lib.gpx_mi_prec_column(dev.h, ptr(Y), n, n, ld, 0, 0, 1, ptr(p), None, ptr(ws), ptr(col), dev.stream))
    np.testing.assert_allclose(col[:n].cpu().numpy(), np.linalg.inv(A)[:, n // 2], rtol=1e-7, atol=1e-9)
    # rank-1 append reproduces the factor of the bordered matrix
    if n >= 2:
        Ud = dev.zeros(n, ld)
        Ud[: n - 1, : n - 1] = dev.upload(np.linalg.cholesky(A[: n - 1, : n - 1]).T.copy())
        knew = dev.upload(A[: n - 1, n - 1].copy())
        gx.check(lib.gpx_chol_append(dev.h, ptr(Ud), n - 1, ld, ptr(knew), float(A[n - 1, n - 1]), ptr(info), dev.stream))
        assert int(info.item()) == 0
        np.testing.assert_allclose(np.triu(Ud[:, :n].cpu().numpy()), Uref, rtol=1e-10, atol=1e-11)


def test_potrf_reports_failing_pivot(gx):
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    n, ld = 200, 256
    A = np.eye(n)
    A[150, 150] = -1.0
    Ad = dev.zeros(n, ld)
    Ad[:, :n] = dev.upload(A)
    info = dev.zeros(1, dtype=gx.torch.int32)
    gx.check(lib.gpx_potrf(dev.h, ptr(Ad), n, ld, ptr(info), dev.stream))
    assert int(info.item()) == 151


@pytest.mark.parametrize("shape", [(1, 1, 1), (3, 130, 5), (129, 257, 33), (260, 131, 200), (128, 128, 16)])
def test_dgemm_tn_sub(gx, shape):
    I, J, K = shape
    rng = np.random.default_rng(I * 1000 + J)
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    A, B, Cm = rng.standard_normal((K, I)), rng.standard_normal((K, J)), rng.standard_normal((I, J))
    lda, ldb, ldc = gx.device.roundup(I), gx.device.roundup(J), gx.device.roundup(J)
    Ad, Bd, Cd = dev.zeros(K, lda), dev.zeros(K, ldb), dev.zeros(I, ldc)
    Ad[:, :I], Bd[:, :J], Cd[:, :J] = dev.upload(A), dev.upload(B), dev.upload(Cm)
    gx.check(lib.gpx_dgemm_tn_sub(dev.h, ptr(Ad), lda, ptr(Bd), ldb, ptr(Cd), ldc, I, J, K, 0, dev.stream))
    np.testing.assert_allclose(Cd[:, :J].cpu().numpy(), Cm - A.T @ B, rtol=1e-12, atol=1e-12)
    assert np.all(Cd[:, J:].cpu().numpy() == 0.0)  # padding untouched


def test_argreduce_and_sum(gx):
    dev, lib, ptr, torch = gx.dev, gx.lib, gx.ptr, gx.torch
    rng = np.random.default_rng(7)
    best, idx, tot = dev.zeros(1), dev.zeros(1, dtype=torch.int64), dev.zeros(1)
    for n in [1, 2, 255, 256, 1025, 70001, 3_000_000]:
        v = rng.standard_normal(n)
        # plant exact ties at the extremes: numpy returns the first
        if n > 10:
            v[[n // 3, n // 2, n - 1]] = v.max() + 1.0
            v[[n // 5, n // 4]] = v.min() - 1.0
        vd = dev.upload(v)
        gx.check(lib.gpx_argreduce(dev.h, ptr(vd), None, None, n, 0, ptr(best), ptr(idx), dev.stream))
        assert int(idx.item()) == int(np.argmax(v)) and best.item() == v.max()
        gx.check(lib.gpx_argreduce(dev.h, ptr(vd), None, None, n, 1, ptr(best), ptr(idx), dev.stream))
        assert int(idx.item()) == int(np.argmin(v)) and best.item() == v.min()
        w = rng.uniform(0.5, 1.5, n)
        mask = (rng.uniform(size=n) < 0.3).astype(np.uint8)
        if mask.all():
            mask[0] = 0
        gx.check(lib.gpx_argreduce(dev.h, ptr(vd), ptr(dev.upload(w)), ptr(dev.upload(mask, dtype=torch.uint8)), n, 0,
                                   ptr(best), ptr(idx), dev.stream))
        s = np.where(mask == 0, v * w, -np.inf)
        assert int(idx.item()) == int(np.argmax(s))
        gx.check(lib.gpx_sum(dev.h, ptr(vd), n, ptr(tot), dev.stream))
        first = tot.item()
        assert abs(first - v.sum()) <= 1e-12 * np.abs(v).sum()
        gx.check(lib.gpx_sum(dev.h, ptr(vd), n, ptr(tot), dev.stream))
        assert tot.item() == first  # deterministic
    allmask = dev.upload(np.ones(5, dtype=np.uint8), dtype=torch.uint8)
    gx.check(lib.gpx_argreduce(dev.h, ptr(dev.zeros(5)), None, ptr(allmask), 5, 0, ptr(best), ptr(idx), dev.stream))
    assert int(idx.item()) == -1


# ------------------------------------------------------------------------------------------------
# mid-size parity against the CPU oracle (sizes the reference itself cannot reach)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,noise,C,M,n", [("se_ard_2d", 1e-6, 3001, 5003, 130), ("matern_5d", 1e-4, 1500, 2100, 67),
                                              ("mehler_3d", 1e-2, 1000, 1300, 40), ("se_ard_10d", 1e-6, 2000, 2500, 257),
                                              ("se_iso_1d", 1e-6, 129, 1, 3), ("se_ard_2d_wide", 1e-6, 1, 300, 5)])
def test_ivar_scores_vs_oracle(gx, name, noise, C, M, n):
    rng = np.random.default_rng(C + M)
    ks = spec(name)
    k = product_kernel(name)
    samp = rng.standard_normal if name.startswith("mehler") else (lambda s: rng.uniform(-1, 1, s))
    cand, mc, design = samp((C, ks.dim)), samp((M, ks.dim)), samp((n, ks.dim))
    w_m, var_m = orc.fast_design_state(ks, design, mc, noise)
    w_c, var_c = orc.fast_design_state(ks, design, cand, noise)
    ref = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, noise)
    space = gx.Space(ks.dim, None, None, noise=None)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, space, mcPoints=mc)
    costs, best = gx.ed.scoreCandidatesIVAR(cf, design, cand)
    assert best == int(np.argmin(ref))
    assert np.max(np.abs(costs - ref) / np.abs(ref)) <= 1e-9
    # and the reference-shaped single evaluation agrees with the batched score
    one = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), n + 1, space, mcPoints=mc).evaluate(np.vstack([design, cand[:1]]))
    assert abs(one - ref[0]) <= 1e-9 * abs(ref[0])


def test_ivar_empty_design_and_duplicates(gx):
    rng = np.random.default_rng(11)
    ks, k = spec("se_ard_2d_wide"), product_kernel("se_ard_2d_wide")
    cand, mc = rng.uniform(-1, 1, (300, 2)), rng.uniform(-1, 1, (900, 2))
    cand[17] = cand[5]  # duplicate candidates, noise 0: pinv 'no reduction' rule once one of them is chosen
    fidx, fcosts = orc.fast_greedy_ivar(ks, cand, mc, 8, 0.0)
    space = gx.Space(2, None, None, noise=None)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 0.0), 1, space, mcPoints=mc)
    idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 8, returnIndices=True)
    assert [int(i) for i in idx] == fidx
    costs0, best0 = gx.ed.scoreCandidatesIVAR(cf, cand[:0], cand)
    assert best0 == fidx[0]
    assert np.max(np.abs(costs0 - fcosts[0]) / np.abs(fcosts[0])) <= 1e-9


def test_greedy_var_mid_vs_oracle(gx):
    rng = np.random.default_rng(3)
    for name, C, N in [("matern_5d", 20011, 150), ("se_ard_10d", 5000, 140)]:
        ks = spec(name)
        pool = rng.uniform(-1, 1, (C, ks.dim))
        fidx, fscores = orc.fast_greedy_var(ks, pool, N)
        idx, trace = _trace_var(gx, name, pool, N, None, [])
        assert [int(i) for i in idx] == fidx, name
        for s in (0, 1, N // 2, N - 1):
            assert np.max(np.abs(trace[s] - fscores[s])) <= 1e-9 * np.max(np.abs(fscores[s]))


def test_greedy_var_factor_property(gx):
    """Size-independent property at a large pool: the appended rows restricted to the picks are the
    Cholesky factor of K(picks, picks), and every running variance equals prior - colsumsq(W)."""
    rng = np.random.default_rng(5)
    name, C, N = "matern_5d", 250_000, 96
    ks = spec(name)
    pool = rng.uniform(-1, 1, (C, 5))
    bind(gx, name)
    eng = gx.engine.GreedyVarEngine(gx.dev, gx.dev.points(pool), N)
    idx = eng.run(N)
    assert len(set(int(i) for i in idx)) == N
    L = eng.W[:N][:, gx.torch.as_tensor(idx, device=eng.W.device)].cpu().numpy().T
    assert np.allclose(np.triu(L, 1), 0.0, atol=1e-9) and np.all(np.diag(L) > 0)
    Kpp = ks.gram(pool[idx], pool[idx])
    np.testing.assert_allclose(L @ L.T, Kpp, rtol=1e-10, atol=1e-10)
    chk = rng.integers(0, C, 200)
    Wc = eng.W[:N][:, gx.torch.as_tensor(chk, device=eng.W.device)].cpu().numpy()
    var = eng.var.cpu().numpy()[chk]
    np.testing.assert_allclose(var, ks.prior(pool[chk]) - np.sum(Wc * Wc, axis=0), rtol=1e-9, atol=1e-11)
    # greedy property: scores of successive picks never increase
    sc = eng.pick_scores[:N].cpu().numpy()
    assert np.all(np.diff(sc) <= 1e-12)


def test_greedy_mi_mid_vs_oracle(gx):
    rng = np.random.default_rng(9)
    ks, k = spec("mehler_3d"), product_kernel("mehler_3d")
    pool = rng.standard_normal((700, 3))
    fidx, fscores = orc.fast_greedy_mi(ks, pool, 1e-2, 12, start=3)
    space = gx.Space(3, None, None, noise=None)
    cf = gx.ed.costFunctionGP_MI(gx.gp.GP(k, 1e-2), 12, space, nmc=700, mcpoints=pool)
    gx.ed.performGreedyMIExperimentalDesign(cf, 12, start=3)
    assert [int(i) for i in cf.lastIndices] == fidx


def test_cfg4_shape_mi_vs_oracle_at_3000(gx):
    """cfg-4's kernel and noise (3-D Mehler t = 0.9, sigma^2 = 1e-2, N(0, I) pool) at |V| = 3 000: 24 greedy MI picks of
    the blocked engine equal the oracle's (the reference itself is O(|V|^4) per step and stops near |V| = 10^3)."""
    pool = np.random.default_rng(4).standard_normal((3000, 3))
    ks, k = spec("mehler_3d"), product_kernel("mehler_3d")
    ref, _ = orc.fast_greedy_mi(ks, pool, 1e-2, 24, start=0)
    cf = gx.ed.costFunctionGP_MI(gx.gp.GP(k, 1e-2), 24, gx.Space(3, None, None), nmc=3000, mcpoints=pool)
    gx.ed.performGreedyMIExperimentalDesign(cf, 24, start=0)
    assert [int(i) for i in cf.lastIndices] == ref
    assert int(cf.lastEngine.info.item()) == 0


def test_posterior_variance_large_vs_oracle(gx):
    rng = np.random.default_rng(13)
    name = "se_ard_10d"
    ks, k = spec(name), product_kernel(name)
    nodes, query = rng.uniform(-1, 1, (600, 10)), rng.uniform(-1, 1, (10_007, 10))
    g = gx.gp.GP(k, 1e-6)
    g.addNodesAndComputeCovariance(nodes)
    var = g.evaluateVariance(query)
    ref = orc.fast_posterior_variance(ks, nodes, query, 1e-6)
    assert np.max(np.abs(var - ref)) <= 1e-9 * np.max(ks.prior(query))


# ------------------------------------------------------------------------------------------------
# BASELINE.json configurations at (or near) full size: properties + oracle spot checks
# ------------------------------------------------------------------------------------------------
def test_cfg3_full_size_conditional_entropy(gx):
    """cfg-3 in full: 5-D Matern, 1 024 points from 250 000 candidates.  Oracle indices for the first 150 steps,
    size-independent properties for the rest."""
    rng = np.random.default_rng(3)
    C, N = 250_000, 1024
    pool = rng.uniform(-1, 1, (C, 5))
    ks = spec("matern_5d")
    bind(gx, "matern_5d")
    eng = gx.engine.GreedyVarEngine(gx.dev, gx.dev.points(pool), N)
    idx = eng.run(N)
    ref, _ = orc.fast_greedy_var(ks, pool, 150)
    assert [int(i) for i in idx[:150]] == ref
    assert len(set(int(i) for i in idx)) == N
    sel = gx.torch.as_tensor(idx, device=eng.W.device)
    L = eng.W[:N][:, sel].cpu().numpy().T
    np.testing.assert_allclose(L @ L.T, ks.gram(pool[idx], pool[idx]), rtol=0, atol=1e-11)
    assert np.all(np.diff(eng.pick_scores[:N].cpu().numpy()) <= 1e-12)
    # selected points have (numerically) zero remaining variance, everything else is positive
    var = eng.var[:C].cpu().numpy()
    assert np.max(np.abs(var[idx])) <= 1e-12 and var.min() >= -1e-12


def test_cfg2_mid_size_greedy_ivar_vs_oracle(gx):
    rng = np.random.default_rng(2)
    C, M, N = 5000, 12000, 16
    cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
    ks, k = spec("se_ard_2d"), product_kernel("se_ard_2d")
    ref, costs = orc.fast_greedy_ivar(ks, cand, mc, N, 1e-6)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 1, gx.Space(2, None, None), mcPoints=mc)
    idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, N, returnIndices=True)
    assert [int(i) for i in idx] == ref
    want = np.array([c[i] for c, i in zip(costs, ref)])
    assert np.max(np.abs(cf.lastScores - want) / np.abs(want)) <= 1e-9


def test_cfg2_full_size_step_properties(gx):
    """BASELINE configs[1] at full size (100 000 candidates x 100 000 integration points, 2-D ARD, n = 255): one
    scoring step through the public call.  The oracle checks a sample of candidates (with the arg-min); the rest of
    the full-size result is pinned by size-independent properties of the criterion: a candidate's cost does not depend
    on where it sits in the candidate array (bit-exact under a permutation), and the integrated variance is additive
    over a partition of the integration points: M cost(M) = M1 cost(M1) + M2 cost(M2)."""
    rng = np.random.default_rng(22)
    C = M = 100_000
    n, noise = 255, 1e-6
    cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
    design = cand[rng.permutation(C)[:n]]
    ks, k = spec("se_ard_2d"), product_kernel("se_ard_2d")

    def cost_fn(points):
        return gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, gx.Space(2, None, None), mcPoints=points)

    costs, best = gx.ed.scoreCandidatesIVAR(cost_fn(mc), design, cand)
    assert costs.shape == (C,) and np.all(np.isfinite(costs)) and costs[best] == costs.min()
    sub = np.unique(np.concatenate([[best], rng.permutation(C)[:96]]))
    w_m, var_m = orc.fast_design_state(ks, design, mc, noise)
    w_c, var_c = orc.fast_design_state(ks, design, cand[sub], noise)
    ref = orc.fast_ivar_scores(ks, cand[sub], mc, w_m, var_m, w_c, var_c, noise)
    assert np.max(np.abs(costs[sub] - ref) / np.abs(ref)) <= 1e-9
    # position independence
    perm = rng.permutation(C)
    costs_p, best_p = gx.ed.scoreCandidatesIVAR(cost_fn(mc), design, cand[perm])
    assert np.array_equal(costs_p, costs[perm])
    assert costs_p[best_p] == costs[best]
    # additivity over the integration points (unequal parts, neither a multiple of the 128-row tile)
    m1 = 37_411
    c1, _ = gx.ed.scoreCandidatesIVAR(cost_fn(mc[:m1]), design, cand)
    c2, _ = gx.ed.scoreCandidatesIVAR(cost_fn(mc[m1:]), design, cand)
    np.testing.assert_allclose(m1 * c1 + (M - m1) * c2, M * costs, rtol=1e-11, atol=0)


def test_cfg5_shape_step_vs_oracle_subset(gx):
    """cfg-5 operand shape (10-D ARD, long K loop, several M-splits) at n = 1024: one scoring step from a given
    design; every 300th candidate and the arg-min are checked against the oracle."""
    rng = np.random.default_rng(5)
    C, M, n, d = 20_000, 30_000, 1024, 10
    cand, mc = rng.uniform(-1, 1, (C, d)), rng.uniform(-1, 1, (M, d))
    design = cand[rng.permutation(C)[:n]]
    ks, k = spec("se_ard_10d"), product_kernel("se_ard_10d")
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 1, gx.Space(d, None, None), mcPoints=mc)
    costs, best = gx.ed.scoreCandidatesIVAR(cf, design, cand)
    sub = np.unique(np.concatenate([[best], np.arange(0, C, 300)]))
    w_m, var_m = orc.fast_design_state(ks, design, mc, 1e-6)
    w_c, var_c = orc.fast_design_state(ks, design, cand[sub], 1e-6)
    ref = orc.fast_ivar_scores(ks, cand[sub], mc, w_m, var_m, w_c, var_c, 1e-6)
    assert np.max(np.abs(costs[sub] - ref) / np.abs(ref)) <= 1e-9
    assert costs[best] == costs.min()


def test_sharded_mi_engine_single_rank_equals_dense_engine(gx):
    """The column-sharded MI engine (left-looking blocked factorisation, Y = U^-T built block row by block row)
    run with one rank must reproduce the dense engine and the oracle; the 2- and 8-rank runs are covered by
    scripts/multigpu_check.py."""
    rng = np.random.default_rng(21)
    for name, V, N, noise in [("mehler_3d", 700, 10, 1e-2), ("matern_5d", 1000, 8, 1e-3)]:
        ks = spec(name)
        bind(gx, name)
        pool = rng.standard_normal((V, ks.dim)) if name.startswith("mehler") else rng.uniform(-1, 1, (V, ks.dim))
        ref, ref_scores = orc.fast_greedy_mi(ks, pool, noise, N, start=2)
        eng = gx.engine.ShardedMIEngine(gx.dev, pool, N, noise)
        eng.score_trace = []
        idx = eng.run(N, start=2)
        assert int(eng.info.item()) == 0
        assert [int(i) for i in idx] == ref, name
        for s, sc in enumerate(eng.score_trace):
            ok = np.isfinite(ref_scores[s])
            assert np.max(np.abs(sc[ok] - ref_scores[s][ok]) / np.abs(ref_scores[s][ok])) <= 1e-8


# ------------------------------------------------------------------------------------------------
# limits and error behaviour of the C ABI
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [13, 16])
def test_max_dimension_ivar_and_gram(gx, d):
    """GPX_MAX_DIM = 16: the Gram prologue then fills the whole 16-row K chunk (d = 13 pads to 16)."""
    from gpexp_b200 import kernels as K
    rng = np.random.default_rng(d)
    cl = list(np.linspace(0.8, 2.0, d))
    ks = orc.KernelSpec.se(cl, 1.3, d)
    k = K.KernelSquaredExponential(cl, 1.3, d)
    cand, mc, design = rng.uniform(-1, 1, (700, d)), rng.uniform(-1, 1, (900, d)), rng.uniform(-1, 1, (37, d))
    np.testing.assert_allclose(gx.gku.calculateCovarianceMatrix(k, design, 1e-6), ks.gram(design, design).T + 1e-6 * np.eye(37),
                               rtol=RTOL_K)
    w_m, var_m = orc.fast_design_state(ks, design, mc, 1e-6)
    w_c, var_c = orc.fast_design_state(ks, design, cand, 1e-6)
    ref = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, 1e-6)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 1, gx.Space(d, None, None), mcPoints=mc)
    costs, best = gx.ed.scoreCandidatesIVAR(cf, design, cand)
    assert best == int(np.argmin(ref)) and np.max(np.abs(costs - ref) / np.abs(ref)) <= 1e-9
    with pytest.raises(gx._lib.GpxError):
        K.KernelSquaredExponential([1.0], 1.0, 17).evaluate(np.zeros((2, 17)), np.zeros((2, 17)))


def test_c_abi_error_codes(gx):
    dev, lib, ptr, torch = gx.dev, gx.lib, gx.ptr, gx.torch
    bind(gx, "se_ard_2d")
    a = dev.zeros(4, 130)
    info = dev.zeros(1, dtype=torch.int32)
    # odd leading dimension / misaligned pointer -> GPX_EALIGN, message available, nothing launched
    assert lib.gpx_potrf(dev.h, ptr(a), 4, 129, ptr(info), dev.stream) == -2
    assert "16-byte" in gx._lib.last_error()
    assert lib.gpx_dgemm_tn_sub(dev.h, ptr(a) + 8, 130, ptr(a), 130, ptr(a), 130, 2, 2, 2, 0, dev.stream) == -2
    # bad arguments -> GPX_EINVAL
    assert lib.gpx_kernel_pairwise(dev.h, ptr(a), 3, 130, ptr(a), 5, 130, ptr(a), dev.stream) == -1
    assert lib.gpx_gram(dev.h, ptr(a), 2, 130, ptr(a), 200, 130, ptr(a), 130, 0, None, 0.0, dev.stream) == -1  # ld < ny
    assert lib.gpx_argreduce(dev.h, ptr(a), None, None, -1, 0, ptr(a), ptr(info), dev.stream) == -1
    # a fresh handle has no kernel -> GPX_ENOKERNEL
    h2 = C.c_void_p()
    assert lib.gpx_create(dev.index, C.byref(h2)) == 0
    assert lib.gpx_prior_diag(h2, ptr(a), 4, 130, ptr(a), dev.stream) == -3
    import ctypes
    bad = (ctypes.c_double * 3)(0.5, 0.5, 1.0)
    assert lib.gpx_set_kernel(h2, 7, 2, bad, 3) == -1           # unknown family
    assert lib.gpx_set_kernel(h2, 0, 17, bad, 18) == -4          # dimension above GPX_MAX_DIM
    assert lib.gpx_set_kernel(h2, 2, 2, (ctypes.c_double * 2)(0.5, 1.0), 2) == -1  # Mehler |t| >= 1
    assert lib.gpx_destroy(h2) == 0
    # empty inputs are no-ops that succeed
    assert lib.gpx_gram(dev.h, ptr(a), 0, 130, ptr(a), 0, 130, ptr(a), 130, 0, None, 0.0, dev.stream) == 0
    assert lib.gpx_append_row(dev.h, 0, ptr(a), None, ptr(a), 0, 130, ptr(a), 130, 0, ptr(a), dev.stream) == 0
    from gpexp_b200 import kernels as K
    assert K.KernelSquaredExponential([0.5], 1.0, 2).evaluate(np.zeros((0, 2)), np.zeros((0, 2))).shape == (0,)


def test_score_ivar_unpadded_operands_use_the_generic_core(gx):
    """Raw C-ABI call with leading dimensions that are NOT multiples of 128: gpx_score_ivar must fall back from the
    TMA kernel (whole-tile reads) to the predicated cp.async core and give the same scores."""
    dev, lib, ptr, torch = gx.dev, gx.lib, gx.ptr, gx.torch
    rng = np.random.default_rng(33)
    ks = spec("matern_5d")
    bind(gx, "matern_5d")
    M, Cn, n, noise = 301, 203, 21, 1e-4
    mc, cand, design = rng.uniform(-1, 1, (M, 5)), rng.uniform(-1, 1, (Cn, 5)), rng.uniform(-1, 1, (n, 5))
    w_m, var_m = orc.fast_design_state(ks, design, mc, noise)
    w_c, var_c = orc.fast_design_state(ks, design, cand, noise)
    ref = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, noise)
    ldm, ldc = 302, 204

    def up(a, ld):
        t = dev.zeros(a.shape[0], ld)
        t[:, : a.shape[1]] = dev.upload(a)
        return t
    Xm, Xc = up(mc.T.copy(), ldm), up(cand.T.copy(), ldc)
    Wm, Wc = up(w_m, ldm), up(w_c, ldc)
    vM, vC = up(var_m[None, :], ldm), up(var_c[None, :], ldc)
    ma_rows, cb_rows, mx = dev.zeros(16, ldm), dev.zeros(16, ldc), dev.zeros(1)
    gx.check(lib.gpx_prep_side(dev.h, 0, ptr(Xm), M, ldm, ptr(ma_rows), ldm, ptr(mx), dev.stream))
    assert 0.0 < mx.item() <= 5.0 + 1e-12  # max |alpha| = max sum x^2 on [-1,1]^5
    gx.check(lib.gpx_prep_side(dev.h, 1, ptr(Xc), Cn, ldc, ptr(cb_rows), ldc, None, dev.stream))
    ws = dev.zeros(int(lib.gpx_score_ivar_workspace(dev.h, M, Cn)))
    # both prologue forms: prepared sides on the tensor pipe, and raw coordinates in difference form
    for mode, ra, rb in [(gx._lib.PRO_EXPANDED, ma_rows, cb_rows), (gx._lib.PRO_DIFF, Xm, Xc)]:
        score, best, idx = dev.zeros(ldc), dev.zeros(1), dev.zeros(1, dtype=torch.int64)
        gx.check(lib.gpx_score_ivar(dev.h, mode, ptr(Wm), ldm, ptr(vM), ptr(ra), M, ptr(Wc), ldc, ptr(vC), ptr(rb), Cn, n,
                                    noise, 1e-13, None, ptr(ws), ptr(score), ptr(best), ptr(idx), dev.stream))
        got = score[:Cn].cpu().numpy()
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-9, mode
        assert int(idx.item()) == int(np.argmin(ref)) and best.item() == got.min()


# ------------------------------------------------------------------------------------------------
# SURVEY.md 8(f) widening: marginal log-likelihood and the IVAR gradient, golden vectors of the reference
# ------------------------------------------------------------------------------------------------
def test_next_loglike_golden(gx, golden):
    z = golden("next")
    for name in sorted({k.split("/")[2] for k in z.files if k.startswith("next/loglike/")}):
        k = product_kernel(name)
        nodes, fvals, noise = z[f"next/loglike/{name}/nodes"], z[f"next/loglike/{name}/fvals"], float(z[f"next/loglike/{name}/noise"])
        ref = float(z[f"next/loglike/{name}/value"])
        got = gx.gp.GP(k, noise).computeLogLike(nodes, fvals)
        # pinv/slogdet vs Cholesky: cond * eps on the quadratic form (fast_loglike meets the same bound on the CPU)
        assert abs(got - ref) <= 1e-7 * abs(ref), (name, got, ref)
        assert abs(got - orc.fast_loglike(spec(name), nodes, fvals, noise)) <= 1e-10 * abs(ref)


def test_next_ivar_gradient_golden(gx, golden):
    z = golden("next")
    for name in sorted({k.split("/")[2] for k in z.files if k.startswith("next/grad/")}):
        k = product_kernel(name)
        design, mc, one = z[f"next/grad/{name}/design"], z[f"next/grad/{name}/mc"], z[f"next/grad/{name}/one"]
        noise, cond = float(z[f"next/grad/{name}/noise"]), float(z[f"next/grad/{name}/cond"])
        tol = max(1e-9, 100 * cond * EPS)
        np.testing.assert_allclose(k.derivative(mc, one), z[f"next/grad/{name}/kderiv"], rtol=RTOL_K, atol=1e-300)
        g = gx.gp.GP(k, noise)
        g.addNodesAndComputeCovariance(design)
        ref = z[f"next/grad/{name}/var_deriv"]
        got = g.evaluateVarianceDerivative(mc[:64])
        assert got.shape == ref.shape
        assert np.max(np.abs(got - ref)) <= tol * np.max(np.abs(ref)), name
        cf = gx.ed.costFunctionGP_IVAR(g, design.shape[0], gx.Space(k.dimension, None, None), mcPoints=mc)
        gref = z[f"next/grad/{name}/ivar_deriv"]
        ggot = cf.derivative(design)
        assert ggot.shape == gref.shape and np.max(np.abs(ggot - gref)) <= tol * np.max(np.abs(gref)), name
    with pytest.raises(AttributeError):
        gm = gx.gp.GP(product_kernel("matern_5d"), 1e-4)
        gm.addNodesAndComputeCovariance(np.zeros((3, 5)) + np.arange(3)[:, None])
        gm.evaluateVarianceDerivative(np.zeros((4, 5)))


def test_ivar_gradient_matches_finite_differences(gx):
    """Property check independent of the reference: with signalSize = 1 the gradient is the true derivative of
    costFunctionGP_IVAR.evaluate with respect to the design coordinates."""
    from gpexp_b200 import kernels as K
    rng = np.random.default_rng(8)
    k = K.KernelSquaredExponential([0.4, 0.6, 0.5], 1.0, 3)
    design, mc = rng.uniform(-1, 1, (7, 3)), rng.uniform(-1, 1, (5000, 3))
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 7, gx.Space(3, None, None), mcPoints=mc)
    g = cf.derivative(design).reshape(7, 3)
    h = 1e-6
    for (j, q) in [(0, 0), (3, 2), (6, 1)]:
        dp, dm = design.copy(), design.copy()
        dp[j, q] += h
        dm[j, q] -= h
        fd = (cf.evaluate(dp) - cf.evaluate(dm)) / (2 * h)
        assert abs(fd - g[j, q]) <= 1e-5 * max(abs(fd), 1e-3), (j, q, fd, g[j, q])


@pytest.fixture(scope="module")
def patched_ref(gx):
    """The UNMODIFIED reference package from baseline/_ref (copied there by __graft_entry__.build() from $GPEXP_REFERENCE;
    git-ignored), with its hot methods rebound by gpexp_b200.install_as_gpExp: its own constructors and optimiser loops run
    on the device path."""
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        pytest.skip("baseline/_ref/gpExp is not present (set GPEXP_REFERENCE and run __graft_entry__.build() to stage it)")
    import gpexp_b200
    ref = gpexp_b200.install_as_gpExp(path)
    import importlib

    class R:
        pass
    r = R()
    r.pkg = ref
    for name in ("kernels", "gp", "gp_kernel_utilities", "experimentalDesign", "approximation"):
        setattr(r, name, importlib.import_module("gpExp." + name))
    r.experimentalDesign.VERBOSE = False
    return r


def _quiet(fn, *a, **k):
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def test_patched_reference_keeps_its_own_host_code(gx, patched_ref):
    r = patched_ref
    from gpexp_b200 import experimentalDesign as ed, gp, kernels
    assert os.path.realpath(r.pkg.__file__).startswith(os.path.realpath(os.path.join(ROOT, "baseline", "_ref")))
    # rebound: the hot methods ...
    assert r.kernels.Kernel.evaluate is kernels.Kernel.evaluate
    assert r.gp.GP.evaluateVariance is gp.GP.evaluateVariance and r.gp.GP.train is gp.GP.train
    assert r.experimentalDesign.costFunctionGP_IVAR.evaluate is ed.costFunctionGP_IVAR.evaluate
    assert r.experimentalDesign.performGreedyVarExperimentalDesign is ed.performGreedyVarExperimentalDesign
    # ... and nothing else: constructors and optimiser loops are the reference's own code
    assert r.kernels.KernelSquaredExponential.__init__.__module__ == "gpExp.kernels"
    assert r.gp.GP.__init__.__module__ == "gpExp.gp" and r.gp.GP.findOptParamsLogLike.__module__ == "gpExp.gp"
    assert r.experimentalDesign.ExperimentalDesignDerivative.begin.__module__ == "gpExp.experimentalDesign"
    assert r.experimentalDesign.costFunctionGP_MI.__init__.__module__ == "gpExp.experimentalDesign"


def test_next_slsqp_polish_golden(gx, golden, patched_ref):
    """ExperimentalDesignDerivative.begin / beginWithVarGreedy (experimentalDesign.py:379-497) -- the REFERENCE's optimiser
    loop, unmodified, over the device cost + gradient: same start design, and the SLSQP polish lands on the reference's
    end design."""
    r = patched_ref
    z = golden("next")
    mc = z["next/slsqp/mc"]
    k = r.kernels.KernelSquaredExponential([0.3, 0.45], 1.7, 2)
    dens = lambda p: np.all(np.abs(p) <= 1.0, axis=1).astype(float)  # noqa: E731
    space = r.approximation.Space(2, None, dens, noise=None)
    cf = r.experimentalDesign.costFunctionGP_IVAR(r.gp.GP(k, 1e-6), 5, space, mcPoints=mc)
    exp = r.experimentalDesign.ExperimentalDesignDerivative(cf, 5, 2)
    start = r.experimentalDesign.performGreedyVarExperimentalDesign(k, mc, 5, 2)
    assert np.array_equal(start, z["next/slsqp/start"])
    assert abs(cf.evaluate(start) - float(z["next/slsqp/cost_start"])) <= 1e-9 * float(z["next/slsqp/cost_start"])
    end = _quiet(exp.begin, [start], list(-np.ones(10)), list(np.ones(10)))
    # SLSQP stops at acc = 1e-6 on the objective: compare the optimum, and the design to the optimiser's own accuracy
    assert abs(cf.evaluate(end) - float(z["next/slsqp/cost_end"])) <= 1e-6
    assert np.max(np.abs(end - z["next/slsqp/end"])) <= 5e-3
    end2 = _quiet(exp.beginWithVarGreedy, None, list(-np.ones(10)), list(np.ones(10)))
    assert np.max(np.abs(end2 - end)) <= 1e-9


def test_next2_batch_greedy_wrapper_golden(gx, golden, patched_ref):
    """ExperimentalDesignGreedyWithDerivatives.begin (experimentalDesign.py:694-751): the reference's batch-greedy loop
    (2 + 2 points; each batch = greedy max-variance start + SLSQP polish) driving the device path."""
    r = patched_ref
    z = golden("next2")
    mc = z["next2/batch/mc"]
    k = r.kernels.KernelSquaredExponential([0.3, 0.45], 1.7, 2)
    srng = np.random.default_rng(7)
    dens = lambda p: np.all(np.abs(p) <= 1.0, axis=1).astype(float)  # noqa: E731
    space = r.approximation.Space(2, lambda s: srng.uniform(-1, 1, s), dens, noise=None)
    red = r.experimentalDesign
    cf = red.costFunctionGP_IVAR(r.gp.GP(k, 1e-6), 2, space, mcPoints=mc)
    pts = _quiet(red.ExperimentalDesignGreedyWithDerivatives(cf, 4, 2, 2).begin)
    cost = red.costFunctionGP_IVAR(r.gp.GP(k, 1e-6), 4, space, mcPoints=mc).evaluate(pts)
    assert pts.shape == (4, 2)
    assert abs(cost - float(z["next2/batch/cost"])) <= 1e-6
    assert np.max(np.abs(pts - z["next2/batch/points"])) <= 5e-3


def test_next2_heteroscedastic_gradient_golden(gx, golden):
    """f2: GP.evaluateVarianceDerivative(noiseFunc=...) and costFunctionGP_IVAR.derivative with a heteroscedastic noise
    function (gp.py:282-341, experimentalDesign.py:170-176) against the unmodified reference."""
    from gpexp_b200 import kernels as K
    from tests.golden.make_golden_shared import QuadNoise
    z = golden("next2")
    nf = QuadNoise()
    for name, kern in [("se_ard_2d_wide", K.KernelSquaredExponential([0.3, 0.45], 1.7, 2)),
                       ("se_iso_1d", K.KernelSquaredExponential([0.05], 1.0, 1))]:
        design, mc = z[f"next2/hetero/{name}/design"], z[f"next2/hetero/{name}/mc"]
        g = gx.gp.GP(kern, 1e-6)
        g.addNodesAndComputeCovariance(design, noiseIn=nf(design))
        got = g.evaluateVarianceDerivative(mc[:48], noiseFunc=nf)
        ref = z[f"next2/hetero/{name}/var_deriv"]
        assert got.shape == ref.shape
        assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref)), name
        cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(kern, 1e-6), len(design), gx.Space(kern.dimension, None, None, noise=nf),
                                       mcPoints=mc)
        assert abs(cf.evaluate(design) - float(z[f"next2/hetero/{name}/ivar_cost"])) <= 1e-9 * float(z[f"next2/hetero/{name}/ivar_cost"])
        gd, rd = cf.derivative(design), z[f"next2/hetero/{name}/ivar_deriv"]
        assert np.max(np.abs(gd - rd)) <= 1e-9 * np.max(np.abs(rd)), name


def test_next2_fitc_golden(gx, golden):
    """f4: FITC sparse GP (gp.py:182-208, gp_kernel_utilities.py:70-104): same inducing points (np.random.permutation under
    the same seed), covariance, Woodbury precision, coefficients, mean, variance and log-likelihood of the reference."""
    z = golden("next2")
    for name in ["se_ard_2d_wide", "matern_5d"]:
        k = product_kernel(name)
        nodes, query, fvals = z[f"next2/fitc/{name}/nodes"], z[f"next2/fitc/{name}/query"], z[f"next2/fitc/{name}/fvals"]
        noise = float(z[f"next2/fitc/{name}/noise"])
        np.random.seed(11)
        g = gx.gp.GP(k, noise, FITC=0.5)
        g.train(nodes, fvals)
        assert np.array_equal(g.fitcnodes, z[f"next2/fitc/{name}/inducing"])
        np.testing.assert_allclose(g.covarianceMatrix, z[f"next2/fitc/{name}/cov"], rtol=1e-10, atol=1e-12)
        pref = z[f"next2/fitc/{name}/prec"]
        # the precision carries 1/g ~ 1/noise entries; compare at the scale of the matrix
        assert np.max(np.abs(g.precisionMatrix - pref)) <= 1e-8 * np.max(np.abs(pref)), name
        cref = z[f"next2/fitc/{name}/coeff"]
        assert np.max(np.abs(g.coeff - cref)) <= 1e-7 * np.max(np.abs(cref))
        var = g.evaluateVariance(query)
        vref = z[f"next2/fitc/{name}/var"]
        # k^T P k with P ~ 1/g ~ 1/noise (1e3 .. 1e4 here) cancels to O(1): eps * |P| * n of round-off on BOTH sides
        # (the reference's inv/pinv and the device's Cholesky pair), so the comparison is at 1e-7 of the variance scale
        vtol = 2e-7 * max(1.0, np.max(np.abs(vref)))
        assert np.max(np.abs(var - vref)) <= vtol, name
        mean, absvar = g.evaluate(query, compvar=1)
        assert np.max(np.abs(mean - z[f"next2/fitc/{name}/mean"])) <= 1e-7 * max(1.0, np.max(np.abs(z[f"next2/fitc/{name}/mean"])))
        assert np.max(np.abs(absvar - z[f"next2/fitc/{name}/absvar"])) <= vtol
        np.random.seed(11)
        ll = gx.gp.GP(k, noise, FITC=0.5).computeLogLike(nodes, fvals)
        assert abs(ll - float(z[f"next2/fitc/{name}/loglike"])) <= 1e-8 * abs(float(z[f"next2/fitc/{name}/loglike"]))
        cov, prec, sn = gx.gku.calculateCovarianceMatrixFITC(k, nodes, noise, z[f"next2/fitc/{name}/inducing"], returnCov=True)
        np.testing.assert_allclose(cov, z[f"next2/fitc/{name}/util_cov"], rtol=1e-10, atol=1e-12)
        assert np.max(np.abs(prec - z[f"next2/fitc/{name}/util_prec"])) <= 1e-8 * np.max(np.abs(pref))


def test_next2_gram_matvec_and_nystrom_golden(gx, golden):
    """f4: covTimesV (gp_kernel_utilities.py:107-142) as one fused Gram x vector kernel, and the Nystrom eigenvalues of
    calculateKernelBasisFunctionsMC (:144-194) from eigsh over that operator; plus a 20 011-point product against numpy."""
    z = golden("next2")
    for name in ["se_ard_2d_wide", "matern_5d", "mehler_3d_b"]:
        k = product_kernel(name)
        pts, b, ref = z[f"next2/matvec/{name}/pts"], z[f"next2/matvec/{name}/b"], z[f"next2/matvec/{name}/Kb"]
        got = gx.gku.covTimesV(b, k, pts)
        assert got.shape == b.shape and np.max(np.abs(got - ref)) <= 1e-11 * np.max(np.abs(ref)), name
    k = product_kernel("se_ard_2d_wide")
    eigv, eigve = gx.gku.calculateKernelBasisFunctionsMC(k, 6, z["next2/nystrom/pts"])
    rv, rve = z["next2/nystrom/eigv"], z["next2/nystrom/eigve"]
    assert np.max(np.abs(eigv - rv)) <= 1e-9 * rv[0]
    for c in range(6):  # eigenvectors are defined up to sign
        assert min(np.max(np.abs(eigve[:, c] - rve[:, c])), np.max(np.abs(eigve[:, c] + rve[:, c]))) <= 1e-6 * np.max(np.abs(rve[:, c]))
    rng = np.random.default_rng(9)
    ks = spec("matern_5d")
    kk = product_kernel("matern_5d")
    P = rng.uniform(-1, 1, (20011, 5))
    v = rng.standard_normal(20011)
    got = gx.gku.covTimesV(v, kk, P)
    rows = rng.permutation(20011)[:64]
    want = ks.gram(P[rows], P) @ v
    assert np.max(np.abs(got[rows] - want)) <= 1e-11 * np.max(np.abs(want))


def test_loglike_gradient_vs_oracle(gx, golden):
    """f3: loglikeParams(returnDeriv=1) (gp.py:447-468).  The reference's own gradient raises IndexError under current
    numpy (kernels.py:140-142 indexes with a float), so parity is against the analytic expression restated in the oracle
    (itself checked against finite differences of the golden-pinned value in tests/test_oracle.py)."""
    z = golden("next")
    from gpexp_b200 import kernels as K
    for name, kern in [("se_ard_2d_wide", K.KernelSquaredExponential([0.3, 0.45], 1.7, 2)),
                       ("se_ard_10d", K.KernelSquaredExponential(list(np.linspace(0.5, 1.5, 10)), 1.0, 10))]:
        pts, y = z[f"next/loglike/{name}/nodes"], z[f"next/loglike/{name}/fvals"]
        for noise in (float(z[f"next/loglike/{name}/noise"]), 1e-3):
            g = gx.gp.GP(kern, noise)
            val, grad = g.loglikeParams(pts, y, returnDeriv=1)
            assert abs(val - orc.fast_loglike(spec(name), pts, y, noise)) <= 1e-9 * abs(val)
            ref = orc.fast_loglike_gradient(spec(name), pts, y, noise)
            assert list(grad.keys()) == list(kern.hyperParam.keys()) + ['noise']
            scale = max(abs(v) for v in ref.values())
            for key, v in ref.items():
                assert abs(grad[key] - v) <= 1e-8 * scale, (name, noise, key, grad[key], v)
    with pytest.raises(AttributeError):
        gx.gp.GP(product_kernel("matern_5d"), 1e-4).loglikeParams(z["next/loglike/matern_5d/nodes"],
                                                                   z["next/loglike/matern_5d/fvals"], returnDeriv=1)


def test_resident_covariance_mode_equals_contraction_mode(gx):
    """The HBM-resident posterior covariance (one rank-1 update pass per step) must give the picks and scores of
    the per-step DMMA contraction, for a grown design and for a design loaded from scratch."""
    rng = np.random.default_rng(44)
    for name, noise, C, M, N in [("se_ard_2d", 1e-6, 3001, 2500, 30), ("matern_5d", 1e-4, 1111, 1300, 20),
                                 ("mehler_3d", 1e-2, 700, 900, 12)]:
        ks = spec(name)
        k = bind(gx, name)
        samp = rng.standard_normal if name.startswith("mehler") else (lambda s: rng.uniform(-1, 1, s))
        cand, mc = samp((C, ks.dim)), samp((M, ks.dim))
        fam, d, params = k._gpx_spec()
        scale = gx.engine.prior_scale(fam, params)
        e1 = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), N, noise, scale)
        e2 = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), N, noise, scale, resident=True)
        e1.score_trace, e2.score_trace = [], []
        i1, i2 = e1.run(N), e2.run(N)
        assert [int(i) for i in i1] == [int(i) for i in i2], name
        for a, b in zip(e1.score_trace, e2.score_trace):
            assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-10
        # from a given design: cov = K - W_M^T W_C built by the DMMA store kernel, then two more greedy steps
        design = cand[[int(i) for i in i1[:7]]]
        f = gx.engine.DesignFactor(gx.dev, gx.dev.points(design), noise)
        e3 = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), 10, noise, scale, resident=True)
        e3.load_design(f)
        e3.score()
        assert int(e3.idx.item()) == int(i1[7])
        np.testing.assert_allclose(e3.scores[:C].cpu().numpy(), e1.score_trace[7], rtol=1e-9)
        e3.append()
        e3.score()
        assert int(e3.idx.item()) == int(i1[8])


@pytest.mark.parametrize("shape", [(1, 1, 1), (3, 130, 5), (129, 257, 33), (260, 131, 200), (512, 700, 1000), (128, 128, 32)])
def test_dgemm_tn_sub_padded_tma_kernel(gx, shape):
    """The TMA + mbarrier update kernel (fully padded operands) against numpy, ragged I / J / K and the symmetric mode."""
    I, J, K = shape
    rng = np.random.default_rng(I * 7 + J)
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    A, B, Cm = rng.standard_normal((K, I)), rng.standard_normal((K, J)), rng.standard_normal((I, J))
    lda, ldb, ldc = gx.device.roundup(I), gx.device.roundup(J), gx.device.roundup(J)
    Ad, Bd, Cd = dev.zeros(K, lda), dev.zeros(K, ldb), dev.zeros(I, ldc)
    Ad[:, :I], Bd[:, :J], Cd[:, :J] = dev.upload(A), dev.upload(B), dev.upload(Cm)
    gx.check(lib.gpx_dgemm_tn_sub_padded(dev.h, ptr(Ad), lda, ptr(Bd), ldb, ptr(Cd), ldc, I, J, K, 0, dev.stream))
    np.testing.assert_allclose(Cd[:, :J].cpu().numpy(), Cm - A.T @ B, rtol=1e-12, atol=1e-12)
    assert np.all(Cd[:, J:].cpu().numpy() == 0.0)
    if I == J:
        Cd[:, :J] = dev.upload(Cm)
        gx.check(lib.gpx_dgemm_tn_sub_padded(dev.h, ptr(Ad), lda, ptr(Ad), lda, ptr(Cd), ldc, I, I, K, 1, dev.stream))
        got, want = Cd[:, :J].cpu().numpy(), Cm - A.T @ A
        np.testing.assert_allclose(np.triu(got), np.triu(want), rtol=1e-12, atol=1e-12)
    # unpadded leading dimension is refused
    assert lib.gpx_dgemm_tn_sub_padded(dev.h, ptr(Ad), 2, ptr(Bd), ldb, ptr(Cd), ldc, max(I, 3), J, K, 0, dev.stream) == -2


# ------------------------------------------------------------------------------------------------
# round 2: BASELINE configs[0] at full size against the unmodified reference, conditioning guards, C-side loops
# ------------------------------------------------------------------------------------------------
def _cfg1(golden, tag):
    z = golden("cfg1")
    return (z["cfg1/cand"], z["cfg1/mc"], float(z[f"cfg1/{tag}/cl"]), float(z[f"cfg1/{tag}/noise"]),
            z[f"cfg1/{tag}/idx"], z[f"cfg1/{tag}/costs"], z[f"cfg1/{tag}/cond"])


def test_cfg1_full_size_golden(gx, golden):
    """configs[0]: 1-D SE cl=0.05, 20 of 1 000 candidates x 10 000 MC points -- every one of the 20 x 1 000 costs of the
    unmodified reference (costFunctionGP_IVAR.evaluate per candidate and step), through the public driver (C-side loop)
    and through the traced step path."""
    cand, mc, cl, noise, idx, ref_costs, _ = _cfg1(golden, "main")
    from gpexp_b200 import kernels as K
    k = K.KernelSquaredExponential([cl], 1.0, 1)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, gx.Space(1, None, None), mcPoints=mc)
    for resident in (False, True):
        got = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 20, returnIndices=True, resident=resident)
        assert [int(i) for i in got] == [int(i) for i in idx], resident
        want = ref_costs[np.arange(20), idx]
        assert np.max(np.abs(cf.lastScores - want) / np.abs(want)) <= 1e-9
        assert cf.illConditionedFrom is None and cf.lastPivots.shape == (20,)
    fam, d, params = k._gpx_spec()
    eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), 20, noise, gx.engine.prior_scale(fam, params))
    eng.score_trace = []
    eng.run(20)
    for s, c in enumerate(eng.score_trace):
        assert np.max(np.abs(c - ref_costs[s]) / np.abs(ref_costs[s])) <= 1e-9, s


def test_cfg1_demo_stress_variant_flags_ill_conditioning(gx, golden):
    """demo.py:52-58 values (cl = 0.3, noise 0.0): the reference's own Gram reaches cond 3e11 at step 10 and 1e17 later
    (fixture cfg1/stress/cond).  Contract: identical picks while cond <= ~1e7 (the documented first 10 steps), picked
    costs within cond * 1e-13, and a GpxConditionWarning naming a step no later than the first pick that differs."""
    import warnings
    cand, mc, cl, noise, idx, ref_costs, cond = _cfg1(golden, "stress")
    from gpexp_b200 import kernels as K
    k = K.KernelSquaredExponential([cl], 1.0, 1)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, gx.Space(1, None, None), mcPoints=mc)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        got = [int(i) for i in gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 20, returnIndices=True, resident=False)]
    assert got[:10] == [int(i) for i in idx[:10]]
    for s in range(10):
        want = ref_costs[s, idx[s]]
        assert abs(cf.lastScores[s] - want) <= max(1e-9, 1e-13 * cond[s]) * abs(want), s
    first_diff = next((s for s in range(20) if got[s] != int(idx[s])), 20)
    assert cf.illConditionedFrom is not None and cf.illConditionedFrom <= first_diff
    assert any(issubclass(x.category, gx.engine.GpxConditionWarning) for x in w)
    assert np.all(np.isfinite(cf.lastScores)) and np.all(np.isfinite(cf.lastPivots))


def test_c_side_loop_equals_step_path(gx):
    """gpx_ivar_greedy_run / gpx_var_greedy_run issue the same arithmetic as the per-step Python path: bit-identical
    picks, scores and pivots, in contraction and resident mode."""
    rng = np.random.default_rng(77)
    cand, mc = rng.uniform(-1, 1, (2300, 2)), rng.uniform(-1, 1, (1700, 2))
    k = bind(gx, "se_ard_2d_wide")
    fam, d, params = k._gpx_spec()
    for resident in (False, True):
        out = []
        for traced in (False, True):
            eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), 17, 1e-6,
                                             gx.engine.prior_scale(fam, params), resident=resident)
            if traced:
                eng.score_trace = []
            eng.run(17)
            out.append((eng.indices(), eng.pick_scores[:17].cpu().numpy(), eng.pivots(), eng.U[:17, :17].cpu().numpy()))
        for a, b in zip(out[0], out[1]):
            if resident:
                # the untraced resident run of this size is the ONE-KERNEL loop: identical picks; scores, pivots and factor
                # entries equal up to the summation order (four partial sums per dot product there, one here): a few
                # ulps of the O(1) terms, which is 1e-13 relative on the smallest entries of U
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-15)
            else:
                assert np.array_equal(a, b), resident
        assert np.array_equal(out[0][0], out[1][0])
    pool = rng.uniform(-1, 1, (5001, 5))
    bind(gx, "matern_5d")
    w = rng.uniform(0.5, 1.5, 5001)
    res = []
    for traced in (False, True):
        eng = gx.engine.GreedyVarEngine(gx.dev, gx.dev.points(pool), 33, weights=w)
        if traced:
            eng.score_trace = []
        eng.run(33, progress=(lambda n: None) if not traced else None)
        res.append((eng.indices(), eng.pick_scores[:33].cpu().numpy(), eng.pivots()))
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)


def test_expanded_form_guard_and_centring(gx):
    """VERDICT r1 weak-3: k = f(alpha + beta + u.v) cancels |x|^2/cl^2 against x.y/cl^2.  (a) coordinates offset by 1e3
    are centred and stay on the tensor-pipe prologue; (b) cl = 1e-3 exceeds the cancellation budget and is routed to the
    difference form; both hold 1e-9 against the oracle; (c) forcing the forms apart on a benign case gives the same
    scores; (d) the posterior-variance (TRSM) path takes the same decision."""
    from gpexp_b200 import kernels as K
    from gpexp_b200.device import prologue_operands
    rng = np.random.default_rng(12)
    L = gx._lib

    def run(kern, ks, cand, mc, design, noise, expect_mode):
        kern._bind(gx.dev)
        fam, d, params = kern._gpx_spec()
        eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), max(len(design), 1), noise,
                                         gx.engine.prior_scale(fam, params))
        eng.load_design(gx.engine.DesignFactor(gx.dev, gx.dev.points(design), noise))
        assert eng.prologue()[0] == expect_mode
        eng.score()
        w_m, var_m = orc.fast_design_state(ks, design, mc, noise)
        w_c, var_c = orc.fast_design_state(ks, design, cand, noise)
        ref = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, noise)
        got = eng.scores[: len(cand)].cpu().numpy()
        assert np.max(np.abs(got - ref) / np.abs(ref)) <= 1e-9
        assert int(eng.idx.item()) == int(np.argmin(ref))
        return got

    # (a) offset by 1e3, cl = 0.05 / 0.08: |alpha| would be ~1e8 without the centre
    off = np.array([1e3, -2e3])
    cand, mc = rng.uniform(-1, 1, (900, 2)) + off, rng.uniform(-1, 1, (1300, 2)) + off
    design = cand[rng.permutation(900)[:40]]
    run(K.KernelSquaredExponential([0.05, 0.08], 1.0, 2), orc.KernelSpec.se([0.05, 0.08], 1.0, 2), cand, mc, design, 1e-6,
        L.PRO_EXPANDED)
    run(K.KernelIsoMatern(0.7, 1.3, 2), orc.KernelSpec.matern32(0.7, 1.3, 2), cand, mc, design, 1e-6, L.PRO_EXPANDED)
    # (b) cl = 1e-3 on [-1,1]: alpha up to 5e5 -> difference form
    cand1, mc1 = rng.uniform(-1, 1, (1100, 1)), rng.uniform(-1, 1, (2500, 1))
    design1 = cand1[rng.permutation(1100)[:30]]
    run(K.KernelSquaredExponential([1e-3], 1.0, 1), orc.KernelSpec.se([1e-3], 1.0, 1), cand1, mc1, design1, 1e-6, L.PRO_DIFF)
    # (c) same benign problem through both forms
    cand2, mc2 = rng.uniform(-1, 1, (700, 3)), rng.uniform(-1, 1, (900, 3))
    design2 = cand2[:25]
    kern, ks = K.KernelMehlerND([0.6, 0.7, 0.5], 3), orc.KernelSpec.mehler([0.6, 0.7, 0.5], 3)
    a = run(kern, ks, cand2, mc2, design2, 1e-2, L.PRO_EXPANDED)
    gx.dev.force_diff_form = True
    try:
        b = run(kern, ks, cand2, mc2, design2, 1e-2, L.PRO_DIFF)
        # (d) posterior variance through the TRSM path in difference form
        g = gx.gp.GP(kern, 1e-2)
        g.addNodesAndComputeCovariance(design2)
        v_diff = g.evaluateVariance(mc2)
    finally:
        gx.dev.force_diff_form = False
    assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-11
    g = gx.gp.GP(kern, 1e-2)
    g.addNodesAndComputeCovariance(design2)
    v_exp = g.evaluateVariance(mc2)
    ref = orc.fast_posterior_variance(ks, design2, mc2, 1e-2)
    scale = np.abs(ref).max()
    assert np.max(np.abs(v_exp - ref)) <= 1e-10 * scale and np.max(np.abs(v_diff - ref)) <= 1e-10 * scale
    # offset coordinates through GP.evaluateVariance as well (centre = mid-range of the query set)
    kse, kso = K.KernelSquaredExponential([0.05, 0.08], 1.0, 2), orc.KernelSpec.se([0.05, 0.08], 1.0, 2)
    g = gx.gp.GP(kse, 1e-6)
    g.addNodesAndComputeCovariance(design)
    v = g.evaluateVariance(mc)
    ref = orc.fast_posterior_variance(kso, design, mc, 1e-6)
    assert np.max(np.abs(v - ref)) <= 1e-9


def test_ring_geometries_give_identical_scores(gx):
    """The lagged-group rings (gpx_set_ivar_ring 1, 2) only reorder when the two warp groups work; every candidate's
    sum is accumulated in the same order, so the scores are bit-identical to the in-step ring -- for d <= 14 (expanded
    form), d = 16 (difference form) and a K tail that is not a multiple of the chunk."""
    rng = np.random.default_rng(21)
    for name, d, n in [("se_ard_2d", 2, 45), ("matern_5d", 5, 16), ("se_ard_10d", 10, 131)]:
        k = bind(gx, name)
        fam, _, params = k._gpx_spec()
        cand, mc = rng.uniform(-1, 1, (1500, d)), rng.uniform(-1, 1, (2100, d))
        eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), n, 1e-4,
                                         gx.engine.prior_scale(fam, params))
        eng.load_design(gx.engine.DesignFactor(gx.dev, gx.dev.points(cand[:n]), 1e-4))
        outs = []
        try:
            for ring in (0, 1, 2):
                gx.check(gx.lib.gpx_set_ivar_ring(gx.dev.h, ring))
                eng.score()
                outs.append(eng.scores[:1500].cpu().numpy().copy())
        finally:
            gx.check(gx.lib.gpx_set_ivar_ring(gx.dev.h, 0))
        assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2]), name
        assert np.all(np.isfinite(outs[0]))


def test_singular_gram_is_jittered_loudly(gx):
    """ADVICE r1: noise 0.0 with a duplicated node makes the Gram singular; the reference's pinv shrugs, a Cholesky
    factor does not exist.  The GP path warns, factors K + jitter and returns finite variances that agree with the
    pseudo-inverse answer away from the null direction."""
    import warnings
    k = product_kernel("se_ard_2d_wide")
    rng = np.random.default_rng(3)
    nodes = rng.uniform(-1, 1, (12, 2))
    nodes[7] = nodes[2]
    q = rng.uniform(-1, 1, (200, 2))
    g = gx.gp.GP(k, 0.0)
    g.addNodesAndComputeCovariance(nodes)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        v = g.evaluateVariance(q)
    assert any(issubclass(x.category, gx.engine.GpxConditionWarning) for x in w)
    ks = spec("se_ard_2d_wide")
    Kdd = ks.gram(nodes, nodes)
    kq = ks.gram(nodes, q)
    ref = ks.prior(q) - np.einsum("iq,ij,jq->q", kq, np.linalg.pinv(Kdd), kq)
    assert np.all(np.isfinite(v)) and np.max(np.abs(v - ref)) <= 1e-6


def test_argreduce_nan_wins_like_numpy(gx):
    dev, lib, ptr, torch = gx.dev, gx.lib, gx.ptr, gx.torch
    v = np.random.default_rng(5).standard_normal(70001)
    v[[40000, 123]] = np.nan
    best, idx = dev.zeros(1), dev.zeros(1, dtype=torch.int64)
    for minimize in (0, 1):
        gx.check(lib.gpx_argreduce(dev.h, ptr(dev.upload(v)), None, None, v.size, minimize, ptr(best), ptr(idx), dev.stream))
        assert int(idx.item()) == 123 == int(np.argmax(v)) == int(np.argmin(v)) and np.isnan(best.item())


def test_mi_cost_function_caches_the_factorisation(gx, golden):
    """ADVICE r1: the reference's usage `for ind in options: costFuncMI.evaluate(ind, indKeep)` must not redo the O(|V|^3)
    set-up per call.  Scores equal the golden ones; the engine object survives; add_candidates invalidates it."""
    z = golden("greedy_mi")
    name = str(z["gmi/1/name"])
    k = product_kernel(name)
    pool, noise = z["gmi/1/pool"], float(z["gmi/1/noise"])
    idx, ref_scores = [int(i) for i in z["gmi/1/idx"]], z["gmi/1/scores"]
    cf = gx.ed.costFunctionGP_MI(gx.gp.GP(k, noise), len(idx), gx.Space(k.dimension, None, None), nmc=len(pool), mcpoints=pool)
    engines = set()
    for step in range(1, 4):
        keep = idx[:step]
        options = [j for j in range(len(pool)) if j not in keep]
        out = np.array([cf.evaluate(j, keep)[0] for j in options])
        engines.add(id(cf._mi_cache["engine"]))
        ref = ref_scores[step][options]
        assert np.max(np.abs(out - ref) / np.abs(ref)) <= 2e-8
        assert options[int(np.argmax(out))] == idx[step]
    assert len(engines) == 1
    # a list that does not extend the previous one replays on the same factorisation
    one = cf.evaluate(options[0], idx[:1])
    assert abs(one[0] - ref_scores[1][options[0]]) <= 2e-8 * abs(ref_scores[1][options[0]]) and id(cf._mi_cache["engine"]) in engines
    np.testing.assert_allclose(cf.invcov, z["gmi/1/invcov"], rtol=0, atol=1e-9 * np.abs(z["gmi/1/invcov"]).max())
    cf.add_candidates(len(pool) - 5, pool[:-5])
    cf.evaluate(0, [3])
    assert id(cf._mi_cache["engine"]) not in engines and cf._mi_cache["engine"].V == len(pool) - 5


def test_dgemm_tn_sub_lower_skips_only_structural_zeros(gx):
    """gpx_dgemm_tn_sub_lower (the Y = U^-T half of the MI set-up): B is one rank's block-cyclic column slice of a
    lower-triangular matrix; skipping the rows above each tile's global column must not change the product."""
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    rng = np.random.default_rng(17)
    V, B, world = 2304, 256, 3
    full = np.tril(rng.standard_normal((V, V)))                     # lower triangular V x V
    K, I = 1800, 256                                                # contraction over the first K rows, I output rows
    A = rng.standard_normal((K, I))
    for rank in range(world):
        blocks = list(range(rank, V // B, world))
        gcols = np.concatenate([np.arange(g * B, (g + 1) * B) for g in blocks])
        Bloc = full[:K, gcols]                                      # local slice (K x nloc)
        nloc = gcols.size
        ld = gx.device.roundup(nloc)
        Ad = dev.zeros(K, 256)
        Ad[:, :I] = dev.upload(A)
        Bd = dev.zeros(K, ld)
        Bd[:, :nloc] = dev.upload(Bloc)
        C0 = rng.standard_normal((I, nloc))
        outs = []
        for lower in (False, True):
            Cd = dev.zeros(I, ld)
            Cd[:, :nloc] = dev.upload(C0)
            if lower:
                gx.check(lib.gpx_dgemm_tn_sub_lower(dev.h, ptr(Ad), 256, ptr(Bd), ld, ptr(Cd), ld, I, nloc, K, B, world, rank,
                                                    dev.stream))
            else:
                gx.check(lib.gpx_dgemm_tn_sub_padded(dev.h, ptr(Ad), 256, ptr(Bd), ld, ptr(Cd), ld, I, nloc, K, 0, dev.stream))
            outs.append(Cd[:, :nloc].cpu().numpy())
        ref = C0 - A.T @ Bloc
        assert np.max(np.abs(outs[0] - ref)) <= 1e-11 * np.max(np.abs(ref))
        assert np.max(np.abs(outs[1] - ref)) <= 1e-11 * np.max(np.abs(ref)), rank


def test_round2_abi_edge_cases(gx):
    """Empty ranges, missing communicator, struct-size handshake and argument validation of the round-2 entry points."""
    import ctypes as C
    dev, lib, ptr, torch, L = gx.dev, gx.lib, gx.ptr, gx.torch, gx._lib
    bind(gx, "se_ard_2d")
    assert lib.gpx_state_bytes(0) == C.sizeof(L.IvarState) and lib.gpx_state_bytes(1) == C.sizeof(L.VarState)
    assert lib.gpx_state_bytes(7) == -1
    # collectives without gpx_comm_init answer GPX_ENOCOMM (-5), never crash
    a = dev.zeros(8)
    assert lib.gpx_comm_size(dev.h) in (0, 1) or lib.gpx_comm_size(dev.h) > 1
    if lib.gpx_comm_size(dev.h) == 0:
        assert lib.gpx_comm_allgather(dev.h, ptr(a), ptr(a), 4, dev.stream) == -5
        assert "gpx_comm_init" in L.last_error()
        assert lib.gpx_comm_bcast(dev.h, ptr(a), 4, 0, dev.stream) == -5
    # ring selection is validated
    assert lib.gpx_set_ivar_ring(dev.h, 3) == -1 and lib.gpx_set_ivar_ring(dev.h, 1) == 0
    # an empty step range is a no-op; a range beyond the capacity is refused
    rng = np.random.default_rng(2)
    k = bind(gx, "se_ard_2d")
    fam, d, params = k._gpx_spec()
    eng = gx.engine.GreedyIVAREngine(dev, dev.points(rng.uniform(-1, 1, (300, 2))), dev.points(rng.uniform(-1, 1, (500, 2))), 4,
                                     1e-6, gx.engine.prior_scale(fam, params))
    st = eng._state()
    assert lib.gpx_ivar_greedy_run(dev.h, C.byref(st), 0, 0, dev.stream) == 0
    assert lib.gpx_ivar_greedy_run(dev.h, C.byref(st), 0, 5, dev.stream) == -1 and "capacity" in L.last_error()
    assert lib.gpx_ivar_greedy_run(dev.h, None, 0, 1, dev.stream) == -1
    eng.run(4)
    assert len(set(int(i) for i in eng.indices())) == 4
    # Gram x vector: empty sides
    ws = dev.zeros(int(lib.gpx_gram_matvec_workspace(16)))
    out = dev.zeros(16)
    X = dev.points(rng.uniform(-1, 1, (16, 2)))
    assert lib.gpx_gram_matvec(dev.h, ptr(X.X), 0, X.ld, ptr(X.X), 16, X.ld, ptr(a), ptr(ws), ptr(out), dev.stream) == 0
    assert lib.gpx_gram_matvec(dev.h, ptr(X.X), 16, X.ld, None, 0, X.ld, None, ptr(ws), ptr(out), dev.stream) == 0
    assert float(out.abs().max().item()) == 0.0
    # the expanded form refuses d > 14 (the prepared side has d + 2 <= 16 rows); the difference form takes it
    k16 = product_kernel("se_ard_10d")
    from gpexp_b200 import kernels as K
    k16 = K.KernelSquaredExponential(list(np.linspace(0.5, 1.5, 16)), 1.0, 16)
    k16._bind(dev)
    P = dev.points(rng.uniform(-1, 1, (130, 16)))
    rows = dev.zeros(16, P.ld)
    assert lib.gpx_prep_side(dev.h, 0, ptr(P.X), 130, P.ld, ptr(rows), P.ld, None, dev.stream) == -4   # GPX_ESIZE
    from gpexp_b200.device import prologue_operands
    assert prologue_operands(P, P)[0] == L.PRO_DIFF
    # block-cyclic helpers validate their description
    assert lib.gpx_dgemm_tn_sub_lower(dev.h, ptr(a), 128, ptr(a), 128, ptr(a), 128, 1, 1, 1, 100, 2, 0, dev.stream) == -1
    assert lib.gpx_local_index_cyclic(dev.h, ptr(a), 256, 2, 2, 10, ptr(dev.zeros(2, dtype=torch.int64)), dev.stream) == -1


def test_reference_hyperparameter_fit_runs_on_the_patched_gp(gx, patched_ref):
    """GP.findOptParamsLogLike (gp.py:498-639) is NOT re-implemented: the reference's own L-BFGS-B loop (finite-difference
    gradient, step 1e-8) calls the patched loglikeParams.  Its end point is determined by round-off at the 1e-10 level of
    the objective (DESIGN.md section 8), so the check is the optimiser's contract, not a golden vector: bounds respected,
    the marginal likelihood does not decrease, the GP is left with the returned hyper-parameters, and every objective value
    on the way equals the oracle's to 1e-9."""
    r = patched_ref
    rng = np.random.default_rng(31)
    X = rng.uniform(-1, 1, (40, 2))
    y = np.sin(3 * X[:, 0]) * np.cos(2 * X[:, 1]) + 1e-3 * rng.standard_normal(40)
    k = r.kernels.KernelSquaredExponential([0.5, 0.5], 1.0, 2)
    g = r.gp.GP(k, 1e-5)
    start = g.loglikeParams(X, y)
    assert abs(start - orc.fast_loglike(orc.KernelSpec.se([0.5, 0.5], 1.0, 2), X, y, 1e-5)) <= 1e-9 * abs(start)
    params, neg = _quiet(g.findOptParamsLogLike, X, y, maxiter=30)
    assert set(params) == {'cl0', 'cl1', 'signalSize', 'noise'}
    assert 0.05 - 1e-12 <= params['cl0'] <= 5.0 + 1e-12 and 1e-12 <= params['noise'] <= 1.0
    assert -neg >= start - 1e-9
    assert g.kernel.hyperParam['cl1'] == params['cl1'] and g.noise == params['noise']
    end = g.loglikeParams(X, y)
    ks = orc.KernelSpec.se([params['cl0'], params['cl1']], params['signalSize'], 2)
    assert abs(end - orc.fast_loglike(ks, X, y, float(params['noise']))) <= 1e-8 * abs(end)


def test_one_kernel_loop_equals_multi_launch_loop(gx):
    """gpx_ivar_greedy_small (whole loop in one cooperative kernel) against gpx_ivar_greedy_run on the same resident state:
    identical picks, pivots and factor rows; scores to 1e-13; continuing a design started by the other path works (the
    state conventions are shared); all three kernel families."""
    if gx.engine.GreedyIVAREngine.ONE_KERNEL_DEFAULT == 0 and not os.environ.get("GPX_TEST_ONE_KERNEL"):
        pytest.skip("one-kernel loop is opt-in (GPX_ONE_KERNEL_PAIRS); set GPX_TEST_ONE_KERNEL=1 to test it")
    rng = np.random.default_rng(5)
    for name, noise, C, M, N in [("se_iso_1d", 1e-6, 1000, 10000, 20), ("matern_5d", 1e-4, 777, 1501, 33),
                                 ("mehler_3d", 1e-2, 500, 900, 12)]:
        ks = spec(name)
        k = bind(gx, name)
        samp = rng.standard_normal if name.startswith("mehler") else (lambda s: rng.uniform(-1, 1, s))
        cand, mc = samp((C, ks.dim)), samp((M, ks.dim))
        fam, d, params = k._gpx_spec()
        scale = gx.engine.prior_scale(fam, params)
        res = []
        limit = 32_000_000
        for pairs in (limit, 0):
            eng = gx.engine.GreedyIVAREngine(gx.dev, gx.dev.points(cand), gx.dev.points(mc), N, noise, scale, resident=True)
            eng.ONE_KERNEL_PAIRS = pairs
            eng.run(N // 2)
            eng.ONE_KERNEL_PAIRS = limit - pairs   # switch paths mid-design
            eng.run(N)
            res.append((eng.indices(), eng.pivots(), eng.Wc[:N, :C].cpu().numpy(), eng.pick_scores[:N].cpu().numpy(),
                        eng.scores[:C].cpu().numpy()))
        assert np.array_equal(res[0][0], res[1][0]), name
        np.testing.assert_allclose(res[0][1], res[1][1], rtol=1e-12, atol=0)
        np.testing.assert_allclose(res[0][2], res[1][2], rtol=1e-11, atol=1e-13)
        np.testing.assert_allclose(res[0][3], res[1][3], rtol=1e-12, atol=0)
        np.testing.assert_allclose(res[0][4], res[1][4], rtol=1e-12, atol=0)
        ref, _ = orc.fast_greedy_ivar(ks, cand, mc, N, noise)
        assert [int(i) for i in res[0][0]] == ref, name
