"""Closed-form IVAR over a box or Gaussian measure (squared-exponential kernels).

CPU: the oracle's Phi against mpmath quadrature of the 1-D factor, the oracle's exact cost against scipy quadrature of the
posterior variance and against a 4-million-point Monte-Carlo estimate, and every rejected combination of the public API.
GPU: gpx_phi_gram against mpmath at 50 digits (tails, flush, block edges with sentinels), evaluate /
scoreCandidatesIVAR / the greedy loop against the oracle, a noise function, and run-to-run identity.

Score bound (tests/measure_oracle.py, fast_ivar_scores_measure): q_c = Phi_cc - 2 w.z + w.y cancels in absolute terms, so a score is
compared within 4 x bound_c,  bound_c = (n + 3) eps [(Phi_cc + 2 sum|w||z| + sum|w||y|) / (var_D(c) + nu_c) + (n + 1) s],
not within a flat relative 1e-9; a pick must be the oracle's arg-min unless the two lie within their tolerances.  The
bound covers rounding only: the designs here keep cond(K_DD + noise I) <= 1e4, below which the forward errors of the two
factorisations (~ cond eps) stay inside it."""
import math

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests import measure_oracle as mo

EPS = float(np.finfo(np.float64).eps)


# ---- CPU: the oracle ----------------------------------------------------------------------------------------------------
def _mp_box_factor(lo, hi, cl, m):
    import mpmath as mp
    mp.mp.dps = 40
    f = lambda x: mp.exp(-((x - m) / cl) ** 2)  # noqa: E731
    pts = sorted({mp.mpf(lo), mp.mpf(hi)} | {mp.mpf(p) for p in (m - 30 * cl, m, m + 30 * cl) if lo < p < hi})
    return mp.quad(f, pts) / (hi - lo)


def _mp_gauss_factor(mu, sd, cl, m):
    import mpmath as mp
    mp.mp.dps = 40
    f = lambda x: mp.exp(-((x - m) / cl) ** 2 - ((x - mu) / sd) ** 2 / 2) / (sd * mp.sqrt(2 * mp.pi))  # noqa: E731
    pts = sorted({mp.mpf(p) for p in (mu - 30 * sd, mu, mu + 30 * sd, m - 30 * cl, m, m + 30 * cl)})
    return mp.quad(f, [-mp.inf] + pts + [mp.inf])


@pytest.mark.parametrize("cl", [1e-3, 3e-2, 1.0, 30.0, 1e3])
def test_box_factor_matches_mpmath(cl):
    """I(m) of U[-1, 1] (measure_phi at x = y = m, s = 1) inside, at the edge, up to 5 cl outside and far outside."""
    kern = orc.KernelSpec.se([cl], 1.0, 1)
    meas = mo.MeasureSpec.box([-1.0], [1.0])
    centres = [0.0, 0.37, -0.999, 1.0, -1.0, 1.0 + 0.5 * cl, -1.0 - 2.0 * cl, 1.0 + 5.0 * cl, 3.0 * cl + 1.0, 40.0 * cl]
    for m in centres:
        got = mo.measure_phi(kern, meas, [[m]], [[m]])[0, 0]
        want = float(_mp_box_factor(-1.0, 1.0, cl, m))
        if want < 1e-290:
            continue   # (40 cl for small cl) below the representable range: flushed, tested on the GPU side
        assert abs(got - want) <= 1e-13 * want, (cl, m, got, want)


@pytest.mark.parametrize("cl", [1e-3, 1.0, 1e3])
@pytest.mark.parametrize("sd", [1e-3, 1.0, 1e3])
def test_gauss_factor_matches_mpmath(cl, sd):
    kern = orc.KernelSpec.se([cl], 1.0, 1)
    mu = 0.25
    meas = mo.MeasureSpec.gauss([mu], [sd])
    scale = math.sqrt(cl * cl + 2 * sd * sd)
    for m in (mu, mu + 0.5 * scale, mu - 2.0 * scale, mu + 4.0 * scale):
        got = mo.measure_phi(kern, meas, [[m]], [[m]])[0, 0]
        want = float(_mp_gauss_factor(mu, sd, cl, m))
        assert abs(got - want) <= 1e-13 * want, (cl, sd, m, got, want)


def _posterior_var(kern, design, noise):
    from scipy.linalg import cho_factor, cho_solve
    K = kern.gram(design, design) + noise * np.eye(len(design))
    cf = cho_factor(K)
    return lambda *x: kern.signal - float(kern.gram(design, np.array([x]))[:, 0] @ cho_solve(cf, kern.gram(design, np.array([x]))[:, 0]))


@pytest.mark.parametrize("kind", ["box", "gauss"])
def test_cost_1d_matches_quadrature(kind):
    from scipy import integrate
    kern = orc.KernelSpec.se([0.3], 1.3, 1)
    design = np.array([[-0.7], [0.1], [0.45], [0.9]])
    var = _posterior_var(kern, design, 1e-6)
    if kind == "box":
        meas = mo.MeasureSpec.box([-1.0], [1.0])
        want = integrate.quad(var, -1.0, 1.0, points=design[:, 0], epsabs=1e-14, epsrel=1e-13, limit=200)[0] / 2.0
    else:
        meas = mo.MeasureSpec.gauss([0.2], [0.6])
        dens = lambda x: math.exp(-0.5 * ((x - 0.2) / 0.6) ** 2) / (0.6 * math.sqrt(2 * math.pi))  # noqa: E731
        want = integrate.quad(lambda x: var(x) * dens(x), -8.0, 8.0, points=design[:, 0], epsabs=1e-14, epsrel=1e-13,
                              limit=200)[0]
    got = mo.fast_ivar_cost_measure(kern, meas, design, 1e-6)
    assert abs(got - want) <= 1e-9, (got, want)


@pytest.mark.parametrize("kind", ["box", "gauss"])
def test_cost_2d_matches_quadrature(kind):
    from scipy import integrate
    kern = orc.KernelSpec.se([0.4, 0.6], 1.0, 2)
    design = np.array([[-0.5, 0.2], [0.3, -0.4], [0.6, 0.7]])
    var = _posterior_var(kern, design, 1e-4)
    opts = {"epsabs": 1e-13, "epsrel": 1e-12, "limit": 100}
    if kind == "box":
        meas = mo.MeasureSpec.box([-1.0, -0.5], [1.0, 1.5])
        want = integrate.nquad(var, [[-1.0, 1.0], [-0.5, 1.5]], opts=opts)[0] / 4.0
    else:
        meas = mo.MeasureSpec.gauss([0.1, -0.2], [0.4, 0.5])
        dens = lambda x, y: math.exp(-0.5 * ((x - 0.1) / 0.4) ** 2 - 0.5 * ((y + 0.2) / 0.5) ** 2) / (2 * math.pi * 0.2)  # noqa: E731
        want = integrate.nquad(lambda x, y: var(x, y) * dens(x, y), [[-3.3, 3.5], [-4.2, 3.8]], opts=opts)[0]
    got = mo.fast_ivar_cost_measure(kern, meas, design, 1e-4)
    assert abs(got - want) <= 1e-9, (got, want)


@pytest.mark.parametrize("kind", ["box", "gauss"])
def test_cost_within_five_standard_errors_of_4m_monte_carlo(kind):
    rng = np.random.default_rng(11)
    kern = orc.KernelSpec.se([0.06, 0.09], 1.0, 2)
    design = rng.uniform(-1.0, 1.0, (40, 2))
    if kind == "box":
        meas, draw = mo.MeasureSpec.box([-1.0, -1.0], [1.0, 1.0]), lambda n: rng.uniform(-1.0, 1.0, (n, 2))
    else:
        meas, draw = mo.MeasureSpec.gauss([0.0, 0.1], [0.3, 0.4]), lambda n: rng.normal([0.0, 0.1], [0.3, 0.4], (n, 2))
    s1 = s2 = 0.0
    M = 4_000_000
    for _ in range(8):
        v = orc.fast_posterior_variance(kern, design, draw(M // 8), 1e-6)
        s1 += v.sum()
        s2 += (v * v).sum()
    mean = s1 / M
    se = math.sqrt((s2 / M - mean * mean) / M)
    exact = mo.fast_ivar_cost_measure(kern, meas, design, 1e-6)
    assert abs(mean - exact) <= 5 * se, (mean, exact, se)


# ---- CPU: rejected combinations (all raise before any device work) ----------------------------------------------------------
def _cf(kern, measure, **kw):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import Space
    return ed.costFunctionGP_IVAR(gp.GP(kern, 1e-6), 3, Space(2, None, None), measure=measure, **kw)


def test_measure_constructors_reject_bad_parameters():
    from gpexp_b200.approximation import GaussianMeasure, UniformMeasure
    for bad in (lambda: UniformMeasure([0.0, 1.0], [1.0, 1.0]), lambda: UniformMeasure([0.0], [np.inf]),
                lambda: GaussianMeasure([0.0], [0.0]), lambda: GaussianMeasure([np.nan], [1.0]),
                lambda: UniformMeasure([0.0, 0.0, 0.0], [1.0, 1.0])):
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(ValueError, match="UniformMeasure"):
        UniformMeasure([-1.0, -1.0, -1.0], 1.0).params(2)


def test_rejected_combinations_name_the_measure():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import kernels
    from gpexp_b200.approximation import GaussianMeasure, UniformMeasure
    se = kernels.KernelSquaredExponential([0.2, 0.3], 1.0, 2)
    cand = np.zeros((10, 2))
    for meas in (UniformMeasure(-1.0, 1.0), GaussianMeasure(0.0, 0.5)):
        name = type(meas).__name__
        cf = _cf(se, meas, mcPoints=np.zeros((5, 2)), mcWeights=np.ones(5))
        with pytest.raises(ValueError, match=name):
            cf.evaluate(np.zeros((3, 2)))
        with pytest.raises(ValueError, match=name):
            ed.performGreedyIVARExperimentalDesign(cf, cand, 2)
        cf = _cf(kernels.KernelIsoMatern(0.2, 1.0, 2), meas)
        with pytest.raises(NotImplementedError, match=name):
            cf.evaluate(np.zeros((3, 2)))
        with pytest.raises(NotImplementedError, match=name):
            ed.performGreedyIVARExperimentalDesign(cf, cand, 2)
        cf = _cf(se, meas)
        with pytest.raises(NotImplementedError, match=name):
            cf.derivative(np.zeros((3, 2)))
        with pytest.raises(NotImplementedError, match=name):
            ed.performGreedyIVARExperimentalDesign(cf, cand, 2, shard=object())
        with pytest.raises(NotImplementedError, match=name):
            ed.beginGreedyIVARExperimentalDesign(cf, cand, 2, resident=True)
        with pytest.raises(NotImplementedError, match=name):
            ed.scoreCandidatesIVAR(cf, np.zeros((2, 2)), cand, shard=object())
        with pytest.raises(NotImplementedError, match=name):
            ed.refineGreedyIVARExperimentalDesign(cf, cand, [0, 1])


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _mp_phi(kind, cl, s, p0, p1, x, y):
    """Phi(x, y) from the closed form at 50 digits (the double inputs taken as exact)."""
    import mpmath as mp
    mp.mp.dps = 50
    out = mp.mpf(s) ** 2
    for q in range(len(cl)):
        c, a, b = mp.mpf(cl[q]), mp.mpf(x[q]), mp.mpf(y[q])
        m = (a + b) / 2
        out *= mp.exp(-(a - b) ** 2 / (4 * c * c))
        if kind == mo.BOX:
            lo, hi = mp.mpf(p0[q]), mp.mpf(p1[q])
            u, v = (lo - m) / c, (hi - m) / c
            # erf(v) - erf(u) as an erfc difference on one side of 0: the tails of erf cancel against 1 at any precision
            diff = mp.erfc(u) - mp.erfc(v) if u >= 0 else mp.erfc(-v) - mp.erfc(-u) if v <= 0 else mp.erf(v) - mp.erf(u)
            out *= c * mp.sqrt(mp.pi) / (2 * (hi - lo)) * diff
        else:
            mu, sd = mp.mpf(p0[q]), mp.mpf(p1[q])
            out *= (1 + 2 * sd * sd / (c * c)) ** mp.mpf(-0.5) * mp.exp(-(m - mu) ** 2 / (c * c + 2 * sd * sd))
    return out


def _phi_device(dev, X, Y, ld=None, fill=None):
    from gpexp_b200 import _lib
    from gpexp_b200.device import ptr
    A, B = dev.points(X), dev.points(Y)
    ld = ld or B.ld
    rows = A.n + 2
    out = dev.zeros(rows, ld)
    if fill is not None:
        out.fill_(fill)
    _lib.check(_lib.lib.gpx_phi_gram(dev.h, ptr(A.X), A.n, A.ld, ptr(B.X), B.n, B.ld, ptr(out), ld, dev.stream), "gpx_phi_gram")
    return out.cpu().numpy()


def _bind(kern_spec, kind, p0, p1):
    import ctypes as C
    from gpexp_b200 import _lib
    from gpexp_b200.device import Device
    dev = Device.get()
    dev.set_kernel(_lib.SE, kern_spec.dim, kern_spec.packed_params())
    dbl = C.POINTER(C.c_double)
    a, b = np.ascontiguousarray(p0, dtype=np.float64), np.ascontiguousarray(p1, dtype=np.float64)
    _lib.check(_lib.lib.gpx_set_measure(dev.h, kind, kern_spec.dim, a.ctypes.data_as(dbl), b.ctypes.data_as(dbl)),
               "gpx_set_measure")
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [mo.BOX, mo.GAUSS])
def test_phi_gram_matches_mpmath_within_ulp_bound(kind):
    """|got - exact| <= (64 + 8 |log(Phi / pref)|) ulp: the log term is the sensitivity of e^S (and of the erfcx tails) to
    the rounding of its arguments.  Probes run from coincident points to far tails; below 2^-1022 the result is 0."""
    rng = np.random.default_rng(5)
    cl, s = np.array([0.05, 0.8, 3.0]), 1.7
    p0, p1 = (np.array([-1.0, -0.5, 0.0]), np.array([1.0, 2.0, 0.25])) if kind == mo.BOX else \
        (np.array([0.1, -0.3, 0.0]), np.array([0.2, 1.5, 1e-3]))
    kern = orc.KernelSpec.se(cl, s, 3)
    dev = _bind(kern, kind, p0, p1)
    X = np.concatenate([rng.uniform(-1.5, 1.5, (40, 3)), [[1.0, 2.0, 0.25], [-1.0, -0.5, 0.0], [1.2, 2.5, 0.4],
                                                          [1.35, 3.0, 2.0]]])
    Y = np.concatenate([X[::3] + rng.normal(0, 0.02, X[::3].shape), [[1.3, 3.5, 3.0]]])
    got = _phi_device(dev, X, Y)
    for i in range(len(X)):
        for j in range(len(Y)):
            exact = _mp_phi(kind, cl, s, p0, p1, X[i], Y[j])
            if exact < 2.0 ** -1022:
                assert got[i, j] == 0.0, (i, j, got[i, j], exact)   # flushed as k is
                continue
            pref = float(s * s) if kind == mo.BOX else s * s * np.prod((1 + 2 * p1 ** 2 / cl ** 2) ** -0.5)
            tol = (64 + 8 * abs(math.log(float(exact) / pref))) * EPS * float(exact)
            assert abs(got[i, j] - float(exact)) <= tol, (i, j, got[i, j], float(exact))
    # the far probe against the origin-side corner lies far below 2^-1022 and must be an exact zero
    flush = _phi_device(dev, [[1.3, 3.5, 3.0]], [[-1.4, -1.0, -3.0]])
    assert flush[0, 0] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("ncols", [255, 256, 257])
def test_block_edges_keep_padding(ncols):
    """Sentinels in the output padding stay untouched by gpx_phi_gram, gpx_phi_diag and gpx_phi_append_row."""
    from gpexp_b200 import _lib
    from gpexp_b200.device import ptr, roundup
    rng = np.random.default_rng(ncols)
    kern = orc.KernelSpec.se([0.3, 0.2], 1.0, 2)
    meas = mo.MeasureSpec.box([-1.0, -1.0], [1.0, 1.0])
    dev = _bind(kern, mo.BOX, meas.p0, meas.p1)
    X, Y = rng.uniform(-1, 1, (7, 2)), rng.uniform(-1, 1, (ncols, 2))
    S = -7.25
    ld = roundup(ncols) + 128
    got = _phi_device(dev, X, Y, ld=ld, fill=S)
    want = mo.measure_phi(kern, meas, X, Y)
    assert np.max(np.abs(got[:7, :ncols] - want) / want) <= 1e-13
    assert np.all(got[:7, ncols:] == S) and np.all(got[7:] == S)
    P = dev.points(Y)
    diag = dev.zeros(ld).fill_(S)
    _lib.check(_lib.lib.gpx_phi_diag(dev.h, ptr(P.X), ncols, P.ld, ptr(diag), dev.stream), "gpx_phi_diag")
    diag = diag.cpu().numpy()
    assert np.max(np.abs(diag[:ncols] - mo.measure_phi_diag(kern, meas, Y)) / diag[:ncols]) <= 1e-13
    assert np.all(diag[ncols:] == S)
    # one Z row from a 3-row Z: rows 0..2 arbitrary, pivot column l, x_p = Y[5]
    n = 3
    Z = dev.upload(np.concatenate([rng.normal(size=(n, P.ld)), np.full((2, P.ld), S)]))
    rec = np.zeros(_lib.GPX_PIVOT_HDR + n)
    rec[2], rec[3:5] = 0.49, Y[5]
    rec[_lib.GPX_PIVOT_HDR:] = rng.normal(size=n)
    zh = Z.cpu().numpy()
    _lib.check(_lib.lib.gpx_phi_append_row(dev.h, ptr(dev.upload(rec)), ptr(P.X), ncols, P.ld, ptr(Z), P.ld, n, dev.stream),
               "gpx_phi_append_row")
    z = Z.cpu().numpy()
    row = (mo.measure_phi(kern, meas, Y[5:6], Y)[0] - rec[_lib.GPX_PIVOT_HDR:] @ zh[:n, :ncols]) / 0.7
    assert np.max(np.abs(z[n, :ncols] - row)) <= 1e-14 * np.max(np.abs(row)) * 8
    pad = ncols + (ncols & 1)      # an odd count writes one zero column to complete its 16-byte pair
    assert np.all(z[n, ncols:pad] == 0.0) and np.all(z[n, pad:] == S) and np.all(z[n + 1] == S)
    assert np.array_equal(z[:n], zh[:n])


CASES = {
    "1d_iso": (orc.KernelSpec.se([0.1], 1.0, 1), 1, 600),
    "2d_ard": (orc.KernelSpec.se([0.06, 0.09], 1.0, 2), 2, 1500),
    "5d": (orc.KernelSpec.se([0.8, 0.9, 1.0, 1.1, 1.2], 1.3, 5), 5, 1500),
}


def _measures(d):
    from gpexp_b200.approximation import GaussianMeasure, UniformMeasure
    return {"box": (UniformMeasure(-1.0, 1.0), mo.MeasureSpec.box([-1.0] * d, [1.0] * d)),
            "gauss": (GaussianMeasure([0.1] * d, [0.5] * d), mo.MeasureSpec.gauss([0.1] * d, [0.5] * d))}


def _kernel(spec):
    from gpexp_b200 import kernels
    return kernels.KernelSquaredExponential(list(spec.cl), spec.signal, spec.dim)


def _check_greedy(spec, ometa, cand, idx, scores, nu):
    """Along the device's own picks: the recorded score of every pick within 4 x bound of the oracle's exact score of
    design + pick, and the pick the oracle's arg-min unless the oracle's winning gap lies within the tolerance (a near
    tie, counted and returned)."""
    nu = np.broadcast_to(np.asarray(nu, dtype=np.float64), (len(cand),))
    ties = 0
    for t, p in enumerate(idx):
        d = list(idx[:t])
        want, bound = mo.fast_ivar_scores_measure(spec, ometa, cand[d], cand, nu[d], nu)
        tol = 4 * bound
        assert abs(scores[t] - want[p]) <= tol[p], (t, scores[t], want[p], tol[p])
        best = int(np.argmin(want))
        if p != best:
            assert want[p] - want[best] <= tol[p] + tol[best], (t, p, best, want[p], want[best])
            ties += 1
    return ties


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("mname", ["box", "gauss"])
def test_greedy_evaluate_and_scoring_match_oracle(case, mname):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import Space
    ed.VERBOSE = False
    spec, d, C = CASES[case]
    meas, ometa = _measures(d)[mname]
    cand = np.random.default_rng(d).uniform(-1.0, 1.0, (C, d))
    N = 20
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel(spec), 1e-6), 4, Space(d, None, None), measure=meas)
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, N, returnIndices=True)
    idx = [int(i) for i in idx]
    assert _check_greedy(spec, ometa, cand, idx, cf.lastScores, 1e-6) <= 2
    assert cf.illConditionedFrom is None and np.all(cf.lastPivots > 0)
    # a given design: scoreCandidatesIVAR (Gram + Cholesky + TRSM + Phi Gram + DMMA) against the direct oracle
    design = cand[idx[:8]]
    costs, best = ed.scoreCandidatesIVAR(cf, design, cand)
    want, bound = mo.fast_ivar_scores_measure(spec, ometa, design, cand, 1e-6)
    assert np.all(np.abs(costs - want) <= 4 * bound), np.max(np.abs(costs - want) / bound)
    assert costs[best] == np.min(costs)
    # evaluate: the exact cost of a design, s - tr Psi
    cost = cf.evaluate(cand[idx[:4]])
    exact = mo.fast_ivar_cost_measure(spec, ometa, cand[idx[:4]], 1e-6)
    assert abs(cost - exact) <= 4 * 7 * 5 * EPS * spec.signal, (cost, exact)


@pytest.mark.gpu
def test_noise_function():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import GaussianMeasure, Space
    ed.VERBOSE = False
    spec = orc.KernelSpec.se([0.15, 0.25], 1.0, 2)
    cand = np.random.default_rng(9).uniform(-1.0, 1.0, (1200, 2))
    nf = lambda x: 1e-4 * (1.0 + x[:, 0] ** 2)  # noqa: E731
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel(spec), 1e-6), 3, Space(2, None, None, noise=nf),
                                measure=GaussianMeasure([0.0, 0.2], [0.5, 0.4]))
    ometa = mo.MeasureSpec.gauss([0.0, 0.2], [0.5, 0.4])
    idx = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf, cand, 15, returnIndices=True)]
    assert _check_greedy(spec, ometa, cand, idx, cf.lastScores, nf(cand)) <= 2
    design = cand[idx[:3]]
    costs, _ = ed.scoreCandidatesIVAR(cf, design, cand)
    want, bound = mo.fast_ivar_scores_measure(spec, ometa, design, cand, nf(design), nf(cand))
    assert np.all(np.abs(costs - want) <= 4 * bound)
    exact = mo.fast_ivar_cost_measure(spec, ometa, design, nf(design))
    assert abs(cf.evaluate(design) - exact) <= 1e-13


@pytest.mark.gpu
def test_run_to_run_identical():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import Space, UniformMeasure
    ed.VERBOSE = False
    spec = orc.KernelSpec.se([0.06, 0.09], 1.0, 2)
    cand = np.random.default_rng(1).uniform(-1.0, 1.0, (5000, 2))
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel(spec), 1e-6), 3, Space(2, None, None), measure=UniformMeasure(-1.0, 1.0))
    runs = []
    for _ in range(2):
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, 30)
        eng.score_trace = []
        eng.run(30)
        runs.append((eng.indices(), np.stack(eng.score_trace)))
    assert np.array_equal(runs[0][0], runs[1][0])
    assert np.array_equal(runs[0][1], runs[1][1])
    a, _ = ed.scoreCandidatesIVAR(cf, cand[:40], cand)
    b, _ = ed.scoreCandidatesIVAR(cf, cand[:40], cand)
    assert np.array_equal(a, b)
