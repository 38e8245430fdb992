"""Closed-form IVAR over a box or Gaussian measure for Mehler kernels (KernelMehler1D, KernelMehlerND).

CPU: the oracle (tests/mehler_measure_oracle.py) against mpmath quadrature of the 1-D factor and of s = int k(x, x) dmu,
the Mercer identity Phi_{N(0,1)} = k_{t^2}, the exact cost against scipy quadrature of the posterior variance, and the
rejection of a Gaussian measure too wide for s to be finite.
GPU: gpx_phi_gram against mpmath at 50 digits within (64 + 8 sum|exponent terms|) ulp, block edges with sentinels, the
Mercer identity against gpx_gram, evaluate / scoreCandidatesIVAR / the greedy loop against the oracle within 4x its
rounding bound (tests/test_ivar_measure.py explains the bound; the designs here keep cond(K_DD + noise I) <= 1e4), the
weighted path with tensor quadrature, run-to-run identity, GPX_EINVAL for an s that is not finite, and the reference's own
KernelMehlerND under install_as_gpExp."""
import math

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests import mehler_measure_oracle as mo

EPS = float(np.finfo(np.float64).eps)
T_VALUES = [0.0, 0.05, -0.05, 0.3, 0.6, 0.9, 0.99]


def _mp_k(t, x, y):
    import mpmath as mp
    r = 1 - t * t
    return mp.exp(-(t * t * x * x - 2 * t * x * y + t * t * y * y) / (2 * r)) / mp.sqrt(r)


def _mp_factor(kind, t, p0, p1, a, b):
    """int k(x, a) k(x, b) dmu(x) in one dimension by mpmath quadrature (the double inputs taken as exact).  The
    integrand is exp(-A (x - x*)^2 + const); the breakpoints lie where it has fallen by 2^-2 .. 2^10 below its largest
    value on the range, so that every subinterval sees a bounded change of the exponent, and the integrand is divided by
    that value (mpmath's error target is absolute)."""
    import mpmath as mp
    mp.mp.dps = 40
    t, a, b, p0, p1 = (mp.mpf(v) for v in (t, a, b, p0, p1))
    f = lambda x: _mp_k(t, x, a) * _mp_k(t, x, b)  # noqa: E731
    r, m = 1 - t * t, (a + b) / 2
    levels = [mp.mpf(2) ** k for k in range(-2, 11)]
    if kind == mo.BOX:
        if t == 0:
            return mp.quad(f, [p0, p1]) / (p1 - p0)
        A, xs = t * t / r, m / t
        d0 = (min(max(xs, p0), p1) - xs) ** 2
        cut = {xs + sg * mp.sqrt(d0 + k / A) for k in levels for sg in (-1, 1)}
        pts = sorted({p0, p1} | {x for x in cut if p0 < x < p1})
        top = f(min(max(xs, p0), p1))
        return mp.quad(lambda x: f(x) / top, pts) / (p1 - p0) * top
    dens = lambda x: mp.exp(-((x - p0) / p1) ** 2 / 2) / (p1 * mp.sqrt(2 * mp.pi))  # noqa: E731
    A = t * t / r + 1 / (2 * p1 * p1)
    xs = (t * m / r + p0 / (2 * p1 * p1)) / A
    pts = sorted({xs} | {xs + sg * mp.sqrt(k / A) for k in levels for sg in (-1, 1)})
    top = f(xs) * dens(xs)
    return mp.quad(lambda x: f(x) * dens(x) / top, [-mp.inf] + pts + [mp.inf]) * top


@pytest.mark.parametrize("t", T_VALUES)
@pytest.mark.parametrize("kind", [mo.BOX, mo.GAUSS])
def test_factor_matches_mpmath(t, kind):
    """1-D Phi(a, b) for a, b inside, at the edge of and far outside U[-1, 1.5], and around N(0.2, 0.8^2)."""
    kern = orc.KernelSpec.mehler([t], 1)
    meas = mo.MeasureSpec.box([-1.0], [1.5]) if kind == mo.BOX else mo.MeasureSpec.gauss([0.2], [0.8])
    pairs = [(0.0, 0.0), (0.3, -0.7), (1.5, 1.5), (-1.0, 1.5), (1.4, 1.6), (3.0, 3.2), (-4.0, -3.5), (7.0, 6.0),
             (-6.0, 5.0), (8.0, 8.5)]
    for a, b in pairs:
        got = mo.mehler_phi(kern, meas, [[a]], [[b]])[0, 0]
        want = float(_mp_factor(kind, t, meas.p0[0], meas.p1[0], a, b))
        if want < 1e-290:
            assert got == 0.0 or abs(got - want) <= 1e-13 * want, (t, a, b, got, want)
            continue
        assert abs(got - want) <= 1e-13 * want, (t, kind, a, b, got, want)


def _mp_prior(kind, t, p0, p1):
    import mpmath as mp
    mp.mp.dps = 40
    t, p0, p1 = mp.mpf(t), mp.mpf(p0), mp.mpf(p1)
    f = lambda x: _mp_k(t, x, x)  # noqa: E731
    if kind == mo.BOX:
        return mp.quad(f, mp.linspace(p0, p1, 9)) / (p1 - p0)
    dens = lambda x: mp.exp(-((x - p0) / p1) ** 2 / 2) / (p1 * mp.sqrt(2 * mp.pi))  # noqa: E731
    return mp.quad(lambda x: f(x) * dens(x), [-mp.inf] + [p0 + k * p1 for k in (-40, -10, 0, 10, 40)] + [mp.inf])


@pytest.mark.parametrize("t", [0.0, 0.3, 0.9, 0.99, -0.05, -0.6, -0.95])
def test_prior_matches_mpmath(t):
    """s = int k(x, x) dmu for c = t / (1 + t) > 0, < 0 and = 0, over boxes across 0, on one side, narrow and far out,
    and Gaussians inside the admissible width."""
    kern = orc.KernelSpec.mehler([t], 1)
    boxes = [(-1.0, 1.0), (0.2, 0.25), (-3.0, -2.0), (2.0, 6.0), (-0.5, 4.0), (5.0, 5.001)]
    for lo, hi in boxes:
        got = mo.mehler_prior(kern, mo.MeasureSpec.box([lo], [hi]))
        want = float(_mp_prior(mo.BOX, t, lo, hi))
        assert abs(got - want) <= 1e-13 * want, (t, lo, hi, got, want)
    limit = math.sqrt((1 + t) / (2 * t)) if t > 0 else math.inf
    for mu, sd in [(0.0, 1.0), (0.7, 0.3), (-1.5, 0.9)]:
        if sd >= limit:
            continue
        got = mo.mehler_prior(kern, mo.MeasureSpec.gauss([mu], [sd]))
        want = float(_mp_prior(mo.GAUSS, t, mu, sd))
        assert abs(got - want) <= 1e-13 * want, (t, mu, sd, got, want)


def test_too_wide_gaussian_raises():
    """s is infinite for 2 c sd^2 >= 1; the oracle and the public API say so before any device work, naming the measure,
    the dimension and the largest admissible std."""
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp, kernels
    from gpexp_b200.approximation import GaussianMeasure, Space
    kern = orc.KernelSpec.mehler([0.2, 0.9], 2)
    with pytest.raises(ValueError, match="dimension 1"):
        mo.mehler_prior(kern, mo.MeasureSpec.gauss([0.0, 0.0], [1.0, 1.05]))
    assert mo.mehler_prior(kern, mo.MeasureSpec.gauss([0.0, 0.0], [1.0, 1.02])) > 0
    meas = GaussianMeasure([0.0, 0.0], [1.0, 1.05])
    cf = ed.costFunctionGP_IVAR(gp.GP(kernels.KernelMehlerND([0.2, 0.9], 2), 1e-2), 3, Space(2, None, None),
                                measure=meas)
    limit = repr(math.sqrt(1.9 / 1.8))
    for call in (lambda: cf.evaluate(np.zeros((3, 2))),
                 lambda: ed.beginGreedyIVARExperimentalDesign(cf, np.zeros((10, 2)), 2),
                 lambda: ed.scoreCandidatesIVAR(cf, np.zeros((2, 2)), np.zeros((10, 2)))):
        with pytest.raises(ValueError, match="GaussianMeasure") as info:
            call()
        assert "dimension 1" in str(info.value) and limit in str(info.value)


@pytest.mark.parametrize("t", [[0.3], [0.9], [-0.6], [0.5, -0.8]])
def test_mercer_identity(t):
    """Under N(0, 1) in every dimension, Phi is the Mehler kernel with parameter t^2."""
    d = len(t)
    kern = orc.KernelSpec.mehler(t, d)
    sq = orc.KernelSpec.mehler(np.square(t), d)
    X = np.random.default_rng(d).normal(size=(30, d)) * 1.5
    got = mo.mehler_phi(kern, mo.MeasureSpec.gauss([0.0] * d, [1.0] * d), X, X)
    want = sq.gram(X, X)
    assert np.max(np.abs(got - want) / want) <= 1e-13


def _posterior_var(kern, design, noise):
    from scipy.linalg import cho_factor, cho_solve
    cf = cho_factor(kern.gram(design, design) + noise * np.eye(len(design)))

    def var(*x):
        kx = kern.gram(design, np.array([x]))[:, 0]
        return float(kern.prior(np.array([x]))[0] - kx @ cho_solve(cf, kx))
    return var


@pytest.mark.parametrize("kind", ["box", "gauss"])
def test_cost_1d_matches_quadrature(kind):
    from scipy import integrate
    design = np.array([[-0.7], [0.1], [0.45], [0.9], [1.6]])
    if kind == "box":
        kern = orc.KernelSpec.mehler([0.9], 1)
        var = _posterior_var(kern, design, 1e-2)
        meas = mo.MeasureSpec.box([-1.0], [2.0])
        want = integrate.quad(var, -1.0, 2.0, points=design[:, 0], epsabs=1e-14, epsrel=1e-13, limit=200)[0] / 3.0
    else:
        kern = orc.KernelSpec.mehler([0.5], 1)
        var = _posterior_var(kern, design, 1e-2)
        meas = mo.MeasureSpec.gauss([0.2], [0.9])
        dens = lambda x: math.exp(-0.5 * ((x - 0.2) / 0.9) ** 2) / (0.9 * math.sqrt(2 * math.pi))  # noqa: E731
        want = integrate.quad(lambda x: var(x) * dens(x), -40.0, 40.0, points=list(design[:, 0]) + [0.2],
                              epsabs=1e-14, epsrel=1e-13, limit=400)[0]
    got = mo.fast_ivar_cost_mehler(kern, meas, design, 1e-2)
    assert abs(got - want) <= 1e-9 * abs(want), (got, want)


@pytest.mark.parametrize("kind", ["box", "gauss"])
def test_cost_2d_matches_quadrature(kind):
    from scipy import integrate
    kern = orc.KernelSpec.mehler([0.7, 0.4], 2)
    design = np.array([[-0.5, 0.2], [0.3, -0.4], [0.6, 0.7], [-0.1, -0.9]])
    var = _posterior_var(kern, design, 1e-3)
    opts = {"epsabs": 1e-13, "epsrel": 1e-12, "limit": 100}
    if kind == "box":
        meas = mo.MeasureSpec.box([-1.0, -0.5], [1.0, 1.5])
        want = integrate.nquad(var, [[-1.0, 1.0], [-0.5, 1.5]], opts=opts)[0] / 4.0
    else:
        meas = mo.MeasureSpec.gauss([0.1, -0.2], [0.4, 0.5])
        dens = lambda x, y: math.exp(-0.5 * ((x - 0.1) / 0.4) ** 2 - 0.5 * ((y + 0.2) / 0.5) ** 2) / (2 * math.pi * 0.2)  # noqa: E731
        want = integrate.nquad(lambda x, y: var(x, y) * dens(x, y), [[-4.9, 5.1], [-6.2, 5.8]], opts=opts)[0]
    got = mo.fast_ivar_cost_mehler(kern, meas, design, 1e-3)
    assert abs(got - want) <= 1e-9 * abs(want), (got, want)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _bind(kern, kind, p0, p1):
    import ctypes as C
    from gpexp_b200 import _lib
    from gpexp_b200.device import Device
    dev = Device.get()
    dev.set_kernel(_lib.MEHLER, kern.dim, kern.packed_params())
    dbl = C.POINTER(C.c_double)
    a, b = np.ascontiguousarray(p0, dtype=np.float64), np.ascontiguousarray(p1, dtype=np.float64)
    rc = _lib.lib.gpx_set_measure(dev.h, kind, kern.dim, a.ctypes.data_as(dbl), b.ctypes.data_as(dbl))
    return dev, rc


def _phi_device(dev, X, Y, ld=None, fill=None):
    from gpexp_b200 import _lib
    from gpexp_b200.device import ptr
    A, B = dev.points(X), dev.points(Y)
    ld = ld or B.ld
    out = dev.zeros(A.n + 2, ld)
    if fill is not None:
        out.fill_(fill)
    _lib.check(_lib.lib.gpx_phi_gram(dev.h, ptr(A.X), A.n, A.ld, ptr(B.X), B.n, B.ld, ptr(out), ld, dev.stream),
               "gpx_phi_gram")
    return out.cpu().numpy()


def _mp_phi(kind, t, p0, p1, x, y):
    """(Phi(x, y), sum over dimensions of |exponent terms|) from the closed form at 50 digits."""
    import mpmath as mp
    mp.mp.dps = 50
    out, terms = mp.mpf(1), mp.mpf(0)
    for q in range(len(t)):
        tq, a, b = mp.mpf(t[q]), mp.mpf(x[q]), mp.mpf(y[q])
        r = 1 - tq * tq
        m = (a + b) / 2
        e_ab = tq * tq * (a - b) ** 2 / (4 * r)
        if kind == mo.BOX:
            lo, hi = mp.mpf(p0[q]), mp.mpf(p1[q])
            if tq == 0:
                out *= mp.exp(-e_ab)
                terms += e_ab
                continue
            u, v = sorted(((tq * lo - m) / mp.sqrt(r), (tq * hi - m) / mp.sqrt(r)))
            diff = mp.erfc(u) - mp.erfc(v) if u >= 0 else mp.erfc(-v) - mp.erfc(-u) if v <= 0 else mp.erf(v) - mp.erf(u)
            w = abs(tq) * (hi - lo) / mp.sqrt(r)
            out *= mp.exp(m * m - e_ab) * mp.sqrt(mp.pi) / 2 * diff / w / r
            terms += e_ab + m * m + min(u * u, v * v)
        else:
            mu, sd = mp.mpf(p0[q]), mp.mpf(p1[q])
            g = r + 2 * tq * tq * sd * sd
            quad = [tq * tq * (2 * sd * sd - 1) * m * m / g, 2 * tq * mu * m / g, -tq * tq * mu * mu / g]
            out *= mp.exp(-e_ab + sum(quad)) / mp.sqrt(r * g)
            terms += e_ab + sum(abs(v) for v in quad)
    return out, float(terms)


T_SETS = {"near0_neg_near1": [1e-3, -0.6, 0.99], "zero_mid_negnear1": [0.0, 0.45, -0.97]}


@pytest.mark.gpu
@pytest.mark.parametrize("tset", list(T_SETS))
@pytest.mark.parametrize("kind", [mo.BOX, mo.GAUSS])
def test_phi_gram_matches_mpmath_within_ulp_bound(tset, kind):
    """|got - exact| <= (64 + 8 sum|exponent terms|) ulp, from coincident points to far tails; below 2^-1022 the result
    is exactly 0."""
    t = np.array(T_SETS[tset])
    rng = np.random.default_rng(7)
    p0, p1 = (np.array([-1.0, -0.5, 0.0]), np.array([1.0, 2.0, 0.25])) if kind == mo.BOX else \
        (np.array([0.1, -0.3, 0.0]), np.array([0.2, 0.7, 0.05]))
    kern = orc.KernelSpec.mehler(t, 3)
    dev, rc = _bind(kern, kind, p0, p1)
    assert rc == 0
    X = np.concatenate([rng.uniform(-1.5, 1.5, (30, 3)), [[1.0, 2.0, 0.25], [-1.0, -0.5, 0.0], [3.0, -4.0, 5.0],
                                                          [6.0, 6.5, -7.0]]])
    Y = np.concatenate([X[::3] + rng.normal(0, 0.02, X[::3].shape), [[-8.0, 9.0, 12.0], [40.0, -40.0, 40.0]]])
    got = _phi_device(dev, X, Y)
    zeros = 0
    for i in range(len(X)):
        for j in range(len(Y)):
            exact, terms = _mp_phi(kind, t, p0, p1, X[i], Y[j])
            if exact < 2.0 ** -1022:
                assert got[i, j] == 0.0, (i, j, got[i, j], exact)
                zeros += 1
                continue
            tol = (64 + 8 * terms) * EPS * float(exact)
            assert abs(got[i, j] - float(exact)) <= tol, (i, j, got[i, j], float(exact), terms)
    assert zeros > 0   # the far probes reach the flush


@pytest.mark.gpu
@pytest.mark.parametrize("ncols", [255, 256, 257])
@pytest.mark.parametrize("kind", [mo.BOX, mo.GAUSS])
def test_block_edges_keep_padding(ncols, kind):
    """Sentinels in the output padding stay untouched by gpx_phi_gram, gpx_phi_diag and gpx_phi_append_row."""
    from gpexp_b200 import _lib
    from gpexp_b200.device import ptr, roundup
    rng = np.random.default_rng(ncols)
    kern = orc.KernelSpec.mehler([0.8, -0.5], 2)
    meas = mo.MeasureSpec.box([-1.0, -1.0], [1.0, 1.0]) if kind == mo.BOX else mo.MeasureSpec.gauss([0.0, 0.1], [0.9, 0.5])
    dev, rc = _bind(kern, kind, meas.p0, meas.p1)
    assert rc == 0
    X, Y = rng.uniform(-1, 1, (7, 2)), rng.uniform(-1, 1, (ncols, 2))
    S = -7.25
    ld = roundup(ncols) + 128
    got = _phi_device(dev, X, Y, ld=ld, fill=S)
    want = mo.mehler_phi(kern, meas, X, Y)
    assert np.max(np.abs(got[:7, :ncols] - want) / want) <= 1e-13
    assert np.all(got[:7, ncols:] == S) and np.all(got[7:] == S)
    P = dev.points(Y)
    diag = dev.zeros(ld).fill_(S)
    _lib.check(_lib.lib.gpx_phi_diag(dev.h, ptr(P.X), ncols, P.ld, ptr(diag), dev.stream), "gpx_phi_diag")
    diag = diag.cpu().numpy()
    assert np.max(np.abs(diag[:ncols] - mo.mehler_phi_diag(kern, meas, Y)) / diag[:ncols]) <= 1e-13
    assert np.all(diag[ncols:] == S)
    n = 3
    Z = dev.upload(np.concatenate([rng.normal(size=(n, P.ld)), np.full((2, P.ld), S)]))
    rec = np.zeros(_lib.GPX_PIVOT_HDR + n)
    rec[2], rec[3:5] = 0.49, Y[5]
    rec[_lib.GPX_PIVOT_HDR:] = rng.normal(size=n)
    zh = Z.cpu().numpy()
    _lib.check(_lib.lib.gpx_phi_append_row(dev.h, ptr(dev.upload(rec)), ptr(P.X), ncols, P.ld, ptr(Z), P.ld, n,
                                           dev.stream), "gpx_phi_append_row")
    z = Z.cpu().numpy()
    row = (mo.mehler_phi(kern, meas, Y[5:6], Y)[0] - rec[_lib.GPX_PIVOT_HDR:] @ zh[:n, :ncols]) / 0.7
    assert np.max(np.abs(z[n, :ncols] - row)) <= 1e-14 * np.max(np.abs(row)) * 8
    pad = ncols + (ncols & 1)
    assert np.all(z[n, ncols:pad] == 0.0) and np.all(z[n, pad:] == S) and np.all(z[n + 1] == S)
    assert np.array_equal(z[:n], zh[:n])


@pytest.mark.gpu
def test_phi_gram_under_standard_normal_is_gram_of_t_squared():
    """gpx_phi_gram under N(0, I) against gpx_gram of the kernel with parameters t^2 (the Mercer identity)."""
    from gpexp_b200 import _lib
    from gpexp_b200.device import ptr
    t = np.array([0.9, -0.5, 0.3])
    kern = orc.KernelSpec.mehler(t, 3)
    dev, rc = _bind(kern, mo.GAUSS, np.zeros(3), np.ones(3))
    assert rc == 0
    X = np.random.default_rng(3).normal(size=(300, 3))
    got = _phi_device(dev, X, X)[:300, :300]
    dev.set_kernel(_lib.MEHLER, 3, t * t)
    A = dev.points(X)
    out = dev.zeros(300, A.ld)
    _lib.check(_lib.lib.gpx_gram(dev.h, ptr(A.X), 300, A.ld, ptr(A.X), 300, A.ld, ptr(out), A.ld, 0, None, 0.0,
                                 dev.stream), "gpx_gram")
    want = out.cpu().numpy()[:, :300]
    assert np.max(np.abs(got - want) / want) <= 1e-12


@pytest.mark.gpu
def test_set_measure_rejects_infinite_prior():
    """GPX_EINVAL, with a message, where s is not finite: a Gaussian wider than the kernel allows, or a box whose
    integral of k(x, x) overflows."""
    from gpexp_b200 import _lib
    kern = orc.KernelSpec.mehler([0.9, 0.2], 2)
    _, rc = _bind(kern, mo.GAUSS, [0.0, 0.0], [1.05, 1.0])
    assert rc == -1 and "too wide" in _lib.last_error()
    _, rc = _bind(kern, mo.BOX, [0.0, 0.0], [40.0, 1.0])
    assert rc == -1 and "not a finite" in _lib.last_error()
    _, rc = _bind(kern, mo.GAUSS, [0.0, 0.0], [1.02, 1.0])
    assert rc == 0


def _kernel(t):
    from gpexp_b200 import kernels
    return kernels.KernelMehler1D(t[0], 1) if len(t) == 1 else kernels.KernelMehlerND(list(t), len(t))


def _measures(d):
    from gpexp_b200.approximation import GaussianMeasure, UniformMeasure
    return {"box": (UniformMeasure(-1.0, 1.5), mo.MeasureSpec.box([-1.0] * d, [1.5] * d)),
            "gauss": (GaussianMeasure([0.1] * d, [0.8] * d), mo.MeasureSpec.gauss([0.1] * d, [0.8] * d))}


def _check_greedy(spec, ometa, cand, idx, scores, nu):
    """Every pick's recorded score within 4 x bound of the oracle's exact score of design + pick, and the pick the
    oracle's arg-min unless the two lie within their tolerances (a near tie, counted and returned)."""
    nu = np.broadcast_to(np.asarray(nu, dtype=np.float64), (len(cand),))
    ties = 0
    for k, p in enumerate(idx):
        d = list(idx[:k])
        want, bound = mo.fast_ivar_scores_mehler(spec, ometa, cand[d], cand, nu[d], nu)
        tol = 4 * bound
        assert abs(scores[k] - want[p]) <= tol[p], (k, scores[k], want[p], tol[p])
        best = int(np.argmin(want))
        if p != best:
            assert want[p] - want[best] <= tol[p] + tol[best], (k, p, best, want[p], want[best])
            ties += 1
    return ties


def _cond(spec, design, nugget):
    return np.linalg.cond(spec.gram(design, design) + np.diag(np.broadcast_to(nugget, (len(design),))))


CASES = {"1d": ([0.9], 500, 16), "2d": ([0.8, 0.6], 1200, 16), "3d": ([0.5, 0.6, 0.7], 1500, 12)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("mname", ["box", "gauss"])
def test_greedy_evaluate_and_scoring_match_oracle(case, mname):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import Space
    ed.VERBOSE = False
    t, C, N = CASES[case]
    d = len(t)
    spec = orc.KernelSpec.mehler(t, d)
    meas, ometa = _measures(d)[mname]
    noise = 1e-2
    cand = np.random.default_rng(d).normal(0.1, 0.8, (C, d))
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel(t), noise), 4, Space(d, None, None), measure=meas)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N)
    eng.score()
    s = mo.mehler_prior(spec, ometa)
    assert abs(float(eng.cost.item()) - s) <= 1e-13 * s
    idx = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf, cand, N, returnIndices=True)]
    assert _cond(spec, cand[idx], noise) <= 1e4
    assert _check_greedy(spec, ometa, cand, idx, cf.lastScores, noise) <= 2
    design = cand[idx[:8]]
    costs, best = ed.scoreCandidatesIVAR(cf, design, cand)
    want, bound = mo.fast_ivar_scores_mehler(spec, ometa, design, cand, noise)
    assert np.all(np.abs(costs - want) <= 4 * bound), np.max(np.abs(costs - want) / bound)
    assert costs[best] == np.min(costs)
    cost = cf.evaluate(cand[idx[:4]])
    exact = mo.fast_ivar_cost_mehler(spec, ometa, cand[idx[:4]], noise)
    assert abs(cost - exact) <= 4 * 7 * 5 * EPS * s, (cost, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("mname", ["box", "gauss"])
def test_noise_function(mname):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import Space
    ed.VERBOSE = False
    t = [0.7, 0.4]
    spec = orc.KernelSpec.mehler(t, 2)
    meas, ometa = _measures(2)[mname]
    cand = np.random.default_rng(9).uniform(-1.0, 1.5, (1200, 2))
    nf = lambda x: 1e-2 * (1.0 + x[:, 0] ** 2)  # noqa: E731
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel(t), 1e-2), 3, Space(2, None, None, noise=nf), measure=meas)
    idx = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True)]
    assert _cond(spec, cand[idx], nf(cand[idx])) <= 1e4
    assert _check_greedy(spec, ometa, cand, idx, cf.lastScores, nf(cand)) <= 2
    design = cand[idx[:3]]
    costs, _ = ed.scoreCandidatesIVAR(cf, design, cand)
    want, bound = mo.fast_ivar_scores_mehler(spec, ometa, design, cand, nf(design), nf(cand))
    assert np.all(np.abs(costs - want) <= 4 * bound)
    exact = mo.fast_ivar_cost_mehler(spec, ometa, design, nf(design))
    assert abs(cf.evaluate(design) - exact) <= 1e-13 * abs(exact) + 4 * 6 * 4 * EPS * mo.mehler_prior(spec, ometa)


def _tensor_rule(nodes, weights, d):
    grids = np.meshgrid(*([nodes] * d), indexing="ij")
    pts = np.stack([g.ravel() for g in grids], axis=1)
    w = np.ones(len(pts))
    for q in range(d):
        w = w * np.meshgrid(*([weights] * d), indexing="ij")[q].ravel()
    return pts, w


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["hermite_1d_t0.5", "hermite_2d_t0.4", "legendre_1d_t0.9", "legendre_2d_t0.9"])
def test_weighted_path_with_tensor_quadrature_agrees(rule):
    """The exact costs equal the existing weighted path's (mcWeights) with the integration points and weights of an
    80-node Gauss-Hermite rule (t <= 0.5, where the integrand's tails let it converge) or a 60-node Gauss-Legendre rule
    on the box, within 1e-9 relative."""
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import GaussianMeasure, Space, UniformMeasure
    ed.VERBOSE = False
    kind, dim, tv = rule.split("_")
    d, tq = int(dim[0]), float(tv[1:])
    t = [tq] if d == 1 else [tq, 0.5 * tq]
    if kind == "hermite":
        mu, sd = 0.1, 0.8
        x, w = np.polynomial.hermite.hermgauss(80)
        pts, wts = _tensor_rule(mu + math.sqrt(2.0) * sd * x, w / math.sqrt(math.pi), d)
        meas = GaussianMeasure([mu] * d, [sd] * d)
    else:
        lo, hi = -1.0, 1.5
        x, w = np.polynomial.legendre.leggauss(60)
        pts, wts = _tensor_rule(0.5 * (hi - lo) * x + 0.5 * (hi + lo), 0.5 * w, d)
        meas = UniformMeasure(lo, hi)
    rng = np.random.default_rng(d)
    cand = rng.uniform(-1.0, 1.5, (700, d))
    design = cand[:6]
    noise = 1e-2
    cf_exact = ed.costFunctionGP_IVAR(gp.GP(_kernel(t), noise), 6, Space(d, None, None), measure=meas)
    cf_w = ed.costFunctionGP_IVAR(gp.GP(_kernel(t), noise), 6, Space(d, None, None), mcPoints=pts, mcWeights=wts)
    a, _ = ed.scoreCandidatesIVAR(cf_exact, design, cand)
    b, _ = ed.scoreCandidatesIVAR(cf_w, design, cand)
    assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-9
    assert abs(cf_exact.evaluate(design) - cf_w.evaluate(design)) <= 1e-9 * abs(cf_exact.evaluate(design))


@pytest.mark.gpu
def test_run_to_run_identical():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp
    from gpexp_b200.approximation import GaussianMeasure, Space
    ed.VERBOSE = False
    cand = np.random.default_rng(1).normal(size=(5000, 3))
    cf = ed.costFunctionGP_IVAR(gp.GP(_kernel([0.9, 0.9, 0.9]), 1e-2), 3, Space(3, None, None),
                                measure=GaussianMeasure(0.0, 1.0))
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


@pytest.mark.gpu
def test_reference_kernel_mehler_nd_with_measure():
    """With the reference staged: its own KernelMehlerND and costFunctionGP_IVAR under install_as_gpExp, with
    `measure` set as an attribute, give the oracle's exact cost."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(root, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        pytest.skip("no reference package available (set GPEXP_REFERENCE and run __graft_entry__.build() to stage it)")
    import gpexp_b200
    from gpexp_b200.approximation import GaussianMeasure
    gpexp_b200.install_as_gpExp(path)
    try:
        import gpExp.approximation as rap
        import gpExp.experimentalDesign as red
        import gpExp.gp as rgp
        import gpExp.kernels as rk
        red.VERBOSE = False
        t = [0.9, 0.5]
        k = rk.KernelMehlerND(t, 2)
        cand = np.random.default_rng(4).normal(size=(400, 2))
        cf = red.costFunctionGP_IVAR(rgp.GP(k, 1e-2), 4, rap.Space(2, None, None, noise=None),
                                     mcPoints=cand[:10])
        cf.measure = GaussianMeasure(0.0, 1.0)
        spec = orc.KernelSpec.mehler(t, 2)
        ometa = mo.MeasureSpec.gauss([0.0, 0.0], [1.0, 1.0])
        design = cand[:4]
        exact = mo.fast_ivar_cost_mehler(spec, ometa, design, 1e-2)
        assert abs(cf.evaluate(design) - exact) <= 1e-12 * abs(exact)
        idx = [int(i) for i in red.performGreedyIVARExperimentalDesign(cf, cand, 8, returnIndices=True)]
        ref, _ = mo.fast_greedy_ivar_mehler(spec, ometa, cand, 8, 1e-2)
        assert idx == ref
    finally:
        for name in [m for m in list(sys.modules) if m == "gpExp" or m.startswith("gpExp.")]:
            del sys.modules[name]
