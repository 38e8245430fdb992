"""Covariance values over the whole exponent range, for every device path that evaluates k(x, y).

The hot paths (Gram, fused Gram/TRSM, the DMMA prologues, the Gram x vector product) use the table-driven exp of
gpx_common.cuh with the signal variance folded into the table; the others (pairwise evaluation, the incremental row
append) use libdevice exp.  Each probe set pairs ONE point x with N points y at exponents chosen from 0 down to -1e12
(and up to +720 for Mehler), for signal variances from 2^-40 to 2^40, and every path is checked against k evaluated
by mpmath at 50 digits from the same float64 coordinates and hyper-parameters.

Contract (eps = 2^-52, A = the sum of the magnitudes of the exponent's terms, which is |a| for SE and Matern):
  normal    |ref| >= (1+t) max(1, s) 2^-1022 and finite: |got - ref| <= (C0 + C1 A) eps |ref|  [+ expanded-form budget]
  below     |got| <= (1+t) max(1, s) 2^-1021, of the sign of k (or 0), never NaN
  overflow  ref > DBL_MAX (Mehler only): got = +inf
t is the Matern distance term (0 for the other families); max(1, s) covers both the libdevice paths, which multiply a
normal-range exp by s, and the table paths, whose product s exp(a) is flushed below 2^-1022.
Then, on exact-argument probes, the table exp's own error is pinned in ulp, and k_s = s k_1 is checked without a
reference.  The second half runs the public designs with small signal variances and un-normalised coordinates against
the CPU oracle.
"""
import mpmath
import numpy as np
import pytest

from oracle import gpexp_oracle as orc

pytestmark = pytest.mark.gpu

mpmath.mp.dps = 50
EPS = 2.0 ** -52
DBL_MAX = float(np.finfo(np.float64).max)
MP_MAX = mpmath.mpf(DBL_MAX)
TINY = 2.0 ** -1022
LN2 = float(mpmath.log(2))
# Relative-error budget of one covariance value in the normal range.  The exponent is accumulated from d rounded terms of
# one sign (SE, Matern) or of magnitude A in total (Mehler), each rounding of the coordinates' difference, the square,
# the hyper-parameter and the running sum costs at most eps/2 of A: a handful of roundings per dimension, but they
# do not all line up, so C1 = 8 covers d <= 16.  exp of the rounded argument turns that absolute error into the same
# relative error.  C0 = 8 covers the exp itself (<= 2 ulp, see test_table_exp_ulp_bound), the product with the signal
# and Matern's (1 + t) factor.
C0, C1 = 8.0, 8.0
# measured maximum of the table exp over every slot, both rounding edges and ten signal variances (|a| <= 700)
TABLE_EXP_ULP = 2.0

SIGNALS = [2.0 ** -40, 1e-3, 0.3, 0.4999, 0.5, 0.7, 1.0, 1.7, 1e3, 2.0 ** 40]
EXPONENTS = [0.0, 1e-300, 1e-17, 1e-8, 1.0, 700.0, 707.5, 707.9, 708.2, 708.39, 708.4, 709.0, 745.0, 746.0, 1e3, 1e6,
             5.81e6, 5.82e6, 1e7, 1e9, 1e12]
MEHLER_POSITIVE = [1.0, 700.0, 709.0, 709.8, 710.0, 720.0]


# ------------------------------------------------------------------------------------------------
# probe sets: one point x, N points Y, the kernel, and the exact k for every pair
# ------------------------------------------------------------------------------------------------
class Probe:
    def __init__(self, name, family, params, x, Y, signal, cond, tpar, ref):
        self.name, self.family, self.params = name, family, np.asarray(params, dtype=np.float64)
        self.x, self.Y, self.signal = np.asarray(x, dtype=np.float64), np.asarray(Y, dtype=np.float64), signal
        self.cond, self.tpar, self.ref = np.asarray(cond), np.asarray(tpar), ref  # ref: list of mpf
        self.d = self.x.size

    def __repr__(self):
        return self.name


def _mp_se(x, y, cl, s):
    a = -sum((mpmath.mpf(float(p)) - mpmath.mpf(float(q))) ** 2 / mpmath.mpf(float(c)) ** 2 for p, q, c in zip(x, y, cl)) / 2
    return s * mpmath.exp(a), abs(a), mpmath.mpf(0)


def _mp_matern(x, y, rho, s):
    r = mpmath.sqrt(sum((mpmath.mpf(float(p)) - mpmath.mpf(float(q))) ** 2 for p, q in zip(x, y)))
    t = mpmath.sqrt(3) * r / mpmath.mpf(rho)
    return mpmath.mpf(s) * (1 + t) * mpmath.exp(-t), t, t


def _mp_mehler(x, y, ts):
    e, cond, s = mpmath.mpf(0), mpmath.mpf(0), mpmath.mpf(1)
    for p, q, t in zip(x, y, ts):
        p, q, t = mpmath.mpf(float(p)), mpmath.mpf(float(q)), mpmath.mpf(float(t))
        c = 1 / (2 * (1 - t * t))
        e -= (p * p * t * t - 2 * t * p * q + q * q * t * t) * c
        cond += (p * p * t * t + abs(2 * t * p * q) + q * q * t * t) * c
        s /= mpmath.sqrt(1 - t * t)
    return s * mpmath.exp(e), cond, mpmath.mpf(0)


def _build(name, family, params, x, Y, signal, fn):
    out = [fn(x, y) for y in Y]
    return Probe(name, family, params, x, Y, signal, [float(c) for _, c, _ in out], [float(t) for _, _, t in out],
                 [k for k, _, _ in out])


def se_probe(d, signal, exps=EXPONENTS):
    cl = np.ones(1) if d == 1 else np.linspace(0.6, 2.1, d)
    x = np.zeros(d) if d == 1 else 0.1 * np.cos(np.arange(d))
    u = np.ones(d) / np.sqrt(d)
    w = np.sqrt(np.sum((u / cl) ** 2))  # a = 1/2 (r w)^2
    Y = np.array([x + u * (np.sqrt(2.0 * a) / w) for a in exps])
    return _build(f"se_d{d}_s{signal:g}", 0, list(cl) + [signal], x, Y, signal, lambda p, q: _mp_se(p, q, cl, signal))


def matern_probe(signal, exps=EXPONENTS):
    rho = 0.8
    x = np.array([0.3, -0.1])
    Y = np.array([x + np.array([0.6, 0.8]) * (t * rho / np.sqrt(3.0)) for t in exps])
    return _build(f"matern_s{signal:g}", 1, [rho, signal], x, Y, signal, lambda p, q: _mp_matern(p, q, rho, signal))


def mehler_probe(t):
    # common x = X: e(y) = -(t^2 X^2 - 2 t X y + t^2 y^2) / (2 (1 - t^2)) peaks at X^2/2 (y = X/t); e(y) = E at
    # y = (X + sqrt((1 - t^2)(X^2 - 2E))) / t, so one x reaches both signs of the exponent
    X = 40.0
    targets = [-a for a in EXPONENTS] + MEHLER_POSITIVE
    Y = np.array([[(X + np.sqrt((1 - t * t) * (X * X - 2.0 * E))) / t] for E in targets])
    return _build(f"mehler_t{t}", 2, [t], [X], Y, float(1 / mpmath.sqrt(1 - mpmath.mpf(t) ** 2)),
                  lambda p, q: _mp_mehler(p, q, [t]))


def _edges_args():
    """Exact arguments next to both rounding edges of every table slot: x = -y^2/2 with y of 26 significant bits (y^2 and
    y^2/2 are exact), |x| <= 700.  Slot j is hit by n = rint(x 256/ln2) = -(256 m + j)."""
    ys = []
    for j in range(256):
        n = -(256 * (1 + (37 * j) % 1000) + j)
        for edge in (n - 0.5, n + 0.5):
            y0 = np.sqrt(-2.0 * edge * LN2 / 256)
            e = np.floor(np.log2(y0)) - 25
            q = np.floor(y0 / 2 ** e)
            ys += [q * 2 ** e, (q + 1) * 2 ** e]
    return np.array(ys)


def exact_se_probe(signal):
    Y = _edges_args()[:, None]
    return _build(f"se_exact_s{signal:g}", 0, [1.0, signal], [0.0], Y, signal, lambda p, q: _mp_se(p, q, [1.0], signal))


# ------------------------------------------------------------------------------------------------
# the device paths: each returns k(x, Y[j]) for every probe as a float64 numpy array
# ------------------------------------------------------------------------------------------------
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
    ns.torch, ns.ed, ns.lib, ns.L, ns.device, ns.engine, ns.gp, ns.gku, ns.Space = \
        torch, ed, _lib.lib, _lib, device, engine, gpmod, gku, Space
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    return ns


class Paths:
    def __init__(self, gx, pr):
        self.gx, self.pr, self.dev, self.lib, self.ptr = gx, pr, gx.dev, gx.lib, gx.ptr
        self.dev.set_kernel(pr.family, pr.d, pr.params)
        self.N = len(pr.Y)
        self.X = self.dev.points(pr.x[None, :])
        self.Yp = self.dev.points(pr.Y)

    def _read(self, t, n=None):
        self.dev.sync()
        return t.reshape(-1)[: (self.N if n is None else n)].cpu().numpy().copy()

    def pairwise(self):
        out = self.dev.zeros(self.N)
        self.gx.check(self.lib.gpx_kernel_pairwise(self.dev.h, self.ptr(self.X.X), 1, self.X.ld, self.ptr(self.Yp.X),
                                                   self.N, self.Yp.ld, self.ptr(out), self.dev.stream))
        return self._read(out)

    def gram(self, odd):
        # two rows (x twice): with an odd ld the second row starts 8 bytes off a 16-byte boundary -> scalar stores
        ld = self.N | 1 if odd else self.Yp.ld
        Xs = self.dev.points(np.vstack([self.pr.x, self.pr.x]))
        out = self.dev.zeros(2 * ld + 2)
        self.gx.check(self.lib.gpx_gram(self.dev.h, self.ptr(Xs.X), 2, Xs.ld, self.ptr(self.Yp.X), self.N, self.Yp.ld,
                                        self.ptr(out), ld, 0, None, 0.0, self.dev.stream))
        self.dev.sync()
        o = out.cpu().numpy()
        assert np.array_equal(o[:self.N], o[ld:ld + self.N], equal_nan=True)
        return o[:self.N].copy()

    def _sides(self, expanded, ldm, ldc):
        """(Ma_rows, Cb_rows, alpha, beta) for one M = 1 / C = N contraction with the given leading dimensions."""
        d = self.pr.d
        xm, yc = self.dev.zeros(d, ldm), self.dev.zeros(d, ldc)
        xm[:, :1] = self.X.X[:d, :1]
        yc[:, : self.N] = self.Yp.X[:d, : self.N]
        if not expanded:
            return xm, yc, 0.0, 0.0
        # centre on x, as the host centres on its data: alpha = 0 and beta_j is the pair's own exponent magnitude, so
        # the cancellation budget below stays per pair (a centre far from x would cancel |x - c|^2 terms of ~1e22 here)
        self.dev.set_center(self.pr.x)
        ra, rb = self.dev.zeros(16, ldm), self.dev.zeros(16, ldc)
        self.gx.check(self.lib.gpx_prep_side(self.dev.h, 0, self.ptr(xm), 1, ldm, self.ptr(ra), ldm, None, self.dev.stream))
        self.gx.check(self.lib.gpx_prep_side(self.dev.h, 1, self.ptr(yc), self.N, ldc, self.ptr(rb), ldc, None,
                                             self.dev.stream))
        self.dev.sync()
        return ra, rb, abs(float(ra[d, 0].item())), np.abs(rb[d + 1, : self.N].cpu().numpy())

    def cov(self, expanded):
        ldm, ldc = 128, self.Yp.ld
        ra, rb, al, be = self._sides(expanded, ldm, ldc)
        out = self.dev.zeros(ldc)
        mode = self.gx.L.PRO_EXPANDED if expanded else self.gx.L.PRO_DIFF
        self.gx.check(self.lib.gpx_cov_from_factors(self.dev.h, mode, None, ldm, self.ptr(ra), 1, None, ldc, self.ptr(rb),
                                                    self.N, 0, self.ptr(out), ldc, self.dev.stream))
        return self._read(out), al + be

    def ivar(self, expanded, padded, ring=None):
        """score[c] = k(x, y_c)^2: M = 1, n = 0, varM = 0, varC = 1, noise 0."""
        # unpadded: even leading dimensions (16-byte rows) that are not multiples of 128 -> the generic core
        ldc = (self.N + 3) & ~1
        ldm, ldc = (128, self.Yp.ld) if padded else (2, ldc if ldc % 128 else ldc + 2)
        ra, rb, al, be = self._sides(expanded, ldm, ldc)
        vM, vC = self.dev.zeros(ldm), self.dev.zeros(ldc) + 1.0
        ws = self.dev.zeros(int(self.lib.gpx_score_ivar_workspace(self.dev.h, 1, self.N)))
        score, best = self.dev.zeros(ldc), self.dev.zeros(1)
        idx = self.dev.zeros(1, dtype=self.gx.torch.int64)
        mode = self.gx.L.PRO_EXPANDED if expanded else self.gx.L.PRO_DIFF
        if ring is not None:
            self.gx.check(self.lib.gpx_set_ivar_ring(self.dev.h, ring))
        try:
            self.gx.check(self.lib.gpx_score_ivar(self.dev.h, mode, None, ldm, self.ptr(vM), self.ptr(ra), 1, None, ldc,
                                                  self.ptr(vC), self.ptr(rb), self.N, 0, 0.0, 0.0, None, self.ptr(ws),
                                                  self.ptr(score), self.ptr(best), self.ptr(idx), self.dev.stream))
            return self._read(score), al + be
        finally:
            if ring is not None:
                self.gx.check(self.lib.gpx_set_ivar_ring(self.dev.h, 1))

    def trsm(self):
        U = self.dev.zeros(128, 128)
        U[0, 0] = 1.0
        W, var = self.dev.zeros(self.Yp.ld), self.dev.zeros(self.Yp.ld)
        self.gx.check(self.lib.gpx_trsm_gram(self.dev.h, self.ptr(U), 1, 128, self.ptr(self.X.X), self.X.ld,
                                             self.ptr(self.Yp.X), self.N, self.Yp.ld, self.ptr(W), self.Yp.ld, self.ptr(var),
                                             self.dev.stream))
        return self._read(W), self._read(var)

    def matvec(self):
        b = self.dev.zeros(2) + 1.0
        ws = self.dev.zeros(int(self.lib.gpx_gram_matvec_workspace(self.N)))
        out = self.dev.zeros(self.N)
        self.gx.check(self.lib.gpx_gram_matvec(self.dev.h, self.ptr(self.Yp.X), self.N, self.Yp.ld, self.ptr(self.X.X), 1,
                                               self.X.ld, self.ptr(b), self.ptr(ws), self.ptr(out), self.dev.stream))
        return self._read(out)

    def append_row(self):
        rec = self.dev.zeros(self.gx.L.GPX_PIVOT_HDR + 16)
        rec[2] = 1.0
        rec[3: 3 + self.pr.d] = self.dev.upload(self.pr.x)
        W, var = self.dev.zeros(self.Yp.ld), self.dev.zeros(self.Yp.ld)
        self.gx.check(self.lib.gpx_append_row(self.dev.h, self.gx.L.ROW_KERNEL, self.ptr(rec), None, self.ptr(self.Yp.X),
                                              self.N, self.Yp.ld, self.ptr(W), self.Yp.ld, 0, self.ptr(var), self.dev.stream))
        return self._read(W)


# ------------------------------------------------------------------------------------------------
# the contract
# ------------------------------------------------------------------------------------------------
def _f(v):
    return float(v) if abs(v) <= DBL_MAX else float("inf") * (1 if v > 0 else -1)


def check_values(pr, got, what, budget=0.0, square=False):
    """Assert the contract of the module docstring for every probe; budget: extra absolute exponent error (scalar or per
    probe) of the expanded form.  square: got holds k^2 (the IVAR path)."""
    budget = np.broadcast_to(np.asarray(budget, dtype=np.float64), (len(pr.ref),))
    bad = []
    for j, (g, ref) in enumerate(zip(got, pr.ref)):
        lo = (1 + pr.tpar[j]) * max(1.0, pr.signal) * TINY
        tol = (C0 + C1 * pr.cond[j]) * EPS + budget[j]
        if square:
            ref, lo, tol = ref * ref, max(lo * lo, TINY), 2 * tol + EPS   # k^2: twice the relative error
        rf = _f(ref)
        if np.isnan(g):
            bad.append((j, "NaN", g, rf))
        elif abs(ref) > MP_MAX * (1 + tol):
            if g != float("inf"):
                bad.append((j, "expected +inf", g, rf))
        elif abs(ref) >= lo:
            if abs(ref) > MP_MAX * (1 - tol) and g == float("inf"):
                continue
            if not abs(mpmath.mpf(g) - ref) <= tol * abs(ref):
                bad.append((j, f"rel err {float(abs(mpmath.mpf(g) - ref) / abs(ref)):.3g} > {tol:.3g}", g, rf))
        else:
            if not (abs(g) <= 2 * lo and g * np.sign(pr.signal) >= 0):
                bad.append((j, "underflow region", g, rf))
    assert not bad, f"{pr.name} {what}: {len(bad)} of {len(got)} probes wrong, first {bad[:4]}"


# probe sets by name, built (and their references evaluated) on first use
PROBE_BUILDERS = {}
for _s in SIGNALS:
    PROBE_BUILDERS[f"se_d1_s{_s:g}"] = (lambda s: lambda: se_probe(1, s))(_s)
    PROBE_BUILDERS[f"matern_s{_s:g}"] = (lambda s: lambda: matern_probe(s))(_s)
for _s in (0.3, 1.0, 1e3):
    PROBE_BUILDERS[f"se_d3_s{_s:g}"] = (lambda s: lambda: se_probe(3, s))(_s)
    PROBE_BUILDERS[f"se_d16_s{_s:g}"] = (lambda s: lambda: se_probe(16, s))(_s)
for _t in (0.3, 0.9):
    PROBE_BUILDERS[f"mehler_t{_t}"] = (lambda t: lambda: mehler_probe(t))(_t)
PROBE_NAMES = list(PROBE_BUILDERS)
_PROBES = {}


def _probe(name):
    if name not in _PROBES:
        _PROBES[name] = PROBE_BUILDERS[name]()
        assert _PROBES[name].name == name
    return _PROBES[name]


@pytest.mark.parametrize("name", PROBE_NAMES)
def test_libdevice_paths(gx, name):
    pr = _probe(name)
    P = Paths(gx, pr)
    check_values(pr, P.pairwise(), "gpx_kernel_pairwise")
    check_values(pr, P.append_row(), "gpx_append_row")


@pytest.mark.parametrize("name", PROBE_NAMES)
def test_gram_paths(gx, name):
    pr = _probe(name)
    P = Paths(gx, pr)
    check_values(pr, P.gram(odd=False), "gpx_gram (paired stores)")
    check_values(pr, P.gram(odd=True), "gpx_gram (odd ld)")
    check_values(pr, P.matvec(), "gpx_gram_matvec")
    W, var = P.trsm()
    check_values(pr, W, "gpx_trsm_gram W")
    # var = k(y,y) - W^2 wherever both terms are finite
    for j, y in enumerate(pr.Y):
        kyy = {0: lambda: _mp_se(pr.x * 0 + y, y, pr.params[:-1], pr.signal)[0],
               1: lambda: mpmath.mpf(pr.signal),
               2: lambda: _mp_mehler(y, y, pr.params)[0]}[pr.family]()
        want = kyy - pr.ref[j] ** 2
        if abs(kyy) < DBL_MAX / 4 and abs(pr.ref[j]) < 1e150:
            scale = abs(kyy) + pr.ref[j] ** 2
            assert abs(mpmath.mpf(var[j]) - want) <= 1e-12 * scale + 1e-300, (pr.name, j, var[j], float(want))


@pytest.mark.parametrize("name", PROBE_NAMES)
def test_dmma_prologue_paths(gx, name):
    pr = _probe(name)
    P = Paths(gx, pr)
    got, _ = P.cov(expanded=False)
    check_values(pr, got, "gpx_cov_from_factors DIFF")
    for padded in (True, False):
        rings = (0, 1, 2) if padded else (None,)
        for ring in rings:
            got, _ = P.ivar(expanded=False, padded=padded, ring=ring)
            check_values(pr, got, f"gpx_score_ivar DIFF padded={padded} ring={ring}", square=True)
    if pr.d + 2 > 16:
        return  # no expanded form at d = 16: the hot kernel runs in difference form (above)
    # expanded form: k = f(alpha + beta + u.v) cancels |alpha| + |beta| in the exponent; Matern takes sqrt of it first,
    # which scales the error by c0^2 / 2 (d t / t = c0^2 d e / 2 t^2, and (1+t) e^-t changes by t/(1+t) dt)
    c0sq = 3.0 / pr.params[0] ** 2 if pr.family == 1 else 1.0
    got, ab = P.cov(expanded=True)
    check_values(pr, got, "gpx_cov_from_factors EXPANDED", budget=8 * EPS * c0sq * ab)
    for padded in (True, False):
        got, ab = P.ivar(expanded=True, padded=padded)
        check_values(pr, got, f"gpx_score_ivar EXPANDED padded={padded}", budget=8 * EPS * c0sq * ab, square=True)


@pytest.mark.parametrize("signal", SIGNALS)
def test_table_exp_ulp_bound(gx, signal):
    """Exact arguments (SE, d = 1, cl = 1, x = 0, dyadic y) at both rounding edges of every table slot: the table exp
    with the signal folded into its table is within TABLE_EXP_ULP of s exp(-y^2/2), on the difference-form DMMA
    prologue and on the Gram x vector product (the Gram kernel's scaled form rounds its argument, so it is not exact)."""
    pr = exact_se_probe(signal)
    P = Paths(gx, pr)
    for what, got in [("cov DIFF", P.cov(expanded=False)[0]), ("matvec", P.matvec())]:
        worst = 0.0
        for g, ref in zip(got, pr.ref):
            if abs(ref) < TINY:
                continue
            ulp = mpmath.mpf(2) ** (mpmath.floor(mpmath.log(abs(ref), 2)) - 52)
            worst = max(worst, float(abs(mpmath.mpf(g) - ref) / ulp))
        assert worst <= TABLE_EXP_ULP, (what, signal, worst)


def test_signal_scaling_without_reference(gx):
    """k_s = s k_1 within 2 ulp wherever k_1 and s k_1 are normal (bit-exact for powers of two), on every table path;
    where s k_1 falls below 2^-1022, k_s is flushed or tiny."""
    base = se_probe(1, 1.0, EXPONENTS + list(np.linspace(0.5, 740, 301)))
    outs = {}
    for s in SIGNALS:
        pr = se_probe(1, s, EXPONENTS + list(np.linspace(0.5, 740, 301)))
        P = Paths(gx, pr)
        outs[s] = {"gram": P.gram(odd=False), "cov": P.cov(expanded=False)[0], "matvec": P.matvec(), "trsm": P.trsm()[0]}
    assert np.array_equal(base.Y, pr.Y)
    for s in SIGNALS:
        for path, got in outs[s].items():
            k1 = outs[1.0][path]
            for g, a in zip(got, k1):
                if a == 0.0:
                    continue  # k_1 flushed: s k_1 says nothing about k_s for s > 1
                want = mpmath.mpf(s) * mpmath.mpf(a)
                if abs(want) < TINY:
                    assert g == 0.0 or abs(g) <= 2 * TINY, (path, s, g, a)
                    continue
                ulp = mpmath.mpf(2) ** (mpmath.floor(mpmath.log(abs(want), 2)) - 52)
                err = abs(mpmath.mpf(g) - want) / ulp
                assert err <= (0 if float(np.log2(s)).is_integer() else 2), (path, s, g, a, float(err))


# ------------------------------------------------------------------------------------------------
# the public designs: small signal variances and un-normalised coordinates against the CPU oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("signal", [0.3, 1e-3])
def test_greedy_ivar_small_signal(gx, signal):
    """cfg-2 geometry (cl = 0.06, 0.09 on [-1, 1]^2: exponents down to about -1100) with a signal variance below 1/2:
    the padded hot kernel sees covariances right at the underflow edge of the table."""
    from gpexp_b200 import kernels as K
    rng = np.random.default_rng(20)
    cand, mc = rng.uniform(-1, 1, (3000, 2)), rng.uniform(-1, 1, (5000, 2))
    ks, k = orc.KernelSpec.se([0.06, 0.09], signal, 2), K.KernelSquaredExponential([0.06, 0.09], signal, 2)
    noise = 1e-6 * signal
    ref, costs = orc.fast_greedy_ivar(ks, cand, mc, 10, noise)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, gx.Space(2, None, None), mcPoints=mc)
    idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 10, returnIndices=True)
    assert [int(i) for i in idx] == ref
    want = np.array([c[i] for c, i in zip(costs, ref)])
    assert np.all(np.isfinite(cf.lastScores))
    assert np.max(np.abs(cf.lastScores - want) / np.abs(want)) <= 1e-9


def test_greedy_mi_and_variance_small_signal(gx):
    from gpexp_b200 import kernels as K
    rng = np.random.default_rng(21)
    ks, k = orc.KernelSpec.se([0.06, 0.09], 0.3, 2), K.KernelSquaredExponential([0.06, 0.09], 0.3, 2)
    pool = rng.uniform(-1, 1, (800, 2))
    fidx, _ = orc.fast_greedy_mi(ks, pool, 1e-4, 12, start=2)
    cf = gx.ed.costFunctionGP_MI(gx.gp.GP(k, 1e-4), 12, gx.Space(2, None, None), nmc=800, mcpoints=pool)
    gx.ed.performGreedyMIExperimentalDesign(cf, 12, start=2)
    assert [int(i) for i in cf.lastIndices] == fidx
    pool = rng.uniform(-1, 1, (4000, 2))
    vidx, vscores = orc.fast_greedy_var(ks, pool, 40)
    k._bind(gx.dev)
    eng = gx.engine.GreedyVarEngine(gx.dev, gx.dev.points(pool), 40)
    eng.score_trace = []
    idx = eng.run(40)
    assert [int(i) for i in idx] == vidx
    for s in (0, 1, 20, 39):
        assert np.all(np.isfinite(eng.score_trace[s]))
        assert np.max(np.abs(eng.score_trace[s] - vscores[s])) <= 1e-9 * np.max(np.abs(vscores[s]))


def test_unnormalised_coordinates_short_length_scale(gx):
    """SE, cl = 0.02, coordinates in [0, 200]^2: far pairs have exponents near -1e8 (below the 32-bit wrap of the table
    exp's argument), a dense patch keeps some covariances far from zero."""
    from gpexp_b200 import kernels as K
    rng = np.random.default_rng(22)
    ks, k = orc.KernelSpec.se([0.02, 0.02], 1.0, 2), K.KernelSquaredExponential([0.02, 0.02], 1.0, 2)

    def pts(n):
        p = rng.uniform(0, 200, (n, 2))
        p[: n // 2] = 100.0 + rng.uniform(0, 0.25, (n // 2, 2))
        return p
    nodes, query = pts(300), pts(3000)
    Kd = gx.gku.calculateCovarianceMatrix(k, nodes)
    Kr = ks.gram(nodes, nodes)
    assert np.all(np.isfinite(Kd)) and np.max(np.abs(Kd - Kr)) <= 1e-12
    g = gx.gp.GP(k, 1e-6)
    g.addNodesAndComputeCovariance(nodes)
    var = g.evaluateVariance(query)
    ref = orc.fast_posterior_variance(ks, nodes, query, 1e-6)
    assert np.all(np.isfinite(var)) and np.max(np.abs(var - ref)) <= 1e-9
    cand, mc = pts(2000), pts(3000)
    ridx, costs = orc.fast_greedy_ivar(ks, cand, mc, 8, 1e-6)
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 1, gx.Space(2, None, None), mcPoints=mc)
    idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 8, returnIndices=True)
    assert [int(i) for i in idx] == ridx
    want = np.array([c[i] for c, i in zip(costs, ridx)])
    assert np.max(np.abs(cf.lastScores - want) / np.abs(want)) <= 1e-9
