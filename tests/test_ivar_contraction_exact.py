"""The IVAR contraction cores pair by pair against exact arithmetic.

A scoring call returns scores, not the pairs S[m, c] = sum_i W_M[i, m] W_C[i, c].  These tests make the covariance
vanish, so that a score becomes a function of S alone:
  - k = 0: integration points and candidates far apart, every covariance exponent between -2e4 and -2e3, where the
    table exp flushes to exactly 0 (test_zero_factors_give_zero_scores proves it on every core);
  - varM = 0, varC = 1, noise = 0, zero_tol = 0: score_c = fl(r_c / M), r_c = sum_m S[m, c]^2;
  - one non-zero column m* of W_M per call: every other pair contributes an exact 0, so r_c = fl(S[m*, c]^2).
On the INT8 core the kernel's arithmetic for such a call is the CPU model of test_ivar_int8_core (exact int32 diagonals,
int64 hi/lo, one rounding, the scale product, the square), so its scores must equal fl(fl(S_model^2) / M) bit for bit,
and S_model must meet 7.04 n u + |S| 2^-53 against the exact S.  A dropped or mis-placed diagonal changes S by
256^-t of its value or more: far below what a score tolerance sees, but always a different bit pattern here.
The DMMA cores (tensor-map, generic, and the store kernel of gpx_cov_from_factors) are checked against the FP64 bound
gamma_n sum_i |W_M[i, m]| |W_C[i, c]|, and the finalisation's mask, NaN and zero_tol rules against known r values.

The column patterns target the INT8 core's weak points: digit-targeted pairs whose S lives in one diagonal D_t
(t = 0 .. 12), worst-case digits that maximise every |D_t| and hi, power-of-two maxima, zero, dominated, subnormal and
far-scaled columns.  W_C holds one pattern per column, and the cycle shifts from call to call, so every pattern meets
the candidate-tile edges (columns 0, 63, 64 and C - 1).
"""
import functools
import operator
from fractions import Fraction

import numpy as np
import pytest

from tests.test_ivar_int8_core import DMMA, I8, L, SLICE_LAUNCHES, i8_dot, i8_parts, slice_column

EPS = 2.0 ** -53                                          # unit roundoff
WORST = float(64 * 2 ** 48 - 0x808080808080) * 2.0 ** -54  # digits a_0 = 64, a_1 .. a_6 = -128 (e = 0)
NS = (1, 31, 32, 33, 255, 4095)
M_STAR = (0, 127, 128, -1)  # integration column of the non-zero W_M column: tile edges and the partial last tile
M_DEF, C_DEF = 1000, 200    # partial last M tile (128) and candidate tile (64)
# kernel family, parameters (d = 1) and the centre of the integration points (candidates at minus it): every covariance
# exponent lies between -2e4 and -2e3
FAMILIES = {
    "se": (0, [1.0, 1.0], 50.0),      # -(x - y)^2 / 2 ~ -5000
    "matern": (1, [0.05, 1.0], 50.0),  # -sqrt(3) |x - y| / 0.05 ~ -3460
    "mehler": (2, [0.9], 20.0),       # -(0.81 x^2 - 1.8 x y + 0.81 y^2) / 0.38 ~ -3600
}


# ------------------------------------------------------------------------------------------------
# column patterns and the exact / model value of every pattern pair
# ------------------------------------------------------------------------------------------------
def digit_column(rng, n, p, e, scale_row, sign):
    """Row `scale_row` (0 for W_M, 1 for W_C) sets the column's exponent e; every row from 2 on holds one non-zero digit
    in slice p, and the other side's scale row is 0.  A W_M digit-p column against a W_C digit-q column has S in
    D_{p+q} alone."""
    x = np.zeros(n)
    if n > 2:
        d = rng.integers(1, (63 if p == 0 else 127) + 1, n - 2).astype(np.float64)
        x[2:] = sign * np.ldexp(d, 8 * (L - 1 - p) + e - 54)
    if n > scale_row:
        x[scale_row] = 0.75 * 2.0 ** e
    return x


def _patterns(n, side):
    rng = np.random.default_rng(7000 + 2 * n + side)
    sgn = 1 if side == 0 else -1
    pats = [("normal", rng.standard_normal(n)),
            ("binades", rng.standard_normal(n) * np.ldexp(1.0, -rng.integers(0, 60, n)))]
    pats += [(f"digit{p}", digit_column(rng, n, p, int(rng.integers(-8, 9)), side, 1 if side == 0 else (-1) ** p))
             for p in range(L)]
    pats += [("worst+", np.full(n, WORST)), ("worst-", np.full(n, -WORST))]
    x = rng.uniform(-0.5, 0.5, n)
    x[n // 2] = 8.0 * sgn
    pats.append(("pow2max", x))                       # column maximum exactly 2^3: the frexp edge
    pats.append(("zero", np.zeros(n)))
    x = rng.standard_normal(n)
    x[n - 1 if side == 0 else 0] = 2.0 ** 20
    pats.append(("dominant", x))
    pats.append(("big", np.full(n, sgn * (1.0 - 2.0 ** -53))))
    if side == 0:
        pats.append(("subnormal", rng.standard_normal(n) * 2.0 ** -1060))  # column maximum itself subnormal
        pats += [("far-", rng.standard_normal(n) * 2.0 ** -500), ("far+", rng.standard_normal(n) * 2.0 ** 300)]
    else:
        x = rng.standard_normal(n)
        x[1::2] *= 2.0 ** -1050                       # subnormal entries in a normal column
        pats.append(("subnormal", x))
        pats += [("far-", rng.standard_normal(n) * 2.0 ** -400), ("far+", rng.standard_normal(n) * 2.0 ** 250)]
    return pats


@functools.lru_cache(maxsize=None)
def patterns(n):
    """(W_M patterns, W_C patterns) of design size n: lists of (name, column)."""
    return _patterns(n, 0), _patterns(n, 1)


def _ints(x):
    """(X, s) with x_i = X_i 2^s exactly (every finite double is an integer times a power of two)."""
    r = [float(v).as_integer_ratio() for v in x]
    k = max(d.bit_length() - 1 for _, d in r)
    return [a << (k - d.bit_length() + 1) for a, d in r], -k


def exact_pair(xm, xc, ints=_ints):
    """(S, sum_i |W_M[i, m] W_C[i, c]|) as Fractions."""
    (a, sa), (b, sb) = ints(xm), ints(xc)
    prods = list(map(operator.mul, a, b))
    scale = Fraction(2) ** (sa + sb)
    return sum(prods) * scale, sum(map(abs, prods)) * scale


def in_bound_domain(em, ec):
    """Where the INT8 per-pair bound holds: both scales 2^(e - 30) and their product 2^(e_m + e_c - 60) are exact, the
    product normal.  Below, S_i8 flushes to 0 (see DESIGN.md section 5)."""
    return em - 30 >= -1074 and ec - 30 >= -1074 and -1022 <= em + ec - 60 <= 1023


@functools.lru_cache(maxsize=None)
def pair_table(n):
    """Every (W_M pattern, W_C pattern) pair of design size n: S_model (the INT8 kernel's S), the exact S and
    sum |a b| as floats.  Asserts the INT8 bound |S_model - S| <= 7.04 n u + |S| 2^-53 on every pair of its domain."""
    pm, pc = patterns(n)
    model = np.zeros((len(pm), len(pc)))
    exact = np.zeros_like(model)
    absdot = np.zeros_like(model)
    cache = {id(x): _ints(x) for _, x in pm + pc}
    checked = 0
    for i, (na, xm) in enumerate(pm):
        for j, (nb, xc) in enumerate(pc):
            got, em, ec = i8_dot(xm, xc)
            S, A = exact_pair(xm, xc, lambda x: cache[id(x)])
            model[i, j], exact[i, j], absdot[i, j] = got, float(S), float(A)
            if in_bound_domain(em, ec):
                u = Fraction(2) ** (em + ec - 54)
                bound = Fraction(704, 100) * n * u + abs(S) * Fraction(2) ** -53
                assert abs(Fraction(got) - S) <= bound, (n, na, nb, got, float(S), float(u))
                checked += 1
            else:
                assert got == 0.0, (n, na, nb, got)  # the scale product underflows: S_i8 flushes to 0
    assert checked >= len(pm) * len(pc) - 2 * len(pc)  # only the subnormal / out-of-range rows leave the domain
    return model, exact, absdot


def i8_expected(model, M):
    """Scores of a k = 0, varM = 0, varC = 1 call with one non-zero W_M column: fl(fl(S^2) / M)."""
    with np.errstate(over="ignore", under="ignore"):
        return np.abs(0.0 - (model * model) / 1.0 / float(M))


def dmma_score_ok(score, S, A, n, M):
    """score = fl(fl(S_d^2) / M) for some S_d within gamma_{n+2} A (+ underflow) of the exact S."""
    g = (n + 2) * EPS / (1 - (n + 2) * EPS)
    tol = g * A + (n + 2) * 2.0 ** -1074
    with np.errstate(over="ignore", under="ignore"):
        lo = np.maximum(np.abs(S) - tol, 0.0)
        hi = np.abs(S) + tol
        lo2 = lo * lo / M * (1 - 16 * EPS) - 2.0 ** -1070
        hi2 = hi * hi / M * (1 + 16 * EPS) + 2.0 ** -1070
    return (score >= lo2) & (score <= hi2)


# ------------------------------------------------------------------------------------------------
# CPU: the model at the edges of its domain
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", NS)
def test_model_meets_bound_on_every_pattern_pair(n):
    model, exact, _ = pair_table(n)
    assert np.all(np.isfinite(model))
    assert n < 3 or np.count_nonzero(model) > model.size // 2  # n < 3 leaves the digit columns without digits


def test_worst_case_digits_at_max_n():
    """K = GPX_I8_MAX_N with a_0 = 64, a_1..6 = -128 on both sides: |D_6| = 2^30 < 2^31 and hi ~ 2^50 < 2^51, the
    extremes the int32 accumulators and i64_to_f64 are sized for."""
    K = 16384
    y = np.full(K, WORST)
    dig, e = slice_column(y)
    assert e == 0 and np.all(dig[0] == 64) and np.all(dig[1:] == -128)
    for sign in (1, -1):
        D, hi, lo, em, ec = i8_parts(y, sign * y)
        if sign == 1:
            assert D == [K * v for v in (4096, -16384, 0, 16384, 2 * 16384, 3 * 16384, 4 * 16384)]
            assert hi == 2 ** 50 - 2 ** 44 + 2 ** 28 and lo == 2 ** 45 + 3 * 2 ** 36 + 2 ** 30
        else:  # -Y has the digits -63, -127 x 5, -128 (+128 is not a balanced digit): D_6 = 1.24 2^30
            assert D[6] == K * (-64 * 128 + 5 * 128 * 127 + 128 * 63) and abs(hi) < 2 ** 50
        assert max(abs(v) for v in D) < 2 ** 31 and abs(lo) < 2 ** 51
        got, _, _ = i8_dot(y, sign * y)
        S = sign * K * Fraction(WORST) ** 2
        u = Fraction(2) ** (em + ec - 54)
        assert abs(Fraction(got) - S) <= Fraction(704, 100) * K * u + abs(S) * Fraction(2) ** -53


@pytest.mark.parametrize("K", [3, 33, 4095])
def test_digit_targeted_pairs_live_in_one_diagonal(K):
    """A W_M digit-p column against a W_C digit-q column: D_t = 0 for every t != p + q, D_{p+q} != 0, and for
    p + q >= 7 the kernel's S is 0 while the exact S stays within the bound."""
    rng = np.random.default_rng(K)
    for p in range(L):
        xm = digit_column(rng, K, p, int(rng.integers(-8, 9)), 0, 1)
        for q in range(L):
            xc = digit_column(rng, K, q, int(rng.integers(-8, 9)), 1, (-1) ** q)
            D, hi, lo, em, ec = i8_parts(xm, xc)
            for t in range(L):
                assert (D[t] != 0) == (t == p + q), (p, q, D)
            got, _, _ = i8_dot(xm, xc)
            S, _ = exact_pair(xm, xc)
            if p + q >= L:
                assert got == 0.0 and S != 0
            else:
                assert Fraction(got) == S  # one diagonal, at most 2^31 256^6: exact in FP64
            u = Fraction(2) ** (em + ec - 54)
            assert abs(Fraction(got) - S) <= Fraction(704, 100) * K * u + abs(S) * Fraction(2) ** -53


# ------------------------------------------------------------------------------------------------
# GPU harness: one k = 0 scoring problem through the C ABI
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    from gpexp_b200 import _lib, device

    class NS_:
        pass
    ns = NS_()
    ns.torch, ns.lib, ns.L, ns.dev, ns.ptr, ns.check = torch, _lib.lib, _lib, device.Device.get(0), device.ptr, _lib.check
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")


def _unpadded(n):
    """An even leading dimension >= n that is not a multiple of 128: the generic core."""
    ld = (n + 3) & ~1
    return ld if ld % 128 else ld + 2


class Problem:
    """M integration points and C candidates of one family, far apart (k = 0), with W_M (n x ldm) and W_C (n x ldc)."""

    def __init__(self, gx, family, expanded, M, C, n, padded=True):
        from gpexp_b200.device import roundup
        self.gx, self.dev, self.lib, self.ptr = gx, gx.dev, gx.lib, gx.ptr
        self.M, self.C, self.n = M, C, n
        fam, params, x0 = FAMILIES[family]
        dev = self.dev
        dev.set_kernel(fam, 1, params)
        self.ldm, self.ldc = (roundup(M), roundup(C)) if padded else (_unpadded(M), _unpadded(C))
        xm, xc = dev.zeros(1, self.ldm), dev.zeros(1, self.ldc)
        xm[0, :M] = dev.upload(x0 + 0.5 * np.sin(np.arange(M)))
        xc[0, :C] = dev.upload(-x0 + 0.5 * np.cos(np.arange(C)))
        self.mode = gx.L.PRO_EXPANDED if expanded else gx.L.PRO_DIFF
        if expanded:
            dev.set_center(np.zeros(1))
            self.ra, self.rb = dev.zeros(16, self.ldm), dev.zeros(16, self.ldc)
            gx.check(self.lib.gpx_prep_side(dev.h, 0, self.ptr(xm), M, self.ldm, self.ptr(self.ra), self.ldm, None,
                                            dev.stream), "gpx_prep_side")
            gx.check(self.lib.gpx_prep_side(dev.h, 1, self.ptr(xc), C, self.ldc, self.ptr(self.rb), self.ldc, None,
                                            dev.stream), "gpx_prep_side")
        else:
            self.ra, self.rb = xm, xc
        self.Wm, self.Wc = dev.zeros(max(n, 1), self.ldm), dev.zeros(max(n, 1), self.ldc)
        self.vM, self.vC = dev.zeros(self.ldm), dev.zeros(self.ldc) + 1.0
        self.ws = dev.zeros(int(self.lib.gpx_score_ivar_workspace(dev.h, M, C)))
        self.out, self.best = dev.zeros(self.ldc), dev.zeros(1)
        self.idx = dev.zeros(1, dtype=gx.torch.int64)
        if n > 0:
            dev.reserve_ivar_scratch(M, C, n)

    def set_wc(self, cols):
        self.Wc[: self.n, : self.C] = self.dev.upload(np.ascontiguousarray(cols))

    def set_wm_column(self, m, x):
        self.Wm.zero_()
        self.Wm[: self.n, m] = self.dev.upload(x)

    def score(self, core, noise=0.0, zero_tol=0.0, mask=None):
        """(scores, best, idx, library launches) of one gpx_score_ivar call on the given core."""
        dev = self.dev
        self.gx.check(self.lib.gpx_set_ivar_core(dev.h, core), "gpx_set_ivar_core")
        try:
            l0 = dev.launches
            self.gx.check(self.lib.gpx_score_ivar(
                dev.h, self.mode, self.ptr(self.Wm), self.ldm, self.ptr(self.vM), self.ptr(self.ra), self.M,
                self.ptr(self.Wc), self.ldc, self.ptr(self.vC), self.ptr(self.rb), self.C, self.n, noise, zero_tol,
                self.ptr(mask), self.ptr(self.ws), self.ptr(self.out), self.ptr(self.best), self.ptr(self.idx),
                dev.stream), "gpx_score_ivar")
            launches = dev.launches - l0
        finally:
            self.gx.check(self.lib.gpx_set_ivar_core(dev.h, I8), "gpx_set_ivar_core")
        dev.sync()
        return (self.out[: self.C].cpu().numpy().copy(), float(self.best.item()), int(self.idx.item()), launches)

    def cov(self, ldcov):
        """gpx_cov_from_factors: k - W_M^T W_C for every pair (M x C of an M x ldcov array)."""
        out = self.dev.zeros(self.M, ldcov)
        self.gx.check(self.lib.gpx_cov_from_factors(
            self.dev.h, self.mode, self.ptr(self.Wm), self.ldm, self.ptr(self.ra), self.M, self.ptr(self.Wc), self.ldc,
            self.ptr(self.rb), self.C, self.n, self.ptr(out), ldcov, self.dev.stream), "gpx_cov_from_factors")
        self.dev.sync()
        return out[:, : self.C].cpu().numpy().copy()


def _cycle(n, shift, C):
    """W_C columns: pattern (c + shift) mod P for column c, and the pattern index of every column."""
    _, pc = patterns(n)
    which = (np.arange(C) + shift) % len(pc)
    return np.stack([pc[w][1] for w in which], axis=1), which


def _describe(n, i, which, bad):
    pm, pc = patterns(n)
    return f"n={n} W_M {pm[i][0]}: W_C columns {list(bad[:6])} ({[pc[which[c]][0] for c in bad[:6]]})"


def _run_i8_patterns(P, n, rot, ms=M_STAR):
    """Every W_M pattern in turn (m* cycling through ms), W_C cycled per call: bit-exact to the model, and each
    call ran the INT8 core (one DMMA call for the launch count)."""
    model, _, _ = pair_table(n)
    pm, _ = patterns(n)
    la = None
    for i, (_, x) in enumerate(pm):
        cols, which = _cycle(n, i + rot, P.C)
        P.set_wc(cols)
        m = ms[(i + rot) % len(ms)] % P.M
        P.set_wm_column(m, x)
        if la is None:
            la = P.score(DMMA)[3]
        got, _, _, lb = P.score(I8)
        assert lb == la + SLICE_LAUNCHES, (la, lb)
        want = i8_expected(model[i, which], P.M)
        bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
        assert bad.size == 0, f"m*={m} " + _describe(n, i, which, bad) + f" got {got[bad[:3]]} want {want[bad[:3]]}"


# ------------------------------------------------------------------------------------------------
# GPU: k = 0 really holds
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("expanded", [False, True])
def test_zero_factors_give_zero_scores(gx, family, expanded):
    """All-zero W: every score is exactly 0 on the INT8, tensor-map and generic cores, and the store kernel returns
    k = 0 for every pair -- the premise of everything below."""
    for padded in (True, False):
        P = Problem(gx, family, expanded, M_DEF, C_DEF, 33, padded=padded)
        cores = (I8, DMMA) if padded else (I8,)  # unpadded operands take the generic core whatever is selected
        launches = {}
        for core in cores:
            got, _, _, launches[core] = P.score(core)
            assert np.all(got == 0.0), (family, expanded, padded, core, got[got != 0][:4])
        if padded:
            assert launches[I8] == launches[DMMA] + SLICE_LAUNCHES
        assert np.all(P.cov(_unpadded(C_DEF)) == 0.0)
        P0 = Problem(gx, family, expanded, M_DEF, C_DEF, 0, padded=padded)
        assert np.all(P0.score(I8)[0] == 0.0) and np.all(P0.cov(_unpadded(C_DEF)) == 0.0)  # n = 0: k^2 and k alone


# ------------------------------------------------------------------------------------------------
# GPU: the INT8 core, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("expanded", [False, True])
def test_i8_pairs_bit_exact(gx, family, expanded, n):
    """All six instantiations (SE, Matern, Mehler x both prologue forms), K tails of the 32-byte chunks, m* at 0, 127,
    128 and M - 1 (partial last M tile): every score equals the model's fl(fl(S_model^2) / M)."""
    P = Problem(gx, family, expanded, M_DEF, C_DEF, n)
    _run_i8_patterns(P, n, rot=list(FAMILIES).index(family) + 2 * expanded)


@pytest.mark.gpu
def test_i8_pairs_bit_exact_in_a_later_m_split(gx):
    """M = 39 950: m* in the middle and at the end of the integration points sits in a later M-split of the grid."""
    P = Problem(gx, "se", True, 39_950, C_DEF, 33)
    _run_i8_patterns(P, 33, rot=0, ms=(-1, 20_000, 39_000, 128))
    P = Problem(gx, "mehler", False, 39_950, C_DEF, 255)
    _run_i8_patterns(P, 255, rot=1, ms=(-1, 31_000, 129))


@pytest.mark.gpu
def test_i8_domain_edges(gx):
    """n = GPX_I8_MAX_N with worst-case digits (|D_6| = 2^30, hi ~ 2^50): bit-exact.  n = GPX_I8_MAX_N + 1, and
    scratch one byte short of gpx_ivar_scratch_bytes: the call takes the DMMA core (no slicing launches, same scores
    as the DMMA core selected explicitly)."""
    lib, dev, torch = gx.lib, gx.dev, gx.torch
    Mn = Cn = 256
    nmax = gx.L.GPX_I8_MAX_N
    signs = np.where(np.arange(Cn) % 2 == 0, 1.0, -1.0)
    for n in (nmax, nmax + 1):
        P = Problem(gx, "se", False, Mn, Cn, n)
        P.set_wc(np.full((n, Cn), WORST) * signs)
        for m, s in ((Mn - 1, 1.0), (0, -1.0)):
            P.set_wm_column(m, np.full(n, s * WORST))
            a, _, _, la = P.score(DMMA)
            b, _, _, lb = P.score(I8)
            if n == nmax:
                assert lb == la + SLICE_LAUNCHES
                for sc in (1.0, -1.0):
                    want = i8_expected(np.array([i8_dot(np.full(n, s * WORST), np.full(n, sc * WORST))[0]]), Mn)[0]
                    assert np.all(b[signs == sc] == want), (m, s, sc, b[signs == sc][:2], want)
            else:
                assert lb == la and np.array_equal(a, b)
            S = n * WORST * WORST
            assert np.all(dmma_score_ok(a, np.full(Cn, S), np.full(Cn, S), n, Mn))
    # scratch one byte short: the DMMA core; exactly enough: the INT8 core.  The device's registration is put back.
    n = 255
    P = Problem(gx, "matern", True, M_DEF, C_DEF, n)
    cols, which = _cycle(n, 0, C_DEF)
    P.set_wc(cols)
    P.set_wm_column(M_DEF - 1, patterns(n)[0][0][1])
    a, _, _, la = P.score(DMMA)
    need = int(lib.gpx_ivar_scratch_bytes(dev.h, M_DEF, C_DEF, n))
    mine = torch.zeros(need, dtype=torch.uint8, device=dev.torch_device)
    try:
        gx.check(lib.gpx_set_ivar_scratch(dev.h, mine.data_ptr(), need - 1), "gpx_set_ivar_scratch")
        b, _, _, lb = P.score(I8)
        assert lb == la and np.array_equal(a, b)
        gx.check(lib.gpx_set_ivar_scratch(dev.h, mine.data_ptr(), need), "gpx_set_ivar_scratch")
        b, _, _, lb = P.score(I8)
        assert lb == la + SLICE_LAUNCHES
        assert np.array_equal(b, i8_expected(pair_table(n)[0][0, which], M_DEF))
    finally:
        own = dev._ivar_scratch
        gx.check(lib.gpx_set_ivar_scratch(dev.h, None if own is None else own.data_ptr(),
                                          0 if own is None else own.numel()), "gpx_set_ivar_scratch")
        dev.sync()


# ------------------------------------------------------------------------------------------------
# GPU: the DMMA cores against the FP64 bound
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("expanded", [False, True])
@pytest.mark.parametrize("padded", [True, False], ids=["tensor-map", "generic"])
def test_dmma_pairs_within_fp64_bound(gx, family, expanded, padded, n):
    """score = fl(fl(S_d^2) / M) with |S_d - S| <= gamma_{n+2} sum_i |W_M[i, m]| |W_C[i, c]| on the tensor-map core
    (padded operands) and on the generic core (leading dimensions not a multiple of 128)."""
    P = Problem(gx, family, expanded, M_DEF, C_DEF, n, padded=padded)
    _, exact, absdot = pair_table(n)
    pm, _ = patterns(n)
    rot = list(FAMILIES).index(family) + 2 * expanded
    for i, (_, x) in enumerate(pm):
        cols, which = _cycle(n, i + rot, C_DEF)
        P.set_wc(cols)
        m = M_STAR[(i + rot) % 4] % M_DEF
        P.set_wm_column(m, x)
        got = P.score(DMMA)[0]
        ok = dmma_score_ok(got, exact[i, which], absdot[i, which], n, M_DEF)
        bad = np.flatnonzero(~ok)
        assert bad.size == 0, f"m*={m} " + _describe(n, i, which, bad) + f" got {got[bad[:3]]}"


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("expanded", [False, True])
def test_cov_from_factors_returns_minus_s(gx, family, expanded, n):
    """gpx_cov_from_factors with k = 0 stores -S, signed, for every pair at once (ragged M = 333, C = 201; W_M and W_C
    columns both cycle through their patterns): within gamma_{n+2} sum |a b| of the exact S."""
    M, C = 333, 201
    P = Problem(gx, family, expanded, M, C, n, padded=False)
    pm, pc = patterns(n)
    _, exact, absdot = pair_table(n)
    rm = (np.arange(M) * 5 + n) % len(pm)
    rc = (np.arange(C) + n) % len(pc)
    P.Wm[:n, :M] = P.dev.upload(np.stack([pm[w][1] for w in rm], axis=1))
    P.set_wc(np.stack([pc[w][1] for w in rc], axis=1))
    got = -P.cov(_unpadded(C))
    S, A = exact[np.ix_(rm, rc)], absdot[np.ix_(rm, rc)]
    g = (n + 2) * EPS / (1 - (n + 2) * EPS)
    with np.errstate(over="ignore"):
        tol = (g * A + 4 * EPS * np.abs(S)) * (1 + 4 * EPS) + (n + 2) * 2.0 ** -1074
        ok = np.abs(got - S) <= tol
    bad = np.argwhere(~ok)
    assert bad.size == 0, [(pm[rm[i]][0], pc[rc[j]][0], got[i, j], S[i, j]) for i, j in bad[:4]]


# ------------------------------------------------------------------------------------------------
# GPU: the finalisation rules
# ------------------------------------------------------------------------------------------------
def _finalise(r, varM_sum, M, varC, noise, zero_tol):
    """The finalisation kernel's arithmetic: |sum(varM)/M - (r / (varC + noise)) / M|, reduction 0 where the
    denominator is <= zero_tol."""
    base = varM_sum / M
    den = varC + noise
    with np.errstate(invalid="ignore", divide="ignore"):
        red = np.where(den <= zero_tol, 0.0, (r / den) / float(M))
    return np.abs(base - red)


def _argmin(scores, mask):
    """np.argmin over unmasked entries: a NaN wins, ties go to the lowest index; (-1, 0.0) if all are masked."""
    live = np.flatnonzero(mask == 0)
    if live.size == 0:
        return -1, 0.0
    nan = live[np.isnan(scores[live])]
    if nan.size:
        return int(nan[0]), float("nan")
    i = int(live[np.argmin(scores[live])])
    return i, float(scores[i])


def _check_pick(best, idx, scores, mask, what):
    wi, wb = _argmin(scores, mask)
    assert idx == wi, (what, idx, wi)
    assert (np.isnan(best) and np.isnan(wb)) or best == wb, (what, best, wb)


def _masks(rng, C, nan_at):
    """A random mask, the same with the NaN candidates masked and unmasked in turn, and everything masked."""
    mk = (rng.random(C) < 0.5).astype(np.uint8)
    a, b = mk.copy(), mk.copy()
    a[nan_at] = 1
    b[nan_at] = 0
    b[nan_at[0]] = 1  # the first NaN masked, the second one live: the live one wins
    return [("random", a), ("nan live", b), ("none", np.zeros(C, np.uint8)), ("all", np.ones(C, np.uint8))]


@pytest.mark.gpu
def test_score_ivar_mask_nan_and_zero_tol(gx):
    """Known r values from the INT8 harness (one W_M column, cycled W_C patterns: many exact ties), varM = 1/2,
    noise = 1/4, zero_tol = 3/4: candidates with varC + noise == zero_tol score base, one ulp above is scored, a NaN
    varC gives a NaN score.  The arg-min over the unmasked candidates follows np.argmin; all masked gives idx = -1."""
    n, C = 33, C_DEF
    P = Problem(gx, "se", False, M_DEF, C, n)
    model, _, _ = pair_table(n)
    cols, which = _cycle(n, 0, C)
    P.set_wc(cols)
    P.set_wm_column(5, patterns(n)[0][0][1])
    r = model[0, which] ** 2
    rng = np.random.default_rng(44)
    varC = np.ones(C)
    at_tol, above, nan_at = [0, 63], [64, C - 1], np.array([70, 150])
    varC[at_tol] = 0.5                   # 0.5 + 0.25 == 0.75 exactly
    varC[above] = 0.5 + 2.0 ** -53       # 0.75 + ulp(0.75)
    noise, zero_tol = 0.25, 0.75
    P.vM[:M_DEF] = 0.5                   # sum exact: base = 1/2
    for with_nan in (False, True):
        v = varC.copy()
        if with_nan:
            v[nan_at] = np.nan
        P.vC[:C] = P.dev.upload(v)
        want = _finalise(r, 0.5 * M_DEF, M_DEF, v, noise, zero_tol)
        assert np.all(want[at_tol] == 0.5) and np.all(want[above] != 0.5)
        for name, mk in _masks(rng, C, nan_at):
            got, best, idx, _ = P.score(I8, noise, zero_tol, P.dev.upload(mk, dtype=gx.torch.uint8))
            assert np.array_equal(got, want, equal_nan=True), name
            _check_pick(best, idx, got, mk, (with_nan, name))
        # ties: the smallest score is taken by several candidates (cycled patterns); mask its first holders
        mn = np.nanmin(want)
        holders = np.flatnonzero(want == mn)
        if holders.size > 1:
            mk = np.zeros(C, np.uint8)
            mk[holders[:-1]] = 1
            if with_nan:
                mk[nan_at] = 1
            got, best, idx, _ = P.score(I8, noise, zero_tol, P.dev.upload(mk, dtype=gx.torch.uint8))
            assert idx == holders[-1] and best == mn


@pytest.mark.gpu
def test_score_ivar_partials_finalisation(gx):
    """gpx_score_ivar_partials on hand-built per-segment sums: the segments are summed in order, the zero_tol rule and
    the arg-min rules are those of gpx_score_ivar."""
    dev, lib, ptr, torch = gx.dev, gx.lib, gx.ptr, gx.torch
    dev.set_kernel(0, 1, [1.0, 1.0])
    rng = np.random.default_rng(45)
    C, M, nseg = 300, 7, 3
    ldp = C + 2
    part = np.zeros((nseg, ldp))
    part[:, :C] = rng.integers(0, 4, (nseg, C)) * 0.125      # small dyadic sums: many ties
    part[1, 10] = 0.1                                         # order-dependent sums
    part[2, 10] = 0.2
    part[0, 20] = part[2, 250] = np.nan                       # NaN partials
    varC = np.ones(C)
    varC[[5, 6]] = 0.5
    varC[[7, 8]] = 0.5 + 2.0 ** -53
    noise, zero_tol = 0.25, 0.75
    r = np.zeros(C)
    for s in range(nseg):
        r = r + part[s, :C]
    want = _finalise(r, 0.5 * M, M, varC, noise, zero_tol)
    assert np.isnan(want[20]) and want[5] == 0.5
    P = dev.upload(part)
    vM, vC = dev.zeros(8) + 0.5, dev.upload(varC)
    score, best, idx = dev.zeros(ldp), dev.zeros(1), dev.zeros(1, dtype=torch.int64)
    for name, mk in _masks(rng, C, np.array([20, 250])) + [("ties", (want != np.nanmin(want)).astype(np.uint8))]:
        m = dev.upload(mk, dtype=torch.uint8)
        gx.check(lib.gpx_score_ivar_partials(dev.h, ptr(P), nseg, ldp, ptr(vM), M, ptr(vC), C, noise, zero_tol, ptr(m),
                                             ptr(score), ptr(best), ptr(idx), dev.stream), "gpx_score_ivar_partials")
        dev.sync()
        got = score[:C].cpu().numpy()
        assert np.array_equal(got, want, equal_nan=True), name
        _check_pick(float(best.item()), int(idx.item()), got, mk, name)
