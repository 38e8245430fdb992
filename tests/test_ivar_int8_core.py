"""The INT8 tensor-core IVAR core (GPX_CORE_I8): the fixed-point slicing model against exact integer arithmetic (CPU),
and the core against the FP64 DMMA core and the oracle on the same engine states (GPU)."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import gpexp_oracle as orc

L = 7  # slices per entry, ivar_i8_kernel's I8_L


# ------------------------------------------------------------------------------------------------
# CPU model of ivar_slice_kernel + the kernel's diagonal accumulation and recombination
# ------------------------------------------------------------------------------------------------
def slice_column(x):
    """(digits [L, K] int8, e) of one column: Y = rint(x 2^(54-e)) in balanced base-256 digits, max|x| < 2^e."""
    mx = float(np.max(np.abs(x))) if x.size else 0.0
    e = int(np.frexp(mx)[1]) if mx > 0.0 else 0
    Y = np.rint(np.ldexp(x, 54 - e)).astype(np.int64)
    dig = np.zeros((L, x.size), dtype=np.int64)
    for p in range(L - 1, 0, -1):
        a = ((Y + 128) & 255) - 128
        dig[p] = a
        Y = (Y - a) >> 8
    dig[0] = Y
    assert np.all(np.abs(dig[0]) <= 64) and np.all((dig[1:] >= -128) & (dig[1:] <= 127))
    return dig, e


def i8_parts(xm, xc):
    """(D, hi, lo, e_m, e_c) of one pair: the int32 diagonals t = 0..6 and their int64 recombination."""
    am, em = slice_column(xm)
    bc, ec = slice_column(xc)
    D = [sum(int(np.dot(am[p], bc[t - p])) for p in range(t + 1)) for t in range(L)]
    assert all(abs(v) < 2 ** 31 for v in D)
    hi = (D[0] << 24) + (D[1] << 16) + (D[2] << 8) + D[3]
    lo = (D[4] << 16) + (D[5] << 8) + D[6]
    assert abs(hi) < 2 ** 51 and abs(lo) < 2 ** 51
    return D, hi, lo, em, ec


def i8_dot(xm, xc):
    """S as the kernel forms it: int32 diagonals t = 0..6, int64 hi/lo, one FP64 rounding, scales 2^(e-30)."""
    _, hi, lo, em, ec = i8_parts(xm, xc)
    return float((hi << 24) + lo) * (np.ldexp(1.0, em - 30) * np.ldexp(1.0, ec - 30)), em, ec


def exact_dot(xm, xc):
    return sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(xm, xc))


def columns(rng, K):
    yield rng.standard_normal(K), rng.standard_normal(K)
    yield rng.uniform(-1, 1, K) * 1e-30, rng.uniform(-1, 1, K) * 1e30              # far from 1: scales only
    big = np.full(K, 1.0 - 2.0 ** -53)
    yield big, -big                                                                 # every digit at its bound
    x = rng.standard_normal(K)
    x[0] = 2.0 ** 20                                                                # one entry dominates its column
    yield x, rng.standard_normal(K) * 2.0 ** -40
    yield np.ldexp(np.ones(K), -rng.integers(0, 60, K)), np.ldexp(-np.ones(K), -rng.integers(0, 60, K))
    z = np.zeros(K)
    z[-1] = 3.0
    yield z, rng.standard_normal(K)                                                 # zero rows, K tail


@pytest.mark.parametrize("K", [1, 3, 31, 33, 255, 4096])
def test_slicing_model_error_bound(K):
    """|S_i8 - S| <= 7.04 K u + |S| 2^-53 with u = 2^(e_m + e_c - 54): the bound quoted in gpx_dmma.cu and DESIGN.md."""
    rng = np.random.default_rng(K)
    for xm, xc in columns(rng, K):
        got, em, ec = i8_dot(xm, xc)
        ref = exact_dot(xm, xc)
        err = abs(Fraction(got) - ref)
        u = Fraction(2) ** (em + ec - 54)
        assert err <= Fraction(704, 100) * K * u + abs(ref) * Fraction(2) ** -53, (K, float(err), float(u))


def test_slices_reconstruct_fixed_point_rounding():
    """The digits are exactly the fixed-point rounding of the column: sum_p a_p 256^(6-p) = rint(x 2^(54-e))."""
    rng = np.random.default_rng(5)
    for x, _ in columns(rng, 257):
        dig, e = slice_column(x)
        Y = sum(dig[p].astype(object) * (256 ** (L - 1 - p)) for p in range(L))
        want = [int(v) for v in np.rint(np.ldexp(x, 54 - e)).astype(np.int64)]
        assert [int(v) for v in Y] == want
        assert all(abs(Fraction(float(v)) - Fraction(int(y)) * Fraction(2) ** (e - 54)) <= Fraction(2) ** (e - 55)
                   for v, y in zip(x, Y))


# ------------------------------------------------------------------------------------------------
# GPU: the core against the DMMA core and the oracle.  Every engine here is built with resident=False: at these sizes
# the default would keep the covariance resident and never run a contraction.
# ------------------------------------------------------------------------------------------------
DMMA, I8 = 1, 2
SLICE_LAUNCHES = 2  # the INT8 core's extra launches per scoring call: ivar_slice_kernel for W_M and for W_C


@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    ed.VERBOSE = False
    from gpexp_b200 import _lib, device, kernels
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ed, ns.lib, ns.L, ns.kernels, ns.gp, ns.Space = torch, ed, _lib.lib, _lib, kernels, gpmod, Space
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")
    ns.dev.force_diff_form = False


def _core(gx, core):
    gx.check(gx.lib.gpx_set_ivar_core(gx.dev.h, core), "gpx_set_ivar_core")


def _case(gx, family, signal=1.0, C=1500, M=2000, seed=3):
    rng = np.random.default_rng(seed)
    K = gx.kernels
    if family == "se":
        cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
        k, noise = K.KernelSquaredExponential([0.06, 0.09], signal, 2), 1e-6 * signal
    elif family == "matern":
        cand, mc = rng.uniform(-1, 1, (C, 3)), rng.uniform(-1, 1, (M, 3))
        k, noise = K.KernelIsoMatern(0.4, signal, 3), 1e-4 * signal
    else:  # Mehler pool: per-point prior variances, far points with tiny factor columns
        cand, mc = rng.standard_normal((C, 3)), rng.standard_normal((M, 3))
        k, noise = K.KernelMehlerND([0.9, 0.8, 0.7], 3), 1e-2
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, noise), 1, gx.Space(cand.shape[1], None, None), mcPoints=mc)
    return cf, cand, mc


def _scores(gx, eng, core):
    """(scores, library launches) of one contraction-mode scoring call on the given core."""
    _core(gx, core)
    try:
        l0 = gx.dev.launches
        eng.score()
        launches = gx.dev.launches - l0
    finally:
        _core(gx, I8)
    return eng.scores[: eng.cand.n].cpu().numpy().copy(), launches


def _compare(gx, eng):
    """DMMA and INT8 scores of one state; asserts the INT8 call really ran the INT8 core."""
    a, la = _scores(gx, eng, DMMA)
    b, lb = _scores(gx, eng, I8)
    assert lb == la + SLICE_LAUNCHES, (la, lb)
    assert np.all(np.isfinite(b))
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["se", "matern", "mehler"])
@pytest.mark.parametrize("diff", [False, True])
def test_i8_matches_dmma_on_greedy_states(gx, family, diff):
    """Same state, both cores: scores agree far inside the 1e-9 contract at n = 1, 3, 31, 33, 255 (K tails of the
    64-byte chunks), and two I8 runs are bit-identical."""
    gx.dev.force_diff_form = diff
    try:
        cf, cand, _ = _case(gx, family)
        eng = gx.ed.beginGreedyIVARExperimentalDesign(cf, cand, 256, resident=False)
        differs = False
        for n in (1, 3, 31, 33, 255):
            eng.run(n)
            a, b = _compare(gx, eng)
            assert np.array_equal(b, _scores(gx, eng, I8)[0])
            assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-11, (family, diff, n)
            differs |= not np.array_equal(a, b)
        assert differs  # two different arithmetics: some score differs in its last bits
    finally:
        gx.dev.force_diff_form = False


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["se", "matern", "mehler"])
def test_i8_and_dmma_pick_the_same_designs(gx, family):
    picks, launches = {}, {}
    try:
        for core in (DMMA, I8):
            _core(gx, core)
            cf, cand, _ = _case(gx, family, C=1200, M=1500, seed=7)
            l0 = gx.dev.launches
            idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 48, returnIndices=True, resident=False)
            launches[core] = gx.dev.launches - l0
            picks[core] = [int(i) for i in idx]
    finally:
        _core(gx, I8)
    assert launches[I8] == launches[DMMA] + SLICE_LAUNCHES * 47  # every step but n = 0 scored on the INT8 core
    assert picks[DMMA] == picks[I8]


@pytest.mark.gpu
@pytest.mark.parametrize("log2_signal", [-40, -20, 0, 20, 40])
def test_i8_signal_range(gx, log2_signal):
    cf, cand, _ = _case(gx, "se", signal=2.0 ** log2_signal, C=1000, M=1300)
    eng = gx.ed.beginGreedyIVARExperimentalDesign(cf, cand, 40, resident=False)
    eng.run(33)
    a, b = _compare(gx, eng)
    assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-11


@pytest.mark.gpu
def test_i8_against_oracle_cfg2_geometry(gx):
    """cfg-2 kernel and noise: picks identical to the oracle and costs within 1e-9 relative, on the default core."""
    rng = np.random.default_rng(30)
    cand, mc = rng.uniform(-1, 1, (3000, 2)), rng.uniform(-1, 1, (5000, 2))
    ks, k = orc.KernelSpec.se([0.06, 0.09], 1.0, 2), gx.kernels.KernelSquaredExponential([0.06, 0.09], 1.0, 2)
    ref, costs = orc.fast_greedy_ivar(ks, cand, mc, 12, 1e-6)
    launches = {}
    for core in (DMMA, I8):  # a fresh cost function each: the first design on one also pays its set-up launches
        cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 1, gx.Space(2, None, None), mcPoints=mc)
        _core(gx, core)
        try:
            l0 = gx.dev.launches
            idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True, resident=False)
            launches[core] = gx.dev.launches - l0
        finally:
            _core(gx, I8)
    assert launches[I8] == launches[DMMA] + SLICE_LAUNCHES * 11
    assert [int(i) for i in idx] == ref
    want = np.array([c[i] for c, i in zip(costs, ref)])
    assert np.max(np.abs(cf.lastScores - want) / np.abs(want)) <= 1e-9


@pytest.mark.gpu
def test_dmma_core_ring_geometries_give_identical_scores(gx):
    """The reference core's three operand rings (gpx_set_ivar_ring) stay bit-identical to each other: with the INT8
    core as the default this is selected explicitly."""
    for family, n in (("se", 45), ("matern", 16), ("mehler", 131)):
        cf, cand, _ = _case(gx, family, C=1500, M=2100, seed=21)
        eng = gx.ed.beginGreedyIVARExperimentalDesign(cf, cand, n + 1, resident=False)
        eng.run(n)
        outs = []
        _core(gx, DMMA)
        try:
            for ring in (0, 1, 2):
                gx.check(gx.lib.gpx_set_ivar_ring(gx.dev.h, ring), "gpx_set_ivar_ring")
                eng.score()
                outs.append(eng.scores[:1500].cpu().numpy().copy())
        finally:
            gx.check(gx.lib.gpx_set_ivar_ring(gx.dev.h, 1), "gpx_set_ivar_ring")
            _core(gx, I8)
        assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2]), family
        assert np.all(np.isfinite(outs[0]))


# the covariance probes of test_covariance_domain.py (mpmath references over the whole exponent range, signals 2^-40 to
# 2^40, Mehler overflow) through the INT8 core's epilogue: an n = 1 padded contraction with zero factor rows, so that
# S = 0 on both cores and score = k^2
def _ivar_n1(gx, P, expanded, core):
    ldm, ldc = 128, P.Yp.ld
    ra, rb, al, be = P._sides(expanded, ldm, ldc)
    Wm, Wc = P.dev.zeros(1, ldm), P.dev.zeros(1, ldc)
    vM, vC = P.dev.zeros(ldm), P.dev.zeros(ldc) + 1.0
    ws = P.dev.zeros(int(gx.lib.gpx_score_ivar_workspace(P.dev.h, 1, P.N)))
    score, best = P.dev.zeros(ldc), P.dev.zeros(1)
    idx = P.dev.zeros(1, dtype=gx.torch.int64)
    mode = gx.L.PRO_EXPANDED if expanded else gx.L.PRO_DIFF
    P.dev.reserve_ivar_scratch(1, P.N, 1)
    _core(gx, core)
    try:
        l0 = P.dev.launches
        gx.check(gx.lib.gpx_score_ivar(P.dev.h, mode, gx.ptr(Wm), ldm, gx.ptr(vM), gx.ptr(ra), 1, gx.ptr(Wc), ldc,
                                       gx.ptr(vC), gx.ptr(rb), P.N, 1, 0.0, 0.0, None, gx.ptr(ws), gx.ptr(score),
                                       gx.ptr(best), gx.ptr(idx), P.dev.stream), "gpx_score_ivar")
        launches = P.dev.launches - l0
    finally:
        _core(gx, I8)
    return P._read(score), al + be, launches


def _domain_probe_names():
    from tests import test_covariance_domain as cd
    return cd.PROBE_NAMES


@pytest.mark.gpu
@pytest.mark.parametrize("name", _domain_probe_names())
def test_i8_epilogue_covariance_domain(gx, name):
    from tests import test_covariance_domain as cd
    pr = cd._probe(name)
    P = cd.Paths(gx, pr)
    forms = (False, True) if pr.d + 2 <= 16 else (False,)
    c0sq = 3.0 / pr.params[0] ** 2 if pr.family == 1 else 1.0
    for expanded in forms:
        got, ab, li8 = _ivar_n1(gx, P, expanded, I8)
        _, _, ldm = _ivar_n1(gx, P, expanded, DMMA)
        assert li8 == ldm + SLICE_LAUNCHES
        budget = 8 * cd.EPS * c0sq * ab if expanded else 0.0
        cd.check_values(pr, got, f"INT8 core {'EXPANDED' if expanded else 'DIFF'}", budget=budget, square=True)
