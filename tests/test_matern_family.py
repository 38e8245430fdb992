"""Matern nu = 1/2 (GPX_MATERN12) and nu = 5/2 (GPX_MATERN52) through every layer: the oracle's closed forms, the ABI
constants, the nu -> family map, covariance values over the whole exponent range on every device path, the refusal of
the expanded-form prologue for nu = 1/2, and the design criteria against the CPU oracle.

k = s p(t) exp(-t), t = c0 |x - y|, c0 = sqrt(2 nu) / rho:  p = 1 (nu = 1/2), 1 + t + t^2/3 (nu = 5/2).
The covariance-domain probes reuse tests/test_covariance_domain.py (Paths, check_values) with `tpar = p(t) - 1`, so its
underflow bound (1 + tpar) max(1, s) 2^-1021 becomes p(t) max(1, s) 2^-1021.
"""
import os
import re
import sys

import mpmath
import numpy as np
import pytest

from oracle import gpexp_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DMMA, I8 = 1, 2
EINVAL = -1
NEW = {"matern12": orc.MATERN12, "matern52": orc.MATERN52}


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_closed_forms_equal_the_bessel_expression(nu):
    """s 2^(1-nu) / Gamma(nu) (c0 r)^nu K_nu(c0 r), c0 = sqrt(2 nu) / rho, from r = 1e-6 to 40 rho; r = 0 gives s."""
    from scipy.special import gamma, kv
    rho, s = 0.37, 1.7
    spec = {0.5: orc.KernelSpec.matern12(rho, s, 2), 1.5: orc.KernelSpec.matern32(rho, s, 2),
            2.5: orc.KernelSpec.matern52(rho, s, 2)}[nu]
    r = np.concatenate([np.geomspace(1e-6, 40 * rho, 400), [0.5 * rho, rho, 2 * rho]])
    x1 = np.zeros((r.size, 2))
    x2 = np.stack([0.6 * r, 0.8 * r], axis=1)
    got = spec.evaluateF(x1, x2)
    z = np.sqrt(2 * nu) * np.hypot(x2[:, 0], x2[:, 1]) / rho
    want = s * 2.0 ** (1 - nu) / gamma(nu) * z ** nu * kv(nu, z)
    assert _rel(got, want) <= 1e-13
    assert np.array_equal(spec.gram(x1[:5], x2[:5]).diagonal(), got[:5])
    assert np.all(spec.evaluateF(np.ones((3, 2)), np.ones((3, 2))) == s)
    assert np.all(orc.matern_closed_form(nu, np.zeros(2), rho, s) == s)


def test_header_constants_equal_the_binding():
    from gpexp_b200 import _lib
    text = open(os.path.join(ROOT, "include", "gpexp_b200.h")).read()
    defs = dict(re.findall(r"#define\s+(GPX_\w+)\s+(-?\d+)\b", text))
    assert (int(defs["GPX_MATERN12"]), int(defs["GPX_MATERN52"])) == (_lib.MATERN12, _lib.MATERN52) == \
        (orc.MATERN12, orc.MATERN52)
    fams = [int(defs[k]) for k in ("GPX_SE", "GPX_MATERN32", "GPX_MEHLER", "GPX_MATERN12", "GPX_MATERN52")]
    assert len(set(fams)) == 5 and fams[:3] == [0, 1, 2]


def test_prior_scale_of_the_new_families():
    from gpexp_b200 import _lib
    from gpexp_b200.engine import prior_scale
    assert prior_scale(_lib.MATERN12, [0.5, 2.5]) == 2.5
    assert prior_scale(_lib.MATERN52, [0.5, -3.0]) == 3.0


def _check_nu_map(cls, fams):
    for nu, fam in [(0.5, fams.MATERN12), (0.5 + 5e-11, fams.MATERN12), (1.5, fams.MATERN32), (2.5, fams.MATERN52),
                    (2.5 - 5e-11, fams.MATERN52)]:
        k = cls(0.3, 1.4, 2, nu=nu)
        assert k._gpx_spec() == (fam, 2, [0.3, 1.4]), nu
    for nu in (2.0, 0.5 + 1e-9, 1.0, 3.5):
        with pytest.raises(UnboundLocalError):
            cls(0.3, 1.4, 2, nu=nu)._gpx_spec()


def test_nu_maps_to_family_standalone():
    from gpexp_b200 import _lib
    from gpexp_b200 import kernels as K
    assert K.KernelIsoMatern(0.3, 1.4, 2).nu == 1.5
    _check_nu_map(K.KernelIsoMatern, _lib)


def test_nu_maps_to_family_on_the_patched_reference():
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        pytest.skip("no reference package available (set GPEXP_REFERENCE and run __graft_entry__.build() to stage it)")
    import gpexp_b200
    from gpexp_b200 import _lib
    gpexp_b200.install_as_gpExp(path)
    try:
        import gpExp.kernels as rk
        _check_nu_map(rk.KernelIsoMatern, _lib)
    finally:
        for name in [m for m in list(sys.modules) if m == "gpExp" or m.startswith("gpExp.")]:
            del sys.modules[name]


# ------------------------------------------------------------------------------------------------
# GPU harness
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    ed.VERBOSE = False
    from gpexp_b200 import _lib, device, engine, kernels
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space

    class NS:
        pass
    ns = NS()
    ns.torch, ns.ed, ns.lib, ns.L, ns.device, ns.engine, ns.gp, ns.kernels, ns.Space = \
        torch, ed, _lib.lib, _lib, device, engine, gpmod, kernels, Space
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")


def _core(gx, core):
    gx.check(gx.lib.gpx_set_ivar_core(gx.dev.h, core), "gpx_set_ivar_core")


# ------------------------------------------------------------------------------------------------
# GPU: covariance values over the whole exponent range (the contract of tests/test_covariance_domain.py)
# ------------------------------------------------------------------------------------------------
# t = c0 r from 0 past the table exp's flush point (t ~ 745), with the steps around where exp(-t) leaves the normal range
T_VALUES = [0.0, 1e-300, 1e-17, 1e-8, 1e-3, 0.5, 1.0, 2.0, 10.0, 100.0, 300.0, 600.0, 700.0, 707.5, 707.9, 708.2,
            708.39, 708.4, 709.0, 720.0, 740.0, 745.0, 746.0, 750.0]


def _mp_matern_nu(nu, rho, s):
    c0 = mpmath.sqrt(2 * mpmath.mpf(nu)) / mpmath.mpf(rho)

    def fn(x, y):
        r = mpmath.sqrt(sum((mpmath.mpf(float(p)) - mpmath.mpf(float(q))) ** 2 for p, q in zip(x, y)))
        t = c0 * r
        p = 1 + t + t * t / 3 if nu == 2.5 else mpmath.mpf(1)
        return mpmath.mpf(s) * p * mpmath.exp(-t), t, p - 1   # (k, exponent magnitude, tpar = p(t) - 1)
    return fn


def matern_nu_probe(family, signal):
    from tests.test_covariance_domain import _build
    nu = 0.5 if family == "matern12" else 2.5
    rho = 0.8
    x = np.array([0.3, -0.1])
    Y = np.array([x + np.array([0.6, 0.8]) * (t * rho / np.sqrt(2 * nu)) for t in T_VALUES])
    return _build(f"{family}_s{signal:g}", NEW[family], [rho, signal], x, Y, signal, _mp_matern_nu(nu, rho, signal))


SIGNALS = [2.0 ** -40, 1e-3, 0.3, 0.4999, 0.5, 0.7, 1.0, 1.7, 1e3, 2.0 ** 40]
_PROBES = {}


def _probe(family, signal):
    key = (family, signal)
    if key not in _PROBES:
        _PROBES[key] = matern_nu_probe(family, signal)
    return _PROBES[key]


@pytest.mark.gpu
@pytest.mark.parametrize("signal", SIGNALS)
@pytest.mark.parametrize("family", list(NEW))
def test_covariance_domain(gx, family, signal):
    """Every path of tests/test_covariance_domain.py: pairwise, append, Gram (paired stores and odd ld), matvec,
    gpx_trsm_gram, gpx_cov_from_factors and gpx_score_ivar (every ring, padded and not); nu = 5/2 also in expanded
    form, with the budget 8 eps (c0^2 / 6) (|alpha| + |beta|) of k's slope in the exponent at e = 0."""
    from tests.test_covariance_domain import DBL_MAX, EPS, Paths, check_values
    pr = _probe(family, signal)
    P = Paths(gx, pr)
    check_values(pr, P.pairwise(), "gpx_kernel_pairwise")
    check_values(pr, P.append_row(), "gpx_append_row")
    check_values(pr, P.gram(odd=False), "gpx_gram (paired stores)")
    check_values(pr, P.gram(odd=True), "gpx_gram (odd ld)")
    check_values(pr, P.matvec(), "gpx_gram_matvec")
    W, var = P.trsm()
    check_values(pr, W, "gpx_trsm_gram W")
    kyy = mpmath.mpf(pr.signal)
    for j in range(len(pr.Y)):
        want = kyy - pr.ref[j] ** 2
        if abs(kyy) < DBL_MAX / 4 and abs(pr.ref[j]) < 1e150:
            assert abs(mpmath.mpf(var[j]) - want) <= 1e-12 * (abs(kyy) + pr.ref[j] ** 2) + 1e-300, (pr.name, j)
    check_values(pr, P.cov(expanded=False)[0], "gpx_cov_from_factors DIFF")
    for padded in (True, False):
        for ring in ((0, 1, 2) if padded else (None,)):
            got, _ = P.ivar(expanded=False, padded=padded, ring=ring)
            check_values(pr, got, f"gpx_score_ivar DIFF padded={padded} ring={ring}", square=True)
    if family == "matern12":
        return  # no expanded form (test_expanded_form_is_refused_for_nu_half)
    c0sq6 = 5.0 / pr.params[0] ** 2 / 6.0
    got, ab = P.cov(expanded=True)
    check_values(pr, got, "gpx_cov_from_factors EXPANDED", budget=8 * EPS * c0sq6 * ab)
    for padded in (True, False):
        got, ab = P.ivar(expanded=True, padded=padded)
        check_values(pr, got, f"gpx_score_ivar EXPANDED padded={padded}", budget=8 * EPS * c0sq6 * ab, square=True)


@pytest.mark.gpu
def test_expanded_form_is_refused_for_nu_half(gx):
    """nu = 1/2: gpx_prep_side reports max|alpha| = +inf, gpx_score_ivar and gpx_cov_from_factors refuse
    GPX_PRO_EXPANDED with GPX_EINVAL, and prologue_operands picks the difference form; nu = 5/2 on centred uniform data
    keeps the expanded form."""
    dev, lib, ptr, L = gx.dev, gx.lib, gx.ptr, gx.L
    rng = np.random.default_rng(5)
    pts = rng.uniform(-1, 1, (300, 2))
    for fam, want in ((L.MATERN12, L.PRO_DIFF), (L.MATERN52, L.PRO_EXPANDED)):
        dev.set_kernel(fam, 2, [0.4, 1.0])
        dev.set_center(np.zeros(2))
        a, b = dev.points(pts[:200]), dev.points(pts[200:])
        mode, ra, rb = gx.device.prologue_operands(a, b)
        assert mode == want, fam
        ma = a.side(L.SIDE_A)[1]
        assert (ma == float("inf")) == (fam == L.MATERN12), (fam, ma)
    dev.set_kernel(L.MATERN12, 2, [0.4, 1.0])
    a, b = dev.points(pts[:200]), dev.points(pts[200:])
    (ra, _), (rb, _) = a.side(L.SIDE_A), b.side(L.SIDE_B)
    M, C = 200, 100
    vM, vC = dev.zeros(a.ld), dev.zeros(b.ld) + 1.0
    ws = dev.zeros(int(lib.gpx_score_ivar_workspace(dev.h, M, C)))
    score, best, idx = dev.zeros(b.ld), dev.zeros(1), dev.zeros(1, dtype=gx.torch.int64)
    for core in (I8, DMMA):
        _core(gx, core)
        try:
            rc = lib.gpx_score_ivar(dev.h, L.PRO_EXPANDED, None, a.ld, ptr(vM), ptr(ra), M, None, b.ld, ptr(vC), ptr(rb), C,
                                    0, 0.0, 0.0, None, ptr(ws), ptr(score), ptr(best), ptr(idx), dev.stream)
        finally:
            _core(gx, I8)
        assert rc == EINVAL and "MATERN12" in L.last_error(), (core, rc, L.last_error())
    out = dev.zeros(M, b.ld)
    rc = lib.gpx_cov_from_factors(dev.h, L.PRO_EXPANDED, None, a.ld, ptr(ra), M, None, b.ld, ptr(rb), C, 0, ptr(out),
                                  b.ld, dev.stream)
    assert rc == EINVAL and "MATERN12" in L.last_error()
    # the same calls in difference form run
    gx.check(lib.gpx_score_ivar(dev.h, L.PRO_DIFF, None, a.ld, ptr(vM), ptr(a.X), M, None, b.ld, ptr(vC), ptr(b.X), C, 0,
                                0.0, 0.0, None, ptr(ws), ptr(score), ptr(best), ptr(idx), dev.stream))
    gx.check(lib.gpx_cov_from_factors(dev.h, L.PRO_DIFF, None, a.ld, ptr(a.X), M, None, b.ld, ptr(b.X), C, 0, ptr(out),
                                      b.ld, dev.stream))
    dev.sync()
    ks = orc.KernelSpec.matern12(0.4, 1.0, 2)
    assert np.max(np.abs(out[:, :C].cpu().numpy() - ks.gram(pts[:200], pts[200:]))) <= 1e-14


# far pairs: the test_ivar_contraction_exact geometry (d = 1, integration points at +50, candidates at -50), with rho
# putting every t = c0 |x - y| between ~2400 and ~4600, far past the table exp's flush point
FAR = {"matern12": (orc.MATERN12, [0.04, 1.0], 50.0), "matern52": (orc.MATERN52, [0.05, 1.0], 50.0)}


@pytest.mark.gpu
@pytest.mark.parametrize("family,expanded", [("matern12", False), ("matern52", False), ("matern52", True)])
def test_far_pairs_give_zero_scores(gx, monkeypatch, family, expanded):
    """All-zero W with every covariance flushed: scores are exactly 0 on the INT8, tensor-map and generic cores, and the
    store kernel returns k = 0 for every pair (test_zero_factors_give_zero_scores for the new families)."""
    from tests import test_ivar_contraction_exact as tce
    monkeypatch.setitem(tce.FAMILIES, family, FAR[family])
    for padded in (True, False):
        P = tce.Problem(gx, family, expanded, tce.M_DEF, tce.C_DEF, 33, padded=padded)
        cores = (I8, DMMA) if padded else (I8,)
        launches = {}
        for core in cores:
            got, _, _, launches[core] = P.score(core)
            assert np.all(got == 0.0), (family, expanded, padded, core, got[got != 0][:4])
        if padded:
            assert launches[I8] == launches[DMMA] + tce.SLICE_LAUNCHES
        assert np.all(P.cov(tce._unpadded(tce.C_DEF)) == 0.0)
        P0 = tce.Problem(gx, family, expanded, tce.M_DEF, tce.C_DEF, 0, padded=padded)
        assert np.all(P0.score(I8)[0] == 0.0) and np.all(P0.cov(tce._unpadded(tce.C_DEF)) == 0.0)


# ------------------------------------------------------------------------------------------------
# GPU: the design criteria against the CPU oracle
# ------------------------------------------------------------------------------------------------
RHO = {"matern12": 0.5, "matern52": 0.3}  # cond(K_DD + 1e-4 I) of the designs below stays <~ 1e5
NOISE = 1e-4


def _kernels(gx, family, signal=1.3, d=3):
    nu = 0.5 if family == "matern12" else 2.5
    ks = (orc.KernelSpec.matern12 if family == "matern12" else orc.KernelSpec.matern52)(RHO[family], signal, d)
    return ks, gx.kernels.KernelIsoMatern(RHO[family], signal, d, nu=nu)


LOOP_MODES = ["trace_i8", "trace_dmma", "trace_resident", "loop_i8", "loop_dmma", "resident", "one_kernel"]
N_PICK = 16


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(NEW))
def test_greedy_ivar_every_loop_mode_matches_oracle(gx, family):
    """INT8 and DMMA contraction, traced and C-side loops, resident multi-launch and the one-kernel loop: identical picks
    and 1e-9 relative scores; then scoreCandidatesIVAR and costFunctionGP_IVAR.evaluate of the oracle's designs."""
    ed = gx.ed
    rng = np.random.default_rng(41)
    cand, mc = rng.uniform(-1, 1, (700, 3)), rng.uniform(-1, 1, (900, 3))
    ks, k = _kernels(gx, family)
    ref_idx, ref_costs = orc.fast_greedy_ivar(ks, cand, mc, N_PICK, NOISE)
    want = np.array([c[i] for c, i in zip(ref_costs, ref_idx)])
    cf = ed.costFunctionGP_IVAR(gx.gp.GP(k, NOISE), 1, gx.Space(3, None, None), mcPoints=mc)
    launches = {}
    for mode in LOOP_MODES:
        _core(gx, DMMA if mode.endswith("dmma") else I8)
        try:
            resident = mode in ("trace_resident", "resident", "one_kernel")
            eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N_PICK, resident=resident)
            if mode.startswith("trace"):
                eng.score_trace = []
            if resident:
                eng.ONE_KERNEL_PAIRS = cand.shape[0] * mc.shape[0] if mode == "one_kernel" else 0
            l0 = gx.dev.launches
            idx = eng.run(N_PICK)
            launches[mode] = gx.dev.launches - l0
        finally:
            _core(gx, I8)
        assert [int(i) for i in idx] == ref_idx, (family, mode)
        assert _rel(eng.pick_scores[:N_PICK].cpu().numpy(), want) <= 1e-9, (family, mode)
        if eng.score_trace is not None:
            for s, c in enumerate(eng.score_trace):
                assert _rel(c, ref_costs[s]) <= 1e-9, (family, mode, s)
    assert launches["one_kernel"] < launches["resident"], launches
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, N_PICK, returnIndices=True)
    assert [int(i) for i in idx] == ref_idx
    assert _rel(cf.lastScores, want) <= 1e-9
    for s in (1, 5, N_PICK - 1):
        costs, best = ed.scoreCandidatesIVAR(cf, cand[ref_idx[:s]], cand)
        assert best == ref_idx[s] and _rel(costs, ref_costs[s]) <= 1e-9, (family, s)
        one = ed.costFunctionGP_IVAR(gx.gp.GP(k, NOISE), s + 1, gx.Space(3, None, None), mcPoints=mc)
        assert _rel(one.evaluate(cand[ref_idx[: s + 1]]), want[s]) <= 1e-9, (family, s)


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(NEW))
def test_gp_posterior_and_loglike_match_oracle(gx, family):
    """GP.evaluateVariance, GP.evaluate (mean; compvar=2 covariance) and the loglikeParams value."""
    rng = np.random.default_rng(42)
    nodes, query = rng.uniform(-1, 1, (120, 3)), rng.uniform(-1, 1, (2000, 3))
    fvals = np.sin(3 * nodes[:, 0]) + nodes[:, 1] * nodes[:, 2]
    ks, k = _kernels(gx, family)
    g = gx.gp.GP(k, NOISE)
    g.train(nodes, fvals)
    var = g.evaluateVariance(query)
    ref = orc.fast_posterior_variance(ks, nodes, query, NOISE)
    assert np.max(np.abs(var - ref)) <= 1e-9 * ks.signal
    from scipy.linalg import cho_factor, cho_solve
    cf = cho_factor(ks.gram(nodes, nodes) + NOISE * np.eye(len(nodes)), lower=True)
    kq = ks.gram(query[:40], nodes)
    mean_ref = kq @ cho_solve(cf, fvals - g.gpPriorMean(nodes))
    cov_ref = ks.gram(query[:40], query[:40]) - kq @ cho_solve(cf, kq.T)
    mean, cov = g.evaluate(query[:40], compvar=2)
    mean0 = mean - g.gpPriorMean(query[:40])
    assert np.max(np.abs(mean0 - mean_ref)) <= 1e-9 * max(1.0, np.max(np.abs(mean_ref)))
    assert np.max(np.abs(cov - cov_ref)) <= 1e-9 * ks.signal
    ll = g.loglikeParams(nodes, fvals)
    ll_ref = orc.fast_loglike(ks, nodes, fvals, NOISE)
    assert abs(ll - ll_ref) <= 1e-9 * abs(ll_ref)
    with pytest.raises(AttributeError):
        g.loglikeParams(nodes, fvals, returnDeriv=1)   # derivatives stay squared-exponential only


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(NEW))
def test_greedy_var_and_mi_match_oracle(gx, family):
    ed = gx.ed
    rng = np.random.default_rng(43)
    ks, k = _kernels(gx, family)
    pool = rng.uniform(-1, 1, (3000, 3))
    vidx, _ = orc.fast_greedy_var(ks, pool, 30)
    pts = ed.performGreedyVarExperimentalDesign(k, pool, 30, 3)
    assert np.array_equal(pts, pool[vidx])
    pool = rng.uniform(-1, 1, (600, 3))
    fidx, _ = orc.fast_greedy_mi(ks, pool, NOISE, 12, start=2)
    cf = ed.costFunctionGP_MI(gx.gp.GP(k, NOISE), 12, gx.Space(3, None, None), nmc=600, mcpoints=pool)
    ed.performGreedyMIExperimentalDesign(cf, 12, start=2)
    assert [int(i) for i in cf.lastIndices] == fidx


def nu_span(p):
    """1e-5 at x0 = -1 to 1e-3 at x0 = 1."""
    return 1e-5 * 1e2 ** np.clip((p[:, 0] + 1.0) / 2.0, 0.0, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(NEW))
def test_noise_function_and_mc_weights(gx, family):
    """The new families under a heteroscedastic noise function and under weighted integration points."""
    ed = gx.ed
    rng = np.random.default_rng(44)
    cand, mc = rng.uniform(-1, 1, (600, 3)), rng.uniform(-1, 1, (800, 3))
    ks, k = _kernels(gx, family)
    ref_idx, ref_costs = orc.fast_greedy_ivar(ks, cand, mc, 12, nu_span(cand))
    cf = ed.costFunctionGP_IVAR(gx.gp.GP(k, 0.5), 1, gx.Space(3, None, None, noise=nu_span), mcPoints=mc)
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True)
    assert [int(i) for i in idx] == ref_idx
    assert _rel(cf.lastScores, [c[i] for c, i in zip(ref_costs, ref_idx)]) <= 1e-9
    w = rng.uniform(0.0, 2.0, mc.shape[0]) / mc.shape[0]
    ref_idx, ref_costs = orc.fast_greedy_ivar(ks, cand, mc, 12, NOISE, mc_weights=w)
    cf = ed.costFunctionGP_IVAR(gx.gp.GP(k, NOISE), 1, gx.Space(3, None, None), mcPoints=mc, mcWeights=w)
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, 12, returnIndices=True)
    assert [int(i) for i in idx] == ref_idx
    assert _rel(cf.lastScores, [c[i] for c, i in zip(ref_costs, ref_idx)]) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(NEW))
def test_i8_and_dmma_pick_the_same_designs(gx, family):
    from tests.test_ivar_int8_core import SLICE_LAUNCHES
    rng = np.random.default_rng(7)
    cand, mc = rng.uniform(-1, 1, (1200, 3)), rng.uniform(-1, 1, (1500, 3))
    _, k = _kernels(gx, family)
    picks, launches = {}, {}
    try:
        for core in (DMMA, I8):
            _core(gx, core)
            cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, NOISE), 1, gx.Space(3, None, None), mcPoints=mc)
            l0 = gx.dev.launches
            idx = gx.ed.performGreedyIVARExperimentalDesign(cf, cand, 48, returnIndices=True, resident=False)
            launches[core] = gx.dev.launches - l0
            picks[core] = [int(i) for i in idx]
    finally:
        _core(gx, I8)
    assert launches[I8] == launches[DMMA] + SLICE_LAUNCHES * 47
    assert picks[DMMA] == picks[I8]
