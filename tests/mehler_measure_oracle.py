"""CPU oracle of the closed-form IVAR over a product measure for Mehler kernels (costFunctionGP_IVAR.measure with
KernelMehlerND / KernelMehler1D, MeasureIVAREngine), built on oracle/gpexp_oracle.py's KernelSpec and the measure
description and box factor of tests/measure_oracle.py.  Plain numpy / scipy, direct formulas:

    mehler_phi, mehler_phi_diag     Phi(a, b) = int k(x, a) k(x, b) dmu(x) for a box or a Gaussian measure
    mehler_prior                    s = int k(x, x) dmu(x)
    fast_ivar_cost_mehler           int var_D dmu = s - tr(L^-1 Phi_DD L^-T) of a design
    fast_ivar_scores_mehler         exact cost of design + {c} for every candidate, and its rounding bound
    fast_greedy_ivar_mehler         the greedy loop over those scores, every factor rebuilt from scratch at every step

One dimension, parameter t (|t| < 1), r = 1 - t^2, m = (a + b) / 2:
    k(x, a) k(x, b) = r^-1 exp(m^2 - t^2 (a - b)^2 / (4 r)) exp(-(t x - m)^2 / r)
    GAUSS N(mu, sd^2), g = r + 2 t^2 sd^2:
        Phi_q = (r g)^-1/2 exp(-t^2 (a - b)^2 / (4 r) + [t^2 (2 sd^2 - 1) m^2 + 2 t mu m - t^2 mu^2] / g)
    BOX [lo, hi], u, v = sorted((t lo - m) / sqrt(r), (t hi - m) / sqrt(r)), w = |t| (hi - lo) / sqrt(r):
        Phi_q = r^-1 exp(m^2 - t^2 (a - b)^2 / (4 r)) J(u, v) / w,   J(u, v) = int_u^v e^{-s^2} ds  (1 e^{-u^2} at w = 0)
    s_q, c = t / (1 + t):
        GAUSS  r^-1/2 (1 - 2 c sd^2)^-1/2 exp(c mu^2 / (1 - 2 c sd^2)), finite only for 2 c sd^2 < 1
        BOX    r^-1/2 / (hi - lo) int_lo^hi e^{c x^2} dx   (erf form for c < 0, Dawson form for c > 0)"""
import math

import numpy as np

from oracle import gpexp_oracle as orc
from tests.measure_oracle import BOX, GAUSS, MeasureSpec, _box_tail_j  # noqa: F401

_GL_X, _GL_W = np.polynomial.legendre.leggauss(10)


def _phi(kern, meas, xa, xb):
    """Phi for coordinates xa[q], xb[q] (arrays that broadcast against each other): the exponents of all dimensions are
    summed before one exp, and values below 2^-1022 are returned as 0."""
    assert kern.family == orc.MEHLER, "this oracle is for Mehler kernels"
    S = 0.0
    F = 1.0
    for q in range(kern.dim):
        t = float(kern.t[q])
        r = (1.0 - t) * (1.0 + t)
        a, b = np.asarray(xa[q], dtype=np.float64), np.asarray(xb[q], dtype=np.float64)
        diff = a - b
        m = 0.5 * (a + b)
        S = S - t * t * diff * diff / (4.0 * r)
        if meas.kind == BOX:
            lo, hi = float(meas.p0[q]), float(meas.p1[q])
            tlo, thi = (t * lo, t * hi) if t >= 0.0 else (t * hi, t * lo)
            w = abs(t) * (hi - lo) / math.sqrt(r)
            u, v = (tlo - m) / math.sqrt(r), (thi - m) / math.sqrt(r)
            E, J = _box_tail_j(u, v, np.full(np.broadcast(u, v).shape, w))
            S = S + m * m + E
            F = F * (J / w if w > 0.0 else 1.0) / r
        else:
            mu, sd = float(meas.p0[q]), float(meas.p1[q])
            g = r + 2.0 * t * t * sd * sd
            S = S + (t * t * (2.0 * sd * sd - 1.0) * m * m + 2.0 * t * mu * m - t * t * mu * mu) / g
            F = F / math.sqrt(r * g)
    out = F * np.exp(S)
    return np.where(np.abs(out) < np.finfo(np.float64).tiny, 0.0, out)


def mehler_phi(kern, meas, X, Y):
    """Phi[i, j] = int k(x, X_i) k(x, Y_j) dmu(x) for a Mehler kernel and a product measure."""
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    return _phi(kern, meas, [X[:, q:q + 1] for q in range(kern.dim)], [Y[None, :, q] for q in range(kern.dim)])


def mehler_phi_diag(kern, meas, X):
    """Phi(x, x) per point."""
    X = np.asarray(X, dtype=np.float64)
    return _phi(kern, meas, [X[:, q] for q in range(kern.dim)], [X[:, q] for q in range(kern.dim)])


def _exp_sq_integral(c, lo, hi):
    """int_lo^hi exp(c x^2) dx.  c < 0: J(sqrt|c| lo, sqrt|c| hi) / sqrt|c| through _box_tail_j.  c > 0, with
    y = sqrt(c) x and Dawson's D(y) = e^{-y^2} int_0^y e^{s^2} ds: e^{v^2} D(v) + e^{u^2} D(-u) across 0,
    e^{b^2} (D(b) - e^{-(b - a)(b + a)} D(a)) on one side (b - a > 1 or its centre times its width > 1 there, so the
    bracket keeps a fixed share of D(b)), and 10-point Gauss-Legendre around the centre where the interval is narrow."""
    from scipy.special import dawsn
    if c == 0.0:
        return hi - lo
    rc = math.sqrt(abs(c))
    u, v, w = rc * lo, rc * hi, rc * (hi - lo)
    if c < 0.0:
        E, J = _box_tail_j(u, v, w)
        return float(np.exp(E) * J) / rc
    ctr = 0.5 * (u + v)
    if w <= 1.0 and abs(ctr) * w <= 1.0:
        h = 0.5 * w
        s = h * _GL_X
        return math.exp(ctr * ctr) * h * float(np.sum(_GL_W * np.exp((2.0 * ctr + s) * s))) / rc
    if u <= 0.0 <= v:
        return (math.exp(v * v) * dawsn(v) + math.exp(u * u) * dawsn(-u)) / rc
    a, b = min(abs(u), abs(v)), max(abs(u), abs(v))
    return math.exp(b * b) * (dawsn(b) - math.exp(-w * (a + b)) * dawsn(a)) / rc


def mehler_prior(kern, meas):
    """s = int k(x, x) dmu(x) = prod_q s_q.  ValueError for a Gaussian measure with 2 c_q sd_q^2 >= 1 (s infinite),
    naming the dimension and the largest admissible std."""
    s = 1.0
    for q in range(kern.dim):
        t = float(kern.t[q])
        if meas.kind == BOX:
            lo, hi = float(meas.p0[q]), float(meas.p1[q])
            s *= _exp_sq_integral(t / (1.0 + t), lo, hi) / ((hi - lo) * math.sqrt((1.0 - t) * (1.0 + t)))
        else:
            mu, sd = float(meas.p0[q]), float(meas.p1[q])
            num = 1.0 + t - 2.0 * t * sd * sd      # (1 + t)(1 - 2 c sd^2)
            if num <= 0.0:
                raise ValueError(f"Gaussian measure too wide in dimension {q}: std must be below "
                                 f"{math.sqrt((1.0 + t) / (2.0 * t))!r} for t = {t!r}")
            s *= math.exp(t * mu * mu / num) / math.sqrt((1.0 - t) * num)
    return s


def _state(kern, meas, design, cand, noise):
    """Direct factors of a design: (W, Z, Psi, var) with K_DD + diag(noise) = L L^T, W = L^-1 K(D, C),
    Z = L^-1 Phi(D, C), Psi = L^-1 Phi_DD L^-T and var = k(c, c) - |W[:, c]|^2."""
    from scipy.linalg import solve_triangular
    n = design.shape[0]
    nug = noise * np.ones(n) if np.isscalar(noise) else np.asarray(noise, dtype=np.float64)
    low = np.linalg.cholesky(kern.gram(design, design) + np.diag(nug))
    w = solve_triangular(low, kern.gram(design, cand), lower=True)
    z = solve_triangular(low, mehler_phi(kern, meas, design, cand), lower=True)
    t = solve_triangular(low, mehler_phi(kern, meas, design, design), lower=True)
    psi = solve_triangular(low, t.T, lower=True)
    return w, z, psi, kern.prior(cand) - np.sum(w * w, axis=0)


def fast_ivar_cost_mehler(kern, meas, design, noise):
    """int var_D(x) dmu(x) = s - tr(L^-1 Phi_DD L^-T) for the design (noise scalar or one nugget per design point)."""
    design = np.asarray(design, dtype=np.float64)
    s = mehler_prior(kern, meas)
    if design.shape[0] == 0:
        return s
    _, _, psi, _ = _state(kern, meas, design, design[:1], noise)
    return s - np.trace(psi)


def fast_ivar_scores_mehler(kern, meas, design, cand, noise, cand_noise=None):
    """Exact cost of design + {c} for every candidate c:
        score_c = |s - tr Psi - q_c / (var_D(c) + nu_c)|,   q_c = Phi_cc - 2 w_c.z_c + w_c.(Psi w_c)
    `noise` is the design's nugget (scalar or one per design point), nu_c = cand_noise[c] (default: the scalar noise);
    the reduction is 0 where var_D(c) + nu_c is numerically zero.  Returns (scores, bound) with
        bound_c = (n + 3) eps [(Phi_cc + 2 sum |w||z| + sum |w||Psi w|) / (var_D(c) + nu_c) + (n + 1) s]
    the bound of tests/measure_oracle.py's fast_ivar_scores_measure with s in place of the signal."""
    design = np.asarray(design, dtype=np.float64)
    cand = np.asarray(cand, dtype=np.float64)
    n = design.shape[0]
    s = mehler_prior(kern, meas)
    nu = np.broadcast_to(noise if cand_noise is None else cand_noise, (cand.shape[0],))
    phic = mehler_phi_diag(kern, meas, cand)
    if n:
        w, z, psi, var = _state(kern, meas, design, cand, noise)
        y = psi @ w
        base = s - np.trace(psi)
        q = phic - 2.0 * np.sum(w * z, axis=0) + np.sum(w * y, axis=0)
        mag = phic + 2.0 * np.sum(np.abs(w * z), axis=0) + np.sum(np.abs(w * y), axis=0)
    else:
        var, base, q, mag = kern.prior(cand), s, phic, phic
    den = var + nu
    tiny = den <= orc.ZERO_VAR_TOL * orc.kern_scale(kern)
    safe = np.where(tiny, 1.0, den)
    eps = np.finfo(np.float64).eps
    return (np.abs(base - np.where(tiny, 0.0, q / safe)),
            (n + 3) * eps * (np.where(tiny, 0.0, mag / safe) + (n + 1) * s))


def fast_greedy_ivar_mehler(kern, meas, cand, n_points, noise, *, with_bounds=False):
    """Greedy IVAR over the exact integral: at every step score all candidates with fast_ivar_scores_mehler (direct
    factors of the current design, no recurrence) and add the arg-min.  `noise` is a scalar or a per-candidate vector nu
    (the design then takes nu at its points).  Returns (indices, per-step score vectors) and with `with_bounds` the
    per-step rounding bounds as a third value."""
    cand = np.asarray(cand, dtype=np.float64)
    nu = np.broadcast_to(np.asarray(noise, dtype=np.float64), (cand.shape[0],))
    ind, costs, bounds = [], [], []
    for _ in range(n_points):
        sc, bd = fast_ivar_scores_mehler(kern, meas, cand[ind], cand, nu[ind], nu)
        costs.append(sc)
        bounds.append(bd)
        ind.append(int(np.argmin(sc)))
    return (ind, costs, bounds) if with_bounds else (ind, costs)
