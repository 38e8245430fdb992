"""CPU oracle of the closed-form IVAR over a product measure for squared-exponential kernels (costFunctionGP_IVAR.measure,
MeasureIVAREngine), built on oracle/gpexp_oracle.py's KernelSpec.  Plain numpy / scipy, direct formulas:

    measure_phi, measure_phi_diag   Phi(a, b) = int k(x, a) k(x, b) dmu(x) for a box or a Gaussian measure
    fast_ivar_cost_measure          int var_D dmu = s - tr(L^-1 Phi_DD L^-T) of a design
    fast_ivar_scores_measure        exact cost of design + {c} for every candidate, and its rounding bound
    fast_greedy_ivar_measure        the greedy loop over those scores, every factor rebuilt from scratch at every step"""
import math
from dataclasses import dataclass

import numpy as np

from oracle import gpexp_oracle as orc

BOX, GAUSS = 1, 2


@dataclass
class MeasureSpec:
    """A product probability measure: BOX = uniform on [lo_q, hi_q] (p0 = lo, p1 = hi), GAUSS = N(mean_q, std_q^2)
    (p0 = mean, p1 = std)."""

    kind: int
    p0: np.ndarray
    p1: np.ndarray

    @staticmethod
    def box(lo, hi):
        return MeasureSpec(BOX, np.atleast_1d(np.asarray(lo, dtype=np.float64)), np.atleast_1d(np.asarray(hi, dtype=np.float64)))

    @staticmethod
    def gauss(mean, std):
        return MeasureSpec(GAUSS, np.atleast_1d(np.asarray(mean, dtype=np.float64)),
                           np.atleast_1d(np.asarray(std, dtype=np.float64)))


_GL_X, _GL_W = np.polynomial.legendre.leggauss(10)


def _box_tail_j(u, v, width):
    """(E, F) with int_u^v exp(-t^2) dt = exp(E) F elementwise (u < v, width = v - u formed from the box's own width,
    not by cancellation of u and v): Gauss-Legendre where the interval is narrow
    (both erf and erfc differences cancel there), erf where the interval holds 0 or starts within 1/2 of it, and the
    erfcx form, whose exponent -a^2 joins the caller's exponent sum, in the tails."""
    from scipy.special import erf, erfcx
    u, v, width = np.broadcast_arrays(np.asarray(u, dtype=np.float64), np.asarray(v, dtype=np.float64), width)
    c = 0.5 * (u + v)
    a = np.minimum(np.abs(u), np.abs(v))
    b = np.maximum(np.abs(u), np.abs(v))
    narrow = (width <= 1.0) & (np.abs(c) * width <= 1.0)
    straddle = ~narrow & (u <= 0.0) & (v >= 0.0)
    near = ~narrow & ~straddle & (a < 0.5)
    tail = ~narrow & ~straddle & ~near
    half_sqrt_pi = 0.5 * math.sqrt(math.pi)
    E = np.where(narrow, -c * c, np.where(tail, -a * a, 0.0))
    h = 0.5 * width
    s = h[..., None] * _GL_X
    with np.errstate(over="ignore", invalid="ignore"):
        gl = h * np.sum(_GL_W * np.exp(-(2.0 * c[..., None] + s) * s), axis=-1)
        F = np.where(narrow, gl,
            np.where(straddle, half_sqrt_pi * (erf(v) + erf(-u)),
            np.where(near, half_sqrt_pi * (erf(b) - erf(a)),
                     half_sqrt_pi * (erfcx(a) - np.exp(-width * (a + b)) * erfcx(b)))))
    return E, F


def _phi(kern, meas, xa, xb):
    """Phi for coordinates xa[q], xb[q] (arrays that broadcast against each other), one dimension at a time."""
    assert kern.family == orc.SE, "the closed form is for squared-exponential kernels"
    S = 0.0
    F = kern.signal * kern.signal
    for q in range(kern.dim):
        cl = kern.cl[q]
        diff = xa[q] - xb[q]
        m = 0.5 * (xa[q] + xb[q])
        S = S - diff * diff / (4.0 * cl * cl)
        if meas.kind == BOX:
            lo, hi = meas.p0[q], meas.p1[q]
            E, J = _box_tail_j((lo - m) / cl, (hi - m) / cl, (hi - lo) / cl)
            S = S + E
            F = F * (J * (cl / (hi - lo)))
        else:
            mu, sd = meas.p0[q], meas.p1[q]
            t = (m - mu) / math.sqrt(cl * cl + 2.0 * sd * sd)
            S = S - t * t
            F = F / math.sqrt(1.0 + 2.0 * sd * sd / (cl * cl))
    out = F * np.exp(S)
    return np.where(np.abs(out) < np.finfo(np.float64).tiny, 0.0, out)


def measure_phi(kern, meas, X, Y):
    """Phi[i, j] = int k(x, X_i) k(x, Y_j) dmu(x) for an SE kernel (iso or ARD) and a product measure:
        s^2 prod_q exp(-(X_iq - Y_jq)^2 / (4 cl_q^2)) I_q(m_q),   m = (X_i + Y_j) / 2
        BOX    I_q(m) = cl sqrt(pi) / (2 (hi - lo)) (erf((hi - m)/cl) - erf((lo - m)/cl))
        GAUSS  I_q(m) = (1 + 2 std^2/cl^2)^-1/2 exp(-(m - mean)^2 / (cl^2 + 2 std^2))
    The exponents of all dimensions are summed before one exp; values below 2^-1022 are returned as 0."""
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    return _phi(kern, meas, [X[:, q:q + 1] for q in range(kern.dim)], [Y[None, :, q] for q in range(kern.dim)])


def measure_phi_diag(kern, meas, X):
    """Phi(x, x) per point."""
    X = np.asarray(X, dtype=np.float64)
    return _phi(kern, meas, [X[:, q] for q in range(kern.dim)], [X[:, q] for q in range(kern.dim)])


def _measure_state(kern, meas, design, cand, noise):
    """Direct factors of a design: (W, Z, Psi, var) with K_DD + diag(noise) = L L^T, W = L^-1 K(D, C),
    Z = L^-1 Phi(D, C), Psi = L^-1 Phi_DD L^-T and var = k(c, c) - |W[:, c]|^2."""
    from scipy.linalg import solve_triangular
    n = design.shape[0]
    nug = noise * np.ones(n) if np.isscalar(noise) else np.asarray(noise, dtype=np.float64)
    low = np.linalg.cholesky(kern.gram(design, design) + np.diag(nug))
    w = solve_triangular(low, kern.gram(design, cand), lower=True)
    z = solve_triangular(low, measure_phi(kern, meas, design, cand), lower=True)
    t = solve_triangular(low, measure_phi(kern, meas, design, design), lower=True)
    psi = solve_triangular(low, t.T, lower=True)
    return w, z, psi, kern.prior(cand) - np.sum(w * w, axis=0)


def fast_ivar_cost_measure(kern, meas, design, noise):
    """int var_D(x) dmu(x) = s - tr(L^-1 Phi_DD L^-T) for the design (noise scalar or one nugget per design point)."""
    design = np.asarray(design, dtype=np.float64)
    if design.shape[0] == 0:
        return kern.signal
    _, _, psi, _ = _measure_state(kern, meas, design, design[:1], noise)
    return kern.signal - np.trace(psi)


def fast_ivar_scores_measure(kern, meas, design, cand, noise, cand_noise=None):
    """Exact cost of design + {c} for every candidate c:
        score_c = |s - tr Psi - q_c / (var_D(c) + nu_c)|,   q_c = Phi_cc - 2 w_c.z_c + w_c.(Psi w_c)
    `noise` is the design's nugget (scalar or one per design point), nu_c = cand_noise[c] (default: the scalar noise);
    the reduction is 0 where var_D(c) + nu_c is numerically zero, as in fast_ivar_scores.  Returns (scores, bound) with
        bound_c = (n + 3) eps [(Phi_cc + 2 sum |w||z| + sum |w||Psi w|) / (var_D(c) + nu_c) + (n + 1) s]
    the rounding bound of q_c / (var + nu) when q_c is formed from stored rows W, Z, Y = Psi W (first term, 0 where the
    reduction is dropped), plus that of s - tr Psi, a sum of n diagonal entries each formed by a length-n substitution."""
    design = np.asarray(design, dtype=np.float64)
    cand = np.asarray(cand, dtype=np.float64)
    n = design.shape[0]
    nu = np.broadcast_to(noise if cand_noise is None else cand_noise, (cand.shape[0],))
    phic = measure_phi_diag(kern, meas, cand)
    if n:
        w, z, psi, var = _measure_state(kern, meas, design, cand, noise)
        y = psi @ w
        base = kern.signal - np.trace(psi)
        q = phic - 2.0 * np.sum(w * z, axis=0) + np.sum(w * y, axis=0)
        mag = phic + 2.0 * np.sum(np.abs(w * z), axis=0) + np.sum(np.abs(w * y), axis=0)
    else:
        var, base, q, mag = kern.prior(cand), kern.signal, phic, phic
    den = var + nu
    tiny = den <= orc.ZERO_VAR_TOL * orc.kern_scale(kern)
    safe = np.where(tiny, 1.0, den)
    eps = np.finfo(np.float64).eps
    return (np.abs(base - np.where(tiny, 0.0, q / safe)),
            (n + 3) * eps * (np.where(tiny, 0.0, mag / safe) + (n + 1) * abs(kern.signal)))


def fast_greedy_ivar_measure(kern, meas, cand, n_points, noise, *, with_bounds=False):
    """Greedy IVAR over the exact integral: at every step score all candidates with fast_ivar_scores_measure (direct
    factors of the current design, no recurrence) and add the arg-min.  `noise` is a scalar or a per-candidate vector nu
    (the design then takes nu at its points).  Returns (indices, per-step score vectors) and with `with_bounds` the
    per-step rounding bounds as a third value."""
    cand = np.asarray(cand, dtype=np.float64)
    nu = np.broadcast_to(np.asarray(noise, dtype=np.float64), (cand.shape[0],))
    ind, costs, bounds = [], [], []
    for _ in range(n_points):
        sc, bd = fast_ivar_scores_measure(kern, meas, cand[ind], cand, nu[ind], nu)
        costs.append(sc)
        bounds.append(bd)
        ind.append(int(np.argmin(sc)))
    return (ind, costs, bounds) if with_bounds else (ind, costs)
