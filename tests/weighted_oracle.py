"""Greedy IVAR oracles with weighted integration points, for the tests and scripts/multigpu_check.py.

The cost of design D is |sum_m w_m var_D(x_m)| instead of the Monte-Carlo mean; w = 1/M is the plain cost.
ref_greedy_ivar_w is oracle/gpexp_oracle.py's pinv loop with the reference's variance (ref_evaluate_variance) weighted;
fast_greedy_ivar_w is fast_greedy_ivar restated with w (and an optional per-candidate noise vector nu, as in
tests/hetero_oracle.py).  Every weighted square is formed as (w v) v, the form the kernels use, so that w = 2^-k scales
each term, and therefore each sum, exactly: with M = 2^k and w = 1/M both reproduce the unweighted oracles bit for bit."""
import math

import numpy as np

from oracle import gpexp_oracle as orc


def ref_ivar_cost_w(kern, design, mc, noise, w):
    """orc.ref_ivar_cost with weights: |sum_m w_m var(x_m)|, var from the reference's pinv arithmetic."""
    _, prec = orc.ref_add_nodes(kern, design, noise)
    var_mc = orc.ref_evaluate_variance(kern, design, prec, mc)
    return abs(np.sum(w * var_mc))


def ref_greedy_ivar_w(kern, cand, mc, n_points, noise, w, noise_func=None):
    """orc.ref_greedy_ivar with the weighted cost; with noise_func the nugget of design+{c} is noise_func(design+{c})
    (the reference's heteroscedastic branch) and `noise` is not used.  Returns (indices, per-step costs)."""
    w = np.asarray(w, dtype=np.float64)
    ind, costs = [], []
    for _ in range(n_points):
        cost = np.full(cand.shape[0], np.inf)
        for c in range(cand.shape[0]):
            pts = np.vstack([cand[ind, :], cand[c:c + 1, :]])
            cost[c] = ref_ivar_cost_w(kern, pts, mc, noise if noise_func is None else noise_func(pts), w)
        costs.append(cost)
        ind.append(int(np.argmin(cost)))
    return ind, costs


def fast_ivar_scores_w(kern, cand, mc, w_m, var_m, w_c, var_c, noise, w, block=4096):
    """orc.fast_ivar_scores with weights: | sum_m w_m var_D(m) - sum_m (w_m cov_D(m,c)) cov_D(m,c) / (var_D(c) + noise) |,
    the reduction 0 where the denominator is numerically zero.  `noise` is a scalar or a per-candidate vector."""
    c = cand.shape[0]
    base = np.sum(w * var_m)
    r = np.zeros(c)
    for c0 in range(0, c, block):
        cov = kern.gram(mc, cand[c0:c0 + block]) - w_m.T @ w_c[:, c0:c0 + block]
        r[c0:c0 + block] = np.sum((w[:, None] * cov) * cov, axis=0)
    den = var_c + noise
    tiny = den <= orc.ZERO_VAR_TOL * orc.kern_scale(kern, cand)
    red = np.where(tiny, 0.0, r / np.where(tiny, 1.0, den))
    return np.abs(base - red)


def fast_greedy_ivar_w(kern, cand, mc, n_points, noise, w, nu=None):
    """orc.fast_greedy_ivar with weights; nu (per-candidate noise vector) replaces the scalar noise when given.
    Returns (indices, per-step costs)."""
    w = np.asarray(w, dtype=np.float64)
    c, m = cand.shape[0], mc.shape[0]
    noise = noise if nu is None else np.asarray(nu, dtype=np.float64)
    w_c = np.zeros((n_points, c))
    w_m = np.zeros((n_points, m))
    var_c = kern.prior(cand).copy()
    var_m = kern.prior(mc).copy()
    ind, costs = [], []
    for n in range(n_points):
        cost = fast_ivar_scores_w(kern, cand, mc, w_m[:n], var_m, w_c[:n], var_c, noise, w)
        costs.append(cost)
        p = int(np.argmin(cost))
        lnn = math.sqrt(var_c[p] + (noise if nu is None else noise[p]))
        col = w_c[:n, p].copy()
        row_c = (kern.gram(cand[p:p + 1], cand)[0] - col @ w_c[:n, :]) / lnn
        row_m = (kern.gram(cand[p:p + 1], mc)[0] - col @ w_m[:n, :]) / lnn
        w_c[n, :] = row_c
        w_m[n, :] = row_m
        var_c -= row_c * row_c
        var_m -= row_m * row_m
        ind.append(p)
    return ind, costs


def gauss_legendre_grid(n, d, lo=-1.0, hi=1.0):
    """Tensor Gauss-Legendre rule of n^d nodes on [lo, hi]^d: (points (n^d, d), weights summing to the box volume)."""
    x, w = np.polynomial.legendre.leggauss(n)
    x = lo + (x + 1.0) * (hi - lo) / 2.0
    w = w * (hi - lo) / 2.0
    grids = np.meshgrid(*([x] * d), indexing="ij")
    wgrid = np.meshgrid(*([w] * d), indexing="ij")
    pts = np.stack([g.ravel() for g in grids], axis=1)
    return pts, np.prod(np.stack([g.ravel() for g in wgrid], axis=1), axis=1)
