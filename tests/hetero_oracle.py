"""Greedy IVAR oracles under a heteroscedastic noise function nu(x), for the tests and scripts/multigpu_check.py.

They are oracle/gpexp_oracle.py's greedy IVAR loops with the scalar noise replaced by nu; the per-step arithmetic is
that module's (ref_ivar_cost, fast_ivar_scores, both of which take a nugget vector).  With a constant nu they are
bit-identical to the float-noise oracles (tests/test_ivar_heteroscedastic.py checks that)."""
import math

import numpy as np

from oracle import gpexp_oracle as orc


def ref_greedy_ivar_nu(kern, cand, mc, n_points, noise_func):
    """orc.ref_greedy_ivar with the reference's heteroscedastic branch (experimentalDesign.py:110-114): the cost of
    design+{c} is ref_ivar_cost with the per-point nugget noise_func(design+{c}).  Returns (indices, per-step costs)."""
    ind, costs = [], []
    for _ in range(n_points):
        cost = np.full(cand.shape[0], np.inf)
        for c in range(cand.shape[0]):
            pts = np.vstack([cand[ind, :], cand[c:c + 1, :]])
            cost[c] = orc.ref_ivar_cost(kern, pts, mc, noise_func(pts))
        costs.append(cost)
        ind.append(int(np.argmin(cost)))
    return ind, costs


def fast_greedy_ivar_nu(kern, cand, mc, n_points, nu):
    """orc.fast_greedy_ivar with a per-candidate noise vector nu: den = var_D(c) + nu[c], and the appended rows are
    divided by sqrt(var_D(p) + nu[p]).  Integration points carry no noise.  Returns (indices, per-step costs)."""
    nu = np.asarray(nu, dtype=np.float64)
    c, m = cand.shape[0], mc.shape[0]
    w_c = np.zeros((n_points, c))
    w_m = np.zeros((n_points, m))
    var_c = kern.prior(cand).copy()
    var_m = kern.prior(mc).copy()
    ind, costs = [], []
    for n in range(n_points):
        cost = orc.fast_ivar_scores(kern, cand, mc, w_m[:n], var_m, w_c[:n], var_c, nu)
        costs.append(cost)
        p = int(np.argmin(cost))
        lnn = math.sqrt(var_c[p] + nu[p])
        col = w_c[:n, p].copy()
        row_c = (kern.gram(cand[p:p + 1], cand)[0] - col @ w_c[:n, :]) / lnn
        row_m = (kern.gram(cand[p:p + 1], mc)[0] - col @ w_m[:n, :]) / lnn
        w_c[n, :] = row_c
        w_m[n, :] = row_m
        var_c -= row_c * row_c
        var_m -= row_m * row_m
        ind.append(p)
    return ind, costs
