"""Greedy MI oracles under a per-point noise nu (one value per pool point), for tests/test_mi_heteroscedastic.py and
scripts/multigpu_check.py.

They restate oracle/gpexp_oracle.py's ref_mi_cost, ref_greedy_mi and fast_greedy_mi with the scalar nugget replaced by
nu on each subset: K_AA + diag nu_A in the numerator, K_S'S' + diag nu_S' in the denominator.  With a constant nu they
are bit-identical to the float-noise oracles (tests/test_mi_heteroscedastic.py checks that)."""
import math

import numpy as np

from oracle import gpexp_oracle as orc


def ref_mi_cost_nu(kern, pool, nu, index, index_added):
    """orc.ref_mi_cost with the scalar nugget replaced by nu on each subset: K_AA + diag nu_A in the numerator and
    K_S'S' + diag nu_S' (S' = V minus A minus {y}) in the denominator."""
    dim = pool.shape[1]
    point = pool[index, :].reshape(1, dim)
    var = kern.evaluate(point, point)
    added = pool[index_added, :].reshape(len(index_added), dim)
    kva = kern.evaluate(added, point)
    cov_num = orc.ref_covariance_matrix(kern, added, nu[index_added])
    numerator = var - np.dot(kva.T, np.dot(np.linalg.pinv(cov_num), kva))
    left = np.setdiff1d(np.arange(pool.shape[0]), index_added)
    left = np.setdiff1d(left, [index])
    pts_left = pool[left, :]
    kvl = kern.evaluate(pts_left, point)
    cov_den = orc.ref_covariance_matrix(kern, pts_left, nu[left])
    denominator = var - np.dot(kvl.T, np.dot(np.linalg.pinv(cov_den), kvl))
    return numerator / denominator


def ref_greedy_mi_nu(kern, pool, nu, n_points, start=0):
    """orc.ref_greedy_mi (the reference's pinv loop) with the per-point noise nu on each subset.  Returns (indices,
    per-step score vectors over the remaining options, per-step option index arrays)."""
    nu = np.asarray(nu, dtype=np.float64)
    ind = [start]
    options = np.setdiff1d(np.arange(pool.shape[0]), ind)
    scores, opts = [], []
    for _ in range(len(ind), n_points):
        out = np.zeros(len(options))
        for j, i in enumerate(options):
            out[j] = ref_mi_cost_nu(kern, pool, nu, int(i), ind)[0]
        scores.append(out)
        opts.append(options.copy())
        new = int(options[np.argmax(out)])
        ind.append(new)
        options = np.setdiff1d(options, new)
    return ind, scores, opts


def fast_greedy_mi_nu(kern, pool, nu, n_points, start=0):
    """orc.fast_greedy_mi with a per-point noise vector nu: the precision is (K_VV + diag nu)^-1, the appended rows are
    divided by sqrt(num[p] + nu[p]) and the denominator is 1/pd[y] - nu[y].  Returns (indices, per-step score vectors of
    length |V| with selected entries = -inf, per-step pivots num[p] + nu[p])."""
    nu = np.asarray(nu, dtype=np.float64)
    v = pool.shape[0]
    prec = np.linalg.inv(kern.gram(pool, pool) + np.diag(nu))
    num = kern.prior(pool).copy()
    w = np.zeros((n_points, v))
    selected = np.zeros(v, dtype=bool)
    ind, scores, pivots = [], [], []
    pd = np.diag(prec).copy()
    us = []

    def take(p):
        nonlocal pd
        n = len(ind)
        pivots.append(num[p] + nu[p])
        lnn = math.sqrt(num[p] + nu[p])
        row = (kern.gram(pool[p:p + 1], pool)[0] - w[:n, p] @ w[:n, :]) / lnn
        w[n, :] = row
        num[:] = num - row * row
        col = prec[:, p].copy()
        for u in us:
            col -= u * u[p]
        u = col / math.sqrt(col[p])
        us.append(u)
        pd = pd - u * u
        selected[p] = True
        ind.append(int(p))

    take(start)
    while len(ind) < n_points:
        den = 1.0 / np.where(selected, 1.0, pd) - nu
        s = np.where(selected, -np.inf, num / den)
        scores.append(s)
        take(int(np.argmax(s)))
    return ind, scores, pivots
