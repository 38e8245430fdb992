"""CPU oracles of the exchange refinement of discrete MI and maximum-variance designs (refineGreedyMIExperimentalDesign,
refineGreedyVarExperimentalDesign), built on oracle/gpexp_oracle.py and tests/ivar_exchange_oracle.py:

    fast_exchange_mi    the queue-ordered MI pass, refactoring A minus the removed point and S = V minus A from scratch at
                        every step: num(y) = var(y | A) with nugget nu_A, den(y) = 1 / [(K_SS + diag nu_S)^-1]_yy - nu_y
    ref_exchange_mi     the same decisions from the reference's pinv loop (ref_mi_cost), for |V| ~ 60
    fast_exchange_var   the queue-ordered maximum-variance pass (nugget 0), A minus the removed point refactored from
                        scratch; the first n_fixed points are never removed
    mi_objective        I(y_A; y_{V minus A}) = 1/2 (logdet S_AA + logdet S_SS - logdet S_VV), S = K + diag nu
    var_objective       logdet K_AA + sum_{i in A} log w_i

The rule for maximised scores: each step removes the oldest exchangeable point, scores every pool point against the other
n - 1 points, and appends the arg-max challenger (lowest index on ties) only if its score exceeds (1 + rtol) x the removed
point's own score; otherwise the removed point returns.  A sweep decides every exchangeable point once; the pass stops
after a sweep without a swap or after max_sweeps."""
import numpy as np
from scipy.linalg import solve_triangular

from oracle import gpexp_oracle as orc


def _decide_max(score, inc, rtol):
    """(winner, swapped, margin), as ivar_exchange_oracle._decide for maximised scores: margin = relative distance of the
    best challenger from the threshold (1 + rtol) score[inc] and, when it swaps in, from the runner-up challenger."""
    c = int(np.argmax(score))
    thr = (1.0 + rtol) * score[inc]
    swapped = bool(score[c] > thr)
    others = np.delete(score, inc)
    others = others[np.isfinite(others)]
    if others.size == 0:
        return int(inc), False, np.inf
    top = -np.partition(-others, min(1, others.size - 1))
    margin = abs(top[0] - thr) / abs(thr)
    if swapped and others.size > 1:
        margin = min(margin, (top[0] - top[1]) / abs(top[0]))
    return (c if swapped else int(inc)), swapped, margin


def _exchange_max(score_all, indices, rtol, max_sweeps, first=0):
    """Returns (final indices in factor order, score of the point put back at every step, swaps per sweep, margins, and
    for every step (removed point, winner, removed point's score, winner's score))."""
    design = [int(i) for i in indices]
    steps = len(design) - first
    scores, swaps, margins, moves = [], [], [], []
    for _ in range(max_sweeps if steps > 0 else 0):
        k = 0
        for _ in range(steps):
            inc = design[first]
            rest = design[:first] + design[first + 1:]
            s = score_all(rest)
            win, swapped, margin = _decide_max(s, inc, rtol)
            design = rest + [win]
            scores.append(float(s[win]))
            margins.append(margin)
            moves.append((inc, win, float(s[inc]), float(s[win])))
            k += swapped
        swaps.append(k)
        if k == 0:
            break
    return design, scores, swaps, margins, moves


def _nu(noise, v):
    return np.broadcast_to(np.asarray(noise, dtype=np.float64), (v,))


def mi_scores(kern, pool, rest, noise):
    """Greedy MI score of every pool point given A = rest, from scratch (-inf on A)."""
    v = pool.shape[0]
    nu = _nu(noise, v)
    prior = kern.prior(pool)
    if rest:
        low = np.linalg.cholesky(kern.gram(pool[rest], pool[rest]) + np.diag(nu[rest]))
        w = solve_triangular(low, kern.gram(pool[rest], pool), lower=True)
        num = prior - np.sum(w * w, axis=0)
    else:
        num = prior.copy()
    s_idx = np.setdiff1d(np.arange(v), rest)
    pd = np.diag(np.linalg.inv(kern.gram(pool[s_idx], pool[s_idx]) + np.diag(nu[s_idx])))
    out = np.full(v, -np.inf)
    out[s_idx] = num[s_idx] / (1.0 / pd - nu[s_idx])
    return out


def fast_exchange_mi(kern, pool, indices, noise, rtol, max_sweeps):
    """The MI exchange pass by brute force.  ``noise`` is a scalar or a per-point vector nu."""
    return _exchange_max(lambda rest: mi_scores(kern, pool, rest, noise), indices, rtol, max_sweeps)


def ref_exchange_mi(kern, pool, indices, noise, rtol, max_sweeps):
    """The same pass with every score from the reference's loop (ref_mi_cost: two pinv's per pool point)."""
    def score_all(rest):
        out = np.full(pool.shape[0], -np.inf)
        for y in np.setdiff1d(np.arange(pool.shape[0]), rest):
            out[y] = float(np.ravel(orc.ref_mi_cost(kern, pool, noise, int(y), list(rest)))[0])
        return out

    return _exchange_max(score_all, indices, rtol, max_sweeps)


def _logdet(m):
    sign, val = np.linalg.slogdet(m)
    assert sign > 0
    return val


def mi_objective(kern, pool, indices, noise):
    """I(y_A; y_{V minus A}) in nats for the noisy observations, Sigma = K + diag nu."""
    v = pool.shape[0]
    sig = kern.gram(pool, pool) + np.diag(_nu(noise, v))
    a = list(indices)
    s = np.setdiff1d(np.arange(v), a)
    return 0.5 * (_logdet(sig[np.ix_(a, a)]) + _logdet(sig[np.ix_(s, s)]) - _logdet(sig))


def precision_state(kern, pool, indices, noise):
    """(U_Q, Us, pd) of the design A = indices from scratch: Q = (K_VV + diag nu)^-1, Q_AA = U_Q^T U_Q,
    Us = U_Q^-T Q(A, V), pd = diag Q - colsumsq(Us)."""
    v = pool.shape[0]
    q = np.linalg.inv(kern.gram(pool, pool) + np.diag(_nu(noise, v)))
    a = list(indices)
    uq = np.linalg.cholesky(q[np.ix_(a, a)]).T
    us = solve_triangular(uq, q[a], trans="T", lower=False)
    return uq, us, np.diag(q) - np.sum(us * us, axis=0)


def var_scores(kern, pool, rest, weights=None):
    """Posterior variance (nugget 0) x weight of every pool point given the design rest, from scratch."""
    var = orc.fast_posterior_variance(kern, pool[rest], pool, 0.0) if rest else kern.prior(pool).copy()
    return var * weights if weights is not None else var


def fast_exchange_var(kern, pool, indices, rtol, max_sweeps, *, weights=None, n_fixed=0):
    """The maximum-variance exchange pass by brute force; positions < n_fixed are never removed."""
    return _exchange_max(lambda rest: var_scores(kern, pool, rest, weights), indices, rtol, max_sweeps, first=n_fixed)


def var_objective(kern, pool, indices, weights=None):
    a = list(indices)
    val = _logdet(kern.gram(pool[a], pool[a]))
    return val + (float(np.sum(np.log(weights[a]))) if weights is not None else 0.0)
