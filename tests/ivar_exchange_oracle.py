"""CPU oracles of the exchange refinement of a discrete IVAR design (refineGreedyIVARExperimentalDesign), built on
oracle/gpexp_oracle.py:

    fast_design_delete   the Givens downdate of the design factor and of the factor rows W (any float dtype)
    fast_exchange_ivar   the queue-ordered exchange pass, refactoring D minus the removed point from scratch at every step
                         and scoring with fast_ivar_scores
    ref_exchange_ivar    the same decisions from the reference's pinv cost loop (ref_ivar_cost), for tiny sizes

The exchange rule: each step removes the oldest design point (position 0), scores every candidate c as the design of the
other n - 1 points plus c, and appends the arg-min challenger (lowest index on ties) only if its cost is below
(1 - rtol) x the removed point's own cost; otherwise the removed point returns.  A sweep is n steps; the pass stops after a
sweep without a swap or after max_sweeps."""
import numpy as np
from scipy.linalg import solve_triangular

from oracle import gpexp_oracle as orc


def fast_design_delete(U, W, var, j):
    """Delete design position j from K_DD + diag(noise) = U^T U, W = U^-T K(D, X), var = k(x,x) - colsumsq(W).

    H = U without column j; Givens rotations on rows (i, i+1), i = j..n-2, zero H[i+1, i] with c = a/rho, s = b/rho,
    rho = hypot(a, b) (the identity when a = b = 0).  The same rotations on rows j..n-1 of W leave the reduced rows in
    j..n-2 and the residual row r in n-1.  Arithmetic in the dtype of the inputs.
    Returns (U' (n-1)x(n-1), W' (n-1)xX, r, var + r^2)."""
    U = np.array(U)
    W = np.array(W)
    n = U.shape[0]
    one, zero = U.dtype.type(1), U.dtype.type(0)
    H = np.delete(U, j, axis=1)
    for i in range(j, n - 1):
        a, b = H[i, i], H[i + 1, i]
        rho = np.hypot(a, b)
        c, s = (a / rho, b / rho) if rho > 0 else (one, zero)
        hi, hn = H[i].copy(), H[i + 1].copy()
        H[i], H[i + 1] = c * hi + s * hn, c * hn - s * hi
        H[i, i], H[i + 1, i] = rho, zero
        wi, wn = W[i].copy(), W[i + 1].copy()
        W[i], W[i + 1] = c * wi + s * wn, c * wn - s * wi
    r = W[n - 1].copy()
    return H[: n - 1], W[: n - 1], r, np.asarray(var) + r * r


def _state(kern, design, nug, x):
    """(W, var) of a given design: W = L^-1 K(D, x), var = k(x,x) - colsumsq(W) (no noise on x)."""
    if design.shape[0] == 0:
        return np.zeros((0, x.shape[0])), kern.prior(x).copy()
    low = np.linalg.cholesky(kern.gram(design, design) + np.diag(nug))
    w = solve_triangular(low, kern.gram(design, x), lower=True)
    return w, kern.prior(x) - np.sum(w * w, axis=0)


def _decide(cost, inc, rtol):
    """(winner, swapped, margin).  margin = relative distance of the deciding comparisons from their flip points: the best
    challenger (candidate other than the removed one) against the threshold (1 - rtol) cost[inc] and, when it swaps in,
    against the runner-up challenger."""
    c = int(np.argmin(cost))
    thr = (1.0 - rtol) * cost[inc]
    swapped = bool(cost[c] < thr)
    others = np.delete(cost, inc)
    if others.size == 0:
        return int(inc), False, np.inf
    best = np.partition(others, min(1, others.size - 1))
    margin = abs(best[0] - thr) / abs(thr)
    if swapped and others.size > 1:
        margin = min(margin, (best[1] - best[0]) / abs(best[0]))
    return (c if swapped else int(inc)), swapped, margin


def _exchange(score_all, indices, rtol, max_sweeps):
    design = [int(i) for i in indices]
    n = len(design)
    costs, swaps, margins = [], [], []
    for _ in range(max_sweeps):
        k = 0
        for _ in range(n):
            inc, rest = design[0], design[1:]
            cost = score_all(rest)
            win, swapped, margin = _decide(cost, inc, rtol)
            design = rest + [win]
            costs.append(float(cost[win]))
            margins.append(margin)
            k += swapped
        swaps.append(k)
        if k == 0:
            break
    return design, costs, swaps, margins


def fast_exchange_ivar(kern, cand, mc, indices, noise, rtol, max_sweeps, *, mc_weights=None):
    """The exchange pass by brute force: at every step D minus the removed point is refactored from scratch and every
    candidate scored with fast_ivar_scores.  ``noise`` is a scalar or a per-candidate vector nu.
    Returns (final indices in queue order, cost after every step, swaps per sweep, decision margin of every step)."""
    nu = np.broadcast_to(np.asarray(noise, dtype=np.float64), (cand.shape[0],))

    def score_all(rest):
        d = cand[rest]
        w_m, var_m = _state(kern, d, nu[rest], mc)
        w_c, var_c = _state(kern, d, nu[rest], cand)
        return orc.fast_ivar_scores(kern, cand, mc, w_m, var_m, w_c, var_c, nu, mc_weights=mc_weights)

    return _exchange(score_all, indices, rtol, max_sweeps)


def ref_exchange_ivar(kern, cand, mc, indices, noise, rtol, max_sweeps, *, mc_weights=None):
    """The same pass with every cost from the reference's own loop (ref_ivar_cost: pinv of the design Gram, Python loop over
    the integration points).  ``noise`` is a float or a per-candidate vector nu."""
    vec = np.ndim(noise) > 0

    def score_all(rest):
        cost = np.empty(cand.shape[0])
        for c in range(cand.shape[0]):
            pts = rest + [c]
            nug = np.asarray(noise, dtype=np.float64)[pts] if vec else float(noise)
            cost[c] = orc.ref_ivar_cost(kern, cand[pts], mc, nug, mc_weights)
        return cost

    return _exchange(score_all, indices, rtol, max_sweeps)


def design_cost(kern, cand, mc, indices, noise, *, mc_weights=None):
    """IVAR cost of the design cand[indices] (nugget noise[indices] for a per-candidate vector)."""
    nu = np.broadcast_to(np.asarray(noise, dtype=np.float64), (cand.shape[0],))
    _, var_m = _state(kern, cand[list(indices)], nu[list(indices)], mc)
    return abs(np.mean(var_m)) if mc_weights is None else abs(np.sum(mc_weights * var_m))
