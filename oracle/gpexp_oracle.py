"""CPU oracle for the GPEXP greedy experimental-design hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``gpexp_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` use it, and only as the checker or as
the timed CPU baseline.  The product path is CUDA-only.

Two layers live here, both plain numpy float64:

* ``ref_*``  -- a *faithful* restatement of the reference's algorithm: the same
  per-row / per-candidate loops and the same ``np.linalg.pinv`` (SVD,
  rcond=1e-15) solves, cited function by function against
  ``/root/reference/gpExp/*.py`` (file:line in each docstring).  These are
  what the reference would compute and (roughly) how long it would take.
* ``fast_*`` -- the vectorised Cholesky / Schur-complement restatement (same
  mathematics, O(n) less work per step) that the CUDA path mirrors.  It is
  proven equal to ``ref_*`` on small cases (tests/test_oracle.py) and is the
  checker at sizes ``ref_*`` cannot reach.

Pinning: the reference ships no tests or golden vectors
(``test/test_kernel.py:1-24`` is an empty licence header), so this oracle is
pinned against outputs of the *unmodified reference itself*, imported in the
build container by ``tests/golden/make_golden.py`` and frozen in
``tests/golden/*.npz`` (indices, per-step scores, variances, Gram matrices).

Each criterion also takes the variants the CUDA path supports, as optional
arguments whose defaults give the plain forms above:

* per-point noise -- ``ref_ivar_cost`` takes a nugget vector, ``ref_greedy_ivar``
  a ``noise_func`` giving the nugget of design+{c}, ``fast_ivar_scores`` /
  ``fast_greedy_ivar`` a per-candidate vector nu, and the three MI functions a
  per-point vector nu (K_AA + diag nu_A, K_SS + diag nu_S);
* weighted integration points -- ``mc_weights`` w makes the IVAR cost
  |sum_m w_m var(x_m)| instead of the Monte-Carlo mean.  Every weighted square
  is formed as (w v) v, the form the kernels use, so that w = 2^-k scales each
  term exactly: with M = 2^k and w = 1/M it reproduces the unweighted cost bit
  for bit;
* Matern nu = 1/2 and nu = 5/2 kernels -- ``KernelSpec.matern12`` /
  ``matern52``, k = s p(t) exp(-t) with t = sqrt(2 nu) |x - y| / rho, the
  scaling the reference uses for nu = 3/2 (kernels.py:87-89).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

SE = 0
MATERN32 = 1
MEHLER = 2
MATERN12 = 3
MATERN52 = 4

FAMILY_NAMES = {SE: "se", MATERN32: "matern32", MEHLER: "mehler", MATERN12: "matern12", MATERN52: "matern52"}
MATERN_NU = {MATERN12: 0.5, MATERN32: 1.5, MATERN52: 2.5}


def matern_closed_form(nu, r, rho, s):
    """s p(t) exp(-t), t = sqrt(2 nu) r / rho, for nu in {1/2, 3/2, 5/2}; r an array of distances.
        nu = 1/2   p = 1
        nu = 3/2   p = 1 + t
        nu = 5/2   p = 1 + t + t^2 / 3"""
    t = np.sqrt(2.0 * nu) * np.asarray(r, dtype=np.float64) / rho
    p = {0.5: 1.0, 1.5: 1.0 + t, 2.5: 1.0 + t + t * t / 3.0}[nu]
    return s * p * np.exp(-t)


# --------------------------------------------------------------------------
# Covariance functions (pairwise semantics)            kernels.py:49-65
# --------------------------------------------------------------------------
@dataclass
class KernelSpec:
    """Family + hyper-parameters of one covariance function.

    family SE        params: cl[d] (correlation lengths), signal   kernels.py:103-123
    family MATERN32  params: rho, signal                           kernels.py:74-91
    family MEHLER    params: t[d]                                  kernels.py:183-228, :250-293
    family MATERN12, MATERN52  params: rho, signal                 matern_closed_form
    """

    family: int
    dim: int
    cl: np.ndarray = field(default_factory=lambda: np.zeros(0))
    signal: float = 1.0
    rho: float = 1.0
    t: np.ndarray = field(default_factory=lambda: np.zeros(0))

    # ---- constructors mirroring the reference class constructors ----------
    @staticmethod
    def se(cl, signal, dim):
        cl = np.asarray(cl, dtype=np.float64).ravel()
        if cl.size == 1:  # kernels.py:106-107 isotropic -> tiled to d
            cl = np.tile(cl, dim)
        assert cl.size == dim
        return KernelSpec(SE, dim, cl=cl.copy(), signal=float(signal))

    @staticmethod
    def matern32(rho, signal, dim):
        return KernelSpec(MATERN32, dim, rho=float(rho), signal=float(signal))

    @staticmethod
    def matern12(rho, signal, dim):
        return KernelSpec(MATERN12, dim, rho=float(rho), signal=float(signal))

    @staticmethod
    def matern52(rho, signal, dim):
        return KernelSpec(MATERN52, dim, rho=float(rho), signal=float(signal))

    @staticmethod
    def mehler(t, dim):
        t = np.asarray(t, dtype=np.float64).ravel()
        assert t.size == dim
        return KernelSpec(MEHLER, dim, t=t.copy())

    # ---- evaluateF: equal-shaped inputs -> (p,) ---------------------------
    def evaluateF(self, x1, x2):
        assert x1.shape == x2.shape
        if self.family == SE:  # kernels.py:121-122
            return self.signal * np.exp(
                -0.5 * np.sum((x1 - x2) ** 2.0 * self.cl ** -2.0, axis=1))
        if self.family == MATERN32:  # kernels.py:87-89
            d = np.sqrt(np.sum((x1 - x2) ** 2.0, axis=1))
            term = np.sqrt(3) * d / self.rho
            return self.signal * (1.0 + term) * np.exp(-term)
        if self.family == MEHLER:  # kernels.py:223-227 product of 1-D, :282-285
            out = np.ones(x1.shape[0])
            for i in range(self.dim):
                t = self.t[i]
                a = x1[:, i]
                b = x2[:, i]
                out = out * ((1.0 - t ** 2.0) ** (-1.0 / 2.0) * np.exp(
                    -(a ** 2.0 * t ** 2.0 - 2.0 * t * a * b + b ** 2.0 * t ** 2.0)
                    / (2.0 * (1.0 - t ** 2.0))))
            return out
        if self.family in (MATERN12, MATERN52):
            d = np.sqrt(np.sum((x1 - x2) ** 2.0, axis=1))
            return matern_closed_form(MATERN_NU[self.family], d, self.rho, self.signal)
        raise ValueError("unknown kernel family")

    # ---- evaluate: pairwise with (1,d) broadcast        kernels.py:49-65 --
    def evaluate(self, x1, x2):
        assert x1.ndim > 1 and x2.ndim > 1
        assert x1.shape[1] == self.dim and x2.shape[1] == self.dim
        n1, n2 = x1.shape[0], x2.shape[0]
        if n1 > n2:
            return self.evaluateF(x1, np.tile(x2, (n1, 1)))
        if n1 < n2:
            return self.evaluateF(np.tile(x1, (n2, 1)), x2)
        return self.evaluateF(x1, x2)

    # ---- vectorised cross-Gram K[i,j] = k(X[i], Y[j]) ----------------------
    def gram(self, X, Y):
        """Same per-element formula as evaluateF, broadcast to (nx, ny)."""
        X = np.asarray(X, dtype=np.float64)
        Y = np.asarray(Y, dtype=np.float64)
        if self.family == SE:
            acc = np.zeros((X.shape[0], Y.shape[0]))
            for i in range(self.dim):
                diff = X[:, i:i + 1] - Y[None, :, i]
                acc += diff ** 2.0 * self.cl[i] ** -2.0
            return self.signal * np.exp(-0.5 * acc)
        if self.family == MATERN32:
            acc = np.zeros((X.shape[0], Y.shape[0]))
            for i in range(self.dim):
                diff = X[:, i:i + 1] - Y[None, :, i]
                acc += diff ** 2.0
            term = np.sqrt(3) * np.sqrt(acc) / self.rho
            return self.signal * (1.0 + term) * np.exp(-term)
        if self.family == MEHLER:
            out = np.ones((X.shape[0], Y.shape[0]))
            for i in range(self.dim):
                t = self.t[i]
                a = X[:, i:i + 1]
                b = Y[None, :, i]
                out = out * ((1.0 - t ** 2.0) ** (-1.0 / 2.0) * np.exp(
                    -(a ** 2.0 * t ** 2.0 - 2.0 * t * a * b + b ** 2.0 * t ** 2.0)
                    / (2.0 * (1.0 - t ** 2.0))))
            return out
        if self.family in (MATERN12, MATERN52):
            acc = np.zeros((X.shape[0], Y.shape[0]))
            for i in range(self.dim):
                diff = X[:, i:i + 1] - Y[None, :, i]
                acc += diff ** 2.0
            return matern_closed_form(MATERN_NU[self.family], np.sqrt(acc), self.rho, self.signal)
        raise ValueError("unknown kernel family")

    def prior(self, X):
        """k(x, x) per point (no noise)."""
        return self.evaluateF(X, X)

    def packed_params(self):
        """Flat parameter vector in the order the C ABI expects (include/gpexp_b200.h)."""
        if self.family == SE:
            return np.concatenate([self.cl, [self.signal]])
        if self.family in (MATERN32, MATERN12, MATERN52):
            return np.array([self.rho, self.signal])
        return self.t.copy()


# --------------------------------------------------------------------------
# Faithful restatement of the reference (loops + pinv)
# --------------------------------------------------------------------------
def ref_covariance_matrix(kern: KernelSpec, points, nugget=0.0):
    """gp_kernel_utilities.py:34-68 -- row loop of pairwise evaluates + diag(nugget)."""
    n, dim = points.shape
    cov = np.zeros((n, n))
    for j in range(n):
        cov[j, :] = kern.evaluate(points, points[j].reshape(1, dim))
    if isinstance(nugget, float):
        dadd = nugget * np.ones(n)
    elif isinstance(nugget, np.ndarray):
        dadd = nugget[:]
    else:  # the reference raises NameError here (gp_kernel_utilities.py:62-67)
        raise NameError("nugget must be float or ndarray")
    return cov + np.diag(dadd)


def ref_add_nodes(kern, nodes, noise):
    """gp.py:176-181 -- covariance + pinv precision."""
    cov = ref_covariance_matrix(kern, nodes, noise)
    return cov, np.linalg.pinv(cov)


def ref_evaluate_variance(kern, nodes, precision, newpt):
    """gp.py:246-256 -- M x n kernel values, python loop over query points, raw (signed) variance."""
    m, n = newpt.shape[0], nodes.shape[0]
    kv = np.zeros((m, n))
    for j in range(n):
        kv[:, j] = kern.evaluate(newpt, nodes[j].reshape(1, kern.dim))
    var_new = kern.evaluate(newpt, newpt)
    var = np.zeros(m)
    for j in range(m):
        var[j] = var_new[j] - np.dot(kv[j, :], np.dot(precision, kv[j, :].T))
    return var


def ref_ivar_cost(kern, design, mc, noise, mc_weights=None):
    """experimentalDesign.py:105-117 -- |mean posterior variance over the MC points|.

    ``noise`` is a float (homoscedastic gp.noise) or an ndarray of per-point
    nuggets (the space.noiseFunc branch, :110-114).  With ``mc_weights`` w the
    cost is |sum_m w_m var(x_m)|.
    """
    _, prec = ref_add_nodes(kern, design, noise)
    var_mc = ref_evaluate_variance(kern, design, prec, mc)
    if mc_weights is None:
        return abs(1.0 / float(mc.shape[0]) * np.sum(var_mc))
    return abs(np.sum(mc_weights * var_mc))


def ref_greedy_var(kern, pool, n_points, weights=None, ind_keep_start=()):
    """experimentalDesign.py:787-845 -- greedy max posterior variance, nugget 0, pinv each step.

    Returns (indices, list of per-step score vectors).  The reference returns
    pool[indices]; indices are what the parity tests compare.
    """
    ind = list(ind_keep_start)
    have = len(ind)
    dim = pool.shape[1]
    c = pool.shape[0]
    scores = []
    while have < n_points:
        if have == 0:
            k = kern.evaluate(pool, pool)  # :816
        else:
            cov = ref_covariance_matrix(kern, pool[ind, :])  # :825 nugget 0.0
            inv = np.linalg.pinv(cov)  # :826
            kv = np.zeros((have, c))
            for i in range(have):  # :829-831
                kv[i, :] = kern.evaluate(pool, pool[ind[i]].reshape(1, dim))
            k = np.zeros(c)
            for i in range(c):  # :834-837
                pt = pool[i].reshape(1, dim)
                k[i] = (kern.evaluate(pt, pt) - np.dot(kv[:, i].T, np.dot(inv, kv[:, i])))[0]
        if weights is not None:
            k = k * weights
        scores.append(k.copy())
        ind.append(int(np.argmax(k)))  # :821 / :841 first maximum
        have += 1
    return ind, scores


def ref_greedy_ivar(kern, cand, mc, n_points, noise, cand_subset=None, *, mc_weights=None, noise_func=None):
    """Discrete greedy IVAR as SURVEY.md section 8(c) defines it (the reference has the
    cost function, experimentalDesign.py:79-117, but no discrete driver): at each step
    evaluate the reference IVAR cost of design+{c} for every candidate c and take
    np.argmin.  With ``noise_func`` the nugget of design+{c} is noise_func(design+{c})
    (the reference's heteroscedastic branch, :110-114) and ``noise`` is not used.
    Returns (indices, per-step cost vectors)."""
    ind = []
    costs = []
    cs = range(cand.shape[0]) if cand_subset is None else cand_subset
    for _ in range(n_points):
        cost = np.full(cand.shape[0], np.inf)
        for c in cs:
            pts = np.vstack([cand[ind, :], cand[c:c + 1, :]])
            nugget = noise if noise_func is None else noise_func(pts)
            cost[c] = ref_ivar_cost(kern, pts, mc, nugget, mc_weights)
        costs.append(cost)
        ind.append(int(np.argmin(cost)))
    return ind, costs


def ref_mi_cost(kern, pool, noise, index, index_added):
    """experimentalDesign.py:252-285 -- var(y|A) / var(y|V minus A minus y), two pinv's.

    ``noise`` is a float or a per-point vector nu, which each subset's Gram takes on
    that subset: K_AA + diag nu_A and K_SS + diag nu_S, S = V minus A minus y."""
    vec = np.ndim(noise) > 0
    dim = pool.shape[1]
    point = pool[index, :].reshape(1, dim)
    var = kern.evaluate(point, point)
    added = pool[index_added, :].reshape(len(index_added), dim)
    kva = kern.evaluate(added, point)
    cov_num = ref_covariance_matrix(kern, added, noise[index_added] if vec else noise)
    numerator = var - np.dot(kva.T, np.dot(np.linalg.pinv(cov_num), kva))
    left = np.setdiff1d(np.arange(pool.shape[0]), index_added)
    left = np.setdiff1d(left, [index])
    pts_left = pool[left, :]
    kvl = kern.evaluate(pts_left, point)
    cov_den = ref_covariance_matrix(kern, pts_left, noise[left] if vec else noise)
    denominator = var - np.dot(kvl.T, np.dot(np.linalg.pinv(cov_den), kvl))
    return numerator / denominator


def ref_greedy_mi(kern, pool, noise, n_points, start=0):
    """experimentalDesign.py:753-785; ``noise`` as in ref_mi_cost.  Returns (indices, per-step
    score vectors over the remaining options, per-step option index arrays)."""
    ind = [start]
    options = np.setdiff1d(np.arange(pool.shape[0]), ind)
    scores, opts = [], []
    for _ in range(len(ind), n_points):
        out = np.zeros(len(options))
        for j, i in enumerate(options):
            out[j] = ref_mi_cost(kern, pool, noise, int(i), ind)[0]
        scores.append(out)
        opts.append(options.copy())
        new = int(options[np.argmax(out)])
        ind.append(new)
        options = np.setdiff1d(options, new)
    return ind, scores, opts


# --------------------------------------------------------------------------
# Vectorised Cholesky / Schur restatement (what the CUDA path mirrors)
# --------------------------------------------------------------------------
def fast_posterior_variance(kern, design, x, noise=0.0):
    """var[j] = k(x_j,x_j) - |L^-1 k(D,x_j)|^2 with K_DD + diag(noise) = L L^T.
    Equals ref_evaluate_variance up to cond(K)*eps (gp.py:251-255)."""
    from scipy.linalg import solve_triangular
    n = design.shape[0]
    nug = noise * np.ones(n) if np.isscalar(noise) else np.asarray(noise)
    kdd = kern.gram(design, design) + np.diag(nug)
    low = np.linalg.cholesky(kdd)
    w = solve_triangular(low, kern.gram(design, x), lower=True)
    return kern.prior(x) - np.sum(w * w, axis=0)


def fast_greedy_var(kern, pool, n_points, weights=None, ind_keep_start=()):
    """Greedy max-variance == diagonally pivoted Cholesky of K_CC (SURVEY.md 3.1).

    W[n,:] = (k(x_p,.) - W[:n,p]^T W[:n,:]) / sqrt(var[p]) ; var -= W[n,:]^2.
    Seeds in ind_keep_start are forced pivots.  Returns (indices, per-step scores).
    """
    c = pool.shape[0]
    var = kern.prior(pool).copy()
    w = np.zeros((n_points, c))
    ind, scores = [], []

    def append(p):
        n = len(ind)
        row = kern.gram(pool[p:p + 1], pool)[0] - w[:n, p] @ w[:n, :]
        row /= math.sqrt(var[p])
        w[n, :] = row
        var[:] = var - row * row
        ind.append(int(p))

    for p in ind_keep_start:
        append(p)
    while len(ind) < n_points:
        k = var * weights if weights is not None else var
        scores.append(k.copy())
        append(int(np.argmax(k)))
    return ind, scores


def fast_ivar_scores(kern, cand, mc, w_m, var_m, w_c, var_c, noise, block=4096, *, mc_weights=None):
    """IVAR cost of design+{c} for every candidate c via the Schur identity (SURVEY.md 3.2):

        cost[c] = | mean_m var_D(m) - (1/M) sum_m cov_D(m,c)^2 / (var_D(c) + noise) |
        cov_D(m,c) = k(m,c) - W_M[:,m] . W_C[:,c]

    ``noise`` is a scalar or a per-candidate vector nu.  With ``mc_weights`` w the mean and
    (1/M) sum_m cov^2 become sum_m w_m var_D(m) and sum_m (w_m cov) cov.
    The reduction is 0 where var_D(c)+noise is numerically zero (SURVEY.md section 7,
    duplicate-candidate rule: pinv drops the null direction)."""
    m = mc.shape[0]
    c = cand.shape[0]
    base = np.sum(var_m) / m if mc_weights is None else np.sum(mc_weights * var_m)
    r = np.zeros(c)
    for c0 in range(0, c, block):
        cov = kern.gram(mc, cand[c0:c0 + block]) - w_m.T @ w_c[:, c0:c0 + block]
        wcov = cov if mc_weights is None else mc_weights[:, None] * cov
        r[c0:c0 + block] = np.sum(wcov * cov, axis=0)
    den = var_c + noise
    tiny = den <= ZERO_VAR_TOL * kern_scale(kern, cand)
    red = r / np.where(tiny, 1.0, den)
    if mc_weights is None:
        red = red / m
    red = np.where(tiny, 0.0, red)
    return np.abs(base - red)


ZERO_VAR_TOL = 1e-13


def kern_scale(kern, pts=None):
    """k(0,0): magnitude of the prior variance, used only to decide 'numerically zero'."""
    if kern.family == MEHLER:
        return float(np.prod((1.0 - kern.t ** 2.0) ** -0.5))
    return abs(kern.signal)


def fast_greedy_ivar(kern, cand, mc, n_points, noise, *, mc_weights=None):
    """Incremental greedy IVAR (SURVEY.md 3.2): append one row to W_M and W_C per step with
    divisor sqrt(var_D(p)+nu[p]), running var updates.  ``noise`` is a scalar or a
    per-candidate vector nu; integration points carry no noise.  ``mc_weights`` as in
    fast_ivar_scores.  Returns (indices, per-step costs)."""
    c, m = cand.shape[0], mc.shape[0]
    nu = np.broadcast_to(noise, (c,))
    w_c = np.zeros((n_points, c))
    w_m = np.zeros((n_points, m))
    var_c = kern.prior(cand).copy()
    var_m = kern.prior(mc).copy()
    ind, costs = [], []
    for n in range(n_points):
        cost = fast_ivar_scores(kern, cand, mc, w_m[:n], var_m, w_c[:n], var_c, nu, mc_weights=mc_weights)
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


def fast_greedy_mi(kern, pool, noise, n_points, start=0, *, with_pivots=False):
    """Greedy MI with the exact restatement of SURVEY.md 3.3:

        numerator(y)   = var(y | A)                 (incremental pivoted-Cholesky rows, nugget=noise)
        denominator(y) = 1 / [(K_SS + noise I)^-1]_yy - noise,   S = V minus A  (y in S)

    and a rank-1 downdate of the precision when a point leaves S.  ``noise`` is a scalar or
    a per-point vector nu: the precision is (K_VV + diag nu)^-1, the appended rows are divided
    by sqrt(num[p] + nu[p]) and the denominator is 1/pd[y] - nu[y].  Returns (indices, per-step
    score vectors of length |V| with selected entries = -inf), and with ``with_pivots`` the
    per-step pivots num[p] + nu[p] as a third value."""
    v = pool.shape[0]
    nu = np.broadcast_to(noise, (v,))
    kvv = kern.gram(pool, pool) + np.diag(nu)
    prec = np.linalg.inv(kvv)
    prior = kern.prior(pool)
    num = prior.copy()
    w = np.zeros((n_points, v))
    selected = np.zeros(v, dtype=bool)
    ind, scores, pivots = [], [], []
    pd = np.diag(prec).copy()
    us = []

    def current_col(p):
        col = prec[:, p].copy()
        for u in us:
            col -= u * u[p]
        return col

    def take(p):
        nonlocal pd
        n = len(ind)
        pivots.append(num[p] + nu[p])
        lnn = math.sqrt(pivots[-1])
        row = (kern.gram(pool[p:p + 1], pool)[0] - w[:n, p] @ w[:n, :]) / lnn
        w[n, :] = row
        num[:] = num - row * row
        col = current_col(p)
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
    return (ind, scores, pivots) if with_pivots else (ind, scores)


# --------------------------------------------------------------------------
# Convenience: build W / var state for a *given* design (used by tests + bench baseline)
# --------------------------------------------------------------------------
def fast_design_state(kern, design, x, noise):
    from scipy.linalg import solve_triangular
    n = design.shape[0]
    if n == 0:
        return np.zeros((0, x.shape[0])), kern.prior(x).copy()
    low = np.linalg.cholesky(kern.gram(design, design) + noise * np.eye(n))
    w = solve_triangular(low, kern.gram(design, x), lower=True)
    return w, kern.prior(x) - np.sum(w * w, axis=0)


# --------------------------------------------------------------------------
# SURVEY.md 8(f) widening: marginal log-likelihood and the IVAR gradient (squared-exponential kernels)
# --------------------------------------------------------------------------
def ref_loglike(kern, pts, evals, noise):
    """gp.py:394-446 -- pinv + slogdet marginal log-likelihood."""
    cov = ref_covariance_matrix(kern, pts, noise)
    inv = np.linalg.pinv(cov)
    _, logdet = np.linalg.slogdet(cov)
    return -0.5 * np.dot(evals, np.dot(inv, evals)) - 0.5 * logdet - len(evals) / 2.0 * np.log(2.0 * np.pi)


def fast_loglike(kern, pts, evals, noise):
    """Cholesky restatement: -1/2 |L^-1 y|^2 - sum log L_ii - n/2 log 2 pi."""
    from scipy.linalg import solve_triangular
    low = np.linalg.cholesky(kern.gram(pts, pts) + noise * np.eye(len(pts)))
    z = solve_triangular(low, evals, lower=True)
    return -0.5 * float(z @ z) - float(np.sum(np.log(np.diag(low)))) - len(evals) / 2.0 * np.log(2.0 * np.pi)


def se_derivative(kern, x1, x2):
    """kernels.py:146-181 -- out[j,i] = 'dK(x1[j], x2)/dx1[j,i]' AS THE REFERENCE COMPUTES IT:
    -signalSize * (x1 - x2)/cl^2 * evaluate(x1, x2).  evaluate already carries signalSize, so the result is
    signalSize times the true derivative; parity means reproducing that."""
    assert kern.family == SE and x2.shape[0] == 1
    r = kern.evaluate(x1, x2)
    return -kern.signal * (x1 - x2) / kern.cl ** 2.0 * r[:, None]


def fast_variance_derivative(kern, design, newpt, noise):
    """gp.py:282-341 (noiseFunc None) restated without the n*d python loop:
        a = K(newpt, D) P ;  T_j[m,k] = -derivative(newpt, p_j)[m,k] ;  dc_(j,k)[c] = derivative(D, p_j)... see below
        out[j*d+k, m] = -2 a[m,j] T_j[m,k] + 2 a[m,j] sum_c dc_(j,k)[c] a[m,c]
    Returns the (n*d, M) matrix; the IVAR gradient (experimentalDesign.py:166-169) is its row mean."""
    n, d = design.shape
    m = newpt.shape[0]
    kdd = kern.gram(design, design) + noise * np.eye(n)
    a = np.linalg.solve(kdd, kern.gram(design, newpt)).T  # (M, n) = totEvals . precision
    out = np.zeros((n * d, m))
    for j in range(n):
        p = design[j:j + 1]
        t_j = -se_derivative(kern, newpt, p)              # derivTotal[j]            gp.py:316
        # derivCovTotal[:, j, k] (gp.py:314,329-330): d K(p_j, p_c) / d p_j,k for every c, as the reference's
        # derivative() computes it = -(derivative of K(p_c, p_j) with respect to p_c)
        dc = -se_derivative(kern, design, p)
        for k in range(d):
            q = a @ dc[:, k]                              # sum_c dc[c] a[m,c]
            out[j * d + k] = -2.0 * a[:, j] * t_j[:, k] + 2.0 * a[:, j] * q
    return out


# --------------------------------------------------------------------------
# SURVEY.md 8(f) rows 2-4 (round 2): heteroscedastic variance derivative, log-likelihood gradient, FITC, Gram x vector
# --------------------------------------------------------------------------
def ref_variance_derivative_hetero(kern, design, newpt, nugget_vec, noise_deriv):
    """gp.py:282-341 with a noise function: the loops of the reference, line for line, for SE kernels.
    nugget_vec = noiseFunc(design) (the per-point nugget the Gram was built with), noise_deriv = noiseFunc.deriv(design).
    The `np.linalg.norm(p - newpt) < 1e-10` adjustment (:317-319) is the norm of the whole difference matrix and is kept."""
    n, d = design.shape
    m = newpt.shape[0]
    prec = np.linalg.pinv(kern.gram(design, design) + np.diag(nugget_vec))
    deriv_cov = np.zeros((n, n, d))
    tot = np.zeros((m, n))
    deriv_total = []
    for zz in range(n):
        p = design[zz:zz + 1]
        ind = np.array([np.linalg.norm(pp - p) < 1e-10 for pp in design])
        deriv_cov[zz] = se_derivative(kern, design, p)
        tot[:, zz] = kern.evaluate(np.tile(p, (m, 1)), newpt)
        deriv_total.append(-se_derivative(kern, newpt, p))
        deriv_cov[zz] += np.tile(ind.reshape(n, 1), d) * noise_deriv
        if np.linalg.norm(p - newpt) < 1e-10:
            raise NotImplementedError("degenerate query: every evaluation point on a design point")
    a = tot @ prec
    out1 = np.zeros((n * d, m))
    out2 = np.zeros((n * d, m))
    for jj in range(n):
        for kk in range(d):
            out1[jj * d + kk] = 2.0 * a[:, jj] * deriv_total[jj][:, kk]
            ds = np.zeros((n, n))
            ds[jj, :] = deriv_cov[:, jj, kk]
            ds[:, jj] = deriv_cov[:, jj, kk]
            out2[jj * d + kk] = -np.sum((a @ ds) * a, axis=1)
    return -(out1 + out2)


def fast_loglike_gradient(kern, pts, evals, noise):
    """gp.py:447-468 with kernels.py:125-144: d loglike / d theta = 1/2 tr((alpha alpha^T - K^-1) dK/dtheta) for
    theta = cl_0..cl_{d-1}, signalSize, and 'noise' (the trace times 2*noise, gp.py:463-464).  Returns a dict keyed like the
    reference's.  PARITY UNPINNED: the reference indexes `x1[:, direction]` with a float (kernels.py:140-142) and raises
    IndexError under numpy >= 1.12, so no golden vector can be produced; this is the expression the reference states, and
    the tests additionally check it against central finite differences of the (golden-pinned) log-likelihood value."""
    assert kern.family == SE
    n, d = pts.shape
    kmat = kern.gram(pts, pts)
    cov = kmat + noise * np.eye(n)
    prec = np.linalg.inv(cov)
    alpha = prec @ evals
    term = np.outer(alpha, alpha) - prec
    out = {}
    for q in range(d):
        diff2 = (pts[:, None, q] - pts[None, :, q]) ** 2.0
        out["cl%d" % q] = 0.5 * float(np.sum(term * kmat * diff2 / kern.cl[q] ** 3.0))
    out["signalSize"] = 0.5 * float(np.sum(term * kmat / kern.signal))
    out["noise"] = 0.5 * float(np.trace(term)) * noise * 2.0
    return out


def ref_fitc(kern, nodes, inducing, noise):
    """gp.py:193-208 / gp_kernel_utilities.py:81-97: FITC covariance Q + G and its Woodbury precision, with the reference's
    pinv / inv calls.  Returns (covariance, precision)."""
    quu = ref_covariance_matrix(kern, inducing, noise)
    inv_quu = np.linalg.pinv(quu)
    kuf = np.array([kern.evaluate(np.tile(s[None, :], (len(nodes), 1)), nodes) for s in inducing])
    q = kuf.T @ inv_quu @ kuf
    kff = ref_covariance_matrix(kern, nodes, noise)
    g = np.diag(kff - q)
    inv_g = np.diag(1.0 / (g + 1e-12))
    prec = inv_g - inv_g @ kuf.T @ np.linalg.inv(quu + kuf @ inv_g @ kuf.T) @ kuf @ inv_g
    return q + np.diag(g), prec


def ref_cov_times_v(kern, pts, b):
    """gp_kernel_utilities.py:107-142: out[i] = kernel.evaluate(pts, pts[i]) . b, one row per iteration."""
    return np.array([np.dot(kern.evaluate(pts, np.tile(pts[i:i + 1], (len(pts), 1))), b) for i in range(len(pts))])
