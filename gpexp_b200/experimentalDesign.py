"""Cost functions and discrete greedy design drivers behind the reference's names (gpExp/experimentalDesign.py), running on
the device-resident engines of gpexp_b200.engine.

    costFunctionGP_IVAR.evaluate / derivative   experimentalDesign.py:79-117, :148-179   (version 1, MC-integrated variance)
    costFunctionGP_MI.evaluate                  experimentalDesign.py:252-285
    performGreedyVarExperimentalDesign          experimentalDesign.py:787-845
    performGreedyMIExperimentalDesign           experimentalDesign.py:753-785
    performGreedyIVARExperimentalDesign,        NEW: the discrete greedy-IVAR driver the north star asks for; the
    beginGreedyIVARExperimentalDesign,          reference only has the per-design cost function (SURVEY.md 3.2 / 8c)
    refineGreedyIVARExperimentalDesign,         NEW: exchange passes that improve a discrete IVAR design on the candidates
    refineGreedyMIExperimentalDesign,           NEW: the same for greedy MI designs on the pool
    refineGreedyVarExperimentalDesign           NEW: the same for greedy maximum-variance designs
    scoreCandidatesIVAR

The continuous optimisers that CALL these cost functions (ExperimentalDesignDerivative / NoDerivative and the batch-greedy
wrappers, experimentalDesign.py:296-751) are deliberately not re-typed here: with the reference importable,
`gpexp_b200.install_as_gpExp()` rebinds the functions of `DEVICE_METHODS` / `DEVICE_FUNCTIONS` onto the reference's own
module, and its optimiser loops then drive the device path unchanged.
"""
import copy
import hashlib
import itertools
import math

import numpy as np

from . import _lib
from ._lib import check, lib
from .approximation import UniformMeasure
from .device import ptr
from .engine import (DesignFactor, GreedyIVAREngine, GreedyVarEngine, MeasureIVAREngine, Shard, ShardedMIEngine,
                     prior_scale)
from .gp_kernel_utilities import _nugget_arg

VERBOSE = True  # the reference prints its progress unconditionally (experimentalDesign.py:812-813)


# ---- costFunctionGP_IVAR --------------------------------------------------------------------------------------------------
def _ivar_mc_points(self, dev):
    """The Monte-Carlo integration points as a device point set, uploaded once per cost function."""
    cached = self.__dict__.get("_mc_dev")
    if cached is None or cached.dev is not dev or cached.n != len(self.mcPoints):
        cached = self.__dict__["_mc_dev"] = dev.points(self.mcPoints)
    return cached


def _ivar_weights(self):
    """The cost function's integration weights `mcWeights` (None: the plain Monte-Carlo mean), checked on the host against
    its integration points: one finite value >= 0 per point and at least one > 0, else ValueError."""
    w = getattr(self, "mcWeights", None)
    if w is None:
        return None
    return _checked_per_point(w, len(self.mcPoints), "mcWeights has", need_positive=True)


def _ivar_measure(self, what=None):
    """The cost function's `measure` as (kind, lower-or-mean, upper-or-std) for its kernel's dimension, or None.
    ValueError with mcWeights set as well, and for a Gaussian measure too wide for a Mehler kernel (int k(x, x) dmu is
    infinite unless std_q^2 < (1 + t_q) / (2 t_q)); NotImplementedError for a kernel other than squared-exponential or
    Mehler and for `what` (the name of a feature the closed form does not support), each naming the measure."""
    m = getattr(self, "measure", None)
    if m is None:
        return None
    if getattr(self, "mcWeights", None) is not None:
        raise ValueError(f"{m!r} integrates exactly and mcWeights weights integration points: set one of the two")
    if what is not None:
        raise NotImplementedError(f"{m!r}: {what} is not implemented for the closed-form measure integral")
    fam, d, params = self.gaussianProcess.kernel._gpx_spec()
    if fam not in (_lib.SE, _lib.MEHLER):
        raise NotImplementedError(f"{m!r}: the closed-form measure integral is implemented for squared-exponential "
                                  f"and Mehler kernels only")
    p0, p1 = m.params(d)
    gauss = not isinstance(m, UniformMeasure)
    if gauss and fam == _lib.MEHLER:
        t = np.asarray(params, dtype=np.float64)
        for q in range(d):
            if t[q] > 0.0 and not p1[q] * p1[q] < (1.0 + t[q]) / (2.0 * t[q]):
                raise ValueError(f"{m!r} is too wide for the Mehler kernel in dimension {q} (t = {t[q]!r}): "
                                 f"int k(x, x) dmu is infinite there unless std < {math.sqrt((1.0 + t[q]) / (2.0 * t[q]))!r}")
    return (_lib.MEASURE_GAUSS if gauss else _lib.MEASURE_BOX), p0, p1


def _ivar_evaluate(self, inputPoints):
    """|mean posterior variance over the MC points| for the design `inputPoints` (:79-117); with weights w
    (`mcWeights`), |sum_m w_m var(x_m)|; with a `measure`, the exact |int var(x) dmu(x)|."""
    assert inputPoints.shape == (self.numInputs, self.space.dimension), \
        ("inputPoints are the wrong size: ", inputPoints.shape)
    if self.version != 1:
        raise NotImplementedError("IVAR version 0 needs a kernel eigen-basis that no shipped kernel provides "
                                  "(experimentalDesign.py:119-146 is unreachable)")
    meas = _ivar_measure(self)
    w = None if meas is not None else _ivar_weights(self)
    gp = self.gaussianProcess
    if self.space.noiseFunc is None:
        gp.addNodesAndComputeCovariance(inputPoints)
    else:
        gp.addNodesAndComputeCovariance(inputPoints, self.space.noiseFunc(inputPoints))
    f = gp._factor
    if meas is not None:
        if not isinstance(f, DesignFactor):
            raise NotImplementedError(f"{self.measure!r}: the closed-form measure integral needs a full GP, not FITC")
        # the design's own points serve as the engine's candidates: only its cost s - tr Psi is read
        eng = MeasureIVAREngine(f.dev, f.design, f.n, 0.0, gp.kernel._gpx_spec(), meas)
        eng.load_design(f)
        eng.score()
        return np.abs(float(eng.cost.item()))
    mc = _ivar_mc_points(self, f.dev)
    _, var = f.solve_gram(mc)
    total = f.dev.zeros(1)
    if w is not None:
        wd = f.dev.upload(w)
        check(lib.gpx_sum_w(f.dev.h, ptr(var), ptr(wd), mc.n, ptr(total), f.dev.stream), "gpx_sum_w")
        return np.abs(float(total.item()))
    check(lib.gpx_sum(f.dev.h, ptr(var), mc.n, ptr(total), f.dev.stream), "gpx_sum")
    return np.abs(float(total.item()) / float(self.nMC))


def _ivar_derivative(self, inputPoints):
    """Gradient of the IVAR cost with respect to the design coordinates, shape (nPoints*dimension,)
    (:148-179, version 1): the row mean over the MC points of GP.evaluateVarianceDerivative, with the noise function's
    own derivative in the heteroscedastic case.  Squared-exponential kernels.  With weights w (`mcWeights`) the row
    reduction is sum_m w_m instead of the mean."""
    gp = self.gaussianProcess
    _ivar_measure(self, "the derivative")
    gp.kernel._require_derivative()
    w = _ivar_weights(self)
    noise_grad = same = None
    if self.space.noiseFunc is None:
        gp.addNodesAndComputeCovariance(inputPoints)
    else:
        nf = self.space.noiseFunc
        gp.addNodesAndComputeCovariance(inputPoints, noiseIn=nf(inputPoints))
        noise_grad = np.asarray(nf.deriv(inputPoints), dtype=np.float64)
        same = np.linalg.norm(inputPoints[:, None, :] - inputPoints[None, :, :], axis=2) < 1e-10
    f = gp._factor
    mc = _ivar_mc_points(self, f.dev)
    full = f.variance_gradient(mc, noise_grad, same)
    rows = f.n * gp.kernel.dimension
    out = f.dev.zeros(max(rows, 1))
    if w is not None:
        wd = f.dev.upload(w)
        check(lib.gpx_rowsum_w(f.dev.h, ptr(full), rows, mc.n, mc.ld, ptr(wd), ptr(out), f.dev.stream), "gpx_rowsum_w")
    else:
        check(lib.gpx_rowsum(f.dev.h, ptr(full), rows, mc.n, mc.ld, 1.0 / float(self.nMC), ptr(out), f.dev.stream),
              "gpx_rowsum")
    return out[:rows].cpu().numpy()


# ---- costFunctionGP_MI ----------------------------------------------------------------------------------------------------
def _mi_noise(self):
    """(scalar noise, per-point noise vector or None) of the cost function's GP: an ndarray gp.noise is the noise at
    each pool point, checked to hold one finite value >= 0 per point."""
    noise = _nugget_arg(self.gaussianProcess.noise)
    if isinstance(noise, np.ndarray):
        return 0.0, _checked_per_point(noise, len(self.mcPoints), "gp.noise has")
    return float(noise), None


def _mi_new_engine(self, n_max, shard=None, keep_factors=False):
    gp = self.gaussianProcess
    noise, nu = _mi_noise(self)
    # left-looking blocked set-up (measured faster than a right-looking dense engine on one GPU as well:
    # |V| = 40 000: 2.33 s vs 2.97 s)
    return ShardedMIEngine(gp.kernel._bind(), self.mcPoints, n_max, noise, shard=shard, pool_noise=nu,
                           keep_factors=keep_factors)


def _mi_evaluate(self, index, indexAdded):
    """MI ratio of candidate `index` given the already chosen `indexAdded` (:252-285); shape (1,).

    The reference pays two pseudo-inverses per call; here the O(|V|^3) factorisation of the pool is built once and kept
    (until the pool, the kernel or the noise changes), the chosen points are replayed only when `indexAdded` stops
    extending the previous call's list, and the scores of ALL candidates for that list are kept, so the reference's loop
    `for ind in options: evaluate(ind, indKeep)` (:776-777) costs one scoring pass per greedy step."""
    added = [int(i) for i in indexAdded]
    gp = self.gaussianProcess
    fam, _, params = gp.kernel._gpx_spec()
    noise, nu = _mi_noise(self)
    noise_key = noise if nu is None else hashlib.sha256(nu.tobytes()).hexdigest()
    key = (fam, tuple(np.ravel(params)), noise_key, id(self.mcPoints), len(self.mcPoints))
    st = self.__dict__.setdefault("_mi_cache", {})
    eng = st.get("engine")
    if eng is None or st.get("key") != key:
        eng = _mi_new_engine(self, max(64, 2 * (len(added) + 1)))
        st.update(engine=eng, key=key, prefix=[], scores=None)
    else:
        gp.kernel._bind(eng.dev)
    if added[: len(st["prefix"])] != st["prefix"] or len(added) > eng.ncap:
        eng.reset(max(64, 2 * (len(added) + 1)))
        st.update(prefix=[], scores=None)
    if len(added) > len(st["prefix"]) or st["scores"] is None:
        for i in added[len(st["prefix"]):]:
            eng.force(i)
        eng.score()
        st.update(prefix=added, scores=eng.global_scores())
    return st["scores"][int(index): int(index) + 1].copy()


class costFunctionBase(object):

    def __init__(self, nInputs, space):
        self.numInputs, self.space = nInputs, space


class costFunctionGP_IVAR(costFunctionBase):
    """Integrated posterior variance of a design, Monte-Carlo version: costFunctionGP_IVAR(gp, nInputs, space,
    version=1, mcPoints=..., mcWeights=...)  (:60-75).  Holds a shallow copy of the GP; without mcPoints, 10 000 samples
    of the space.

    mcWeights (attribute, default None): one float64 weight per integration point (finite, >= 0, at least one > 0),
    used as given, not normalised.  The cost is then |sum_m w_m var(x_m)| instead of the mean over mcPoints: Gauss-Legendre
    or other quadrature weights, importance weights p(x_m)/q(x_m) of a density that can be evaluated but not sampled, or a
    region of interest (weighted IMSE).  w = 1/nMC is the plain cost.  evaluate, derivative and the greedy drivers
    (beginGreedyIVARExperimentalDesign, performGreedyIVARExperimentalDesign, scoreCandidatesIVAR) read it; bad weights
    raise ValueError before any device work.  Under install_as_gpExp(path) the reference's own constructor is kept, so
    there the caller sets `cf.mcWeights = w` after construction.

    measure (attribute or keyword, default None): a gpexp_b200.approximation.UniformMeasure or GaussianMeasure.  The cost
    is then the exact |int var(x) dmu(x)| for a squared-exponential or Mehler kernel, with no integration points and no
    sampling error; evaluate, the greedy drivers and scoreCandidatesIVAR use it (a heteroscedastic space.noiseFunc
    applies as in the Monte-Carlo path).  With a measure, mcPoints is not sampled when not given.  A Mehler kernel's
    prior variance grows like exp(x^2 t / (1 + t)), so its Monte-Carlo estimate under N(0, 1) has infinite variance for
    t >= 1/3; the closed form has none.  ValueError together with mcWeights, and for a GaussianMeasure with
    std_q^2 >= (1 + t_q) / (2 t_q) under a Mehler kernel (the integral is infinite); NotImplementedError for Matern
    kernels, derivative, refineGreedyIVARExperimentalDesign, shard= and resident=True."""

    mcWeights = None
    measure = None

    def __init__(self, gaussianProcess, nInputs, space, version=1, **kwargs):
        costFunctionBase.__init__(self, nInputs, space)
        self.gaussianProcess, self.version = copy.copy(gaussianProcess), version
        if version == 1:
            self.measure = kwargs.get('measure')
            if 'mcPoints' in kwargs:
                pts = kwargs['mcPoints']
            else:
                pts = space.sample((10000, space.dimension)) if self.measure is None else None
            self.mcPoints, self.nMC = pts, 0 if pts is None else len(pts)
            self.mcWeights = kwargs.get('mcWeights')

    evaluate = _ivar_evaluate
    derivative = _ivar_derivative


class costFunctionGP_MI(costFunctionBase):
    """Krause-Guestrin mutual-information ratio var(y|A) / var(y|V minus A minus y) over a candidate pool (:223-285).
    The GP passed in is used directly, not copied (:227); pool = mcpoints[nmc], a 10 x 10 grid (square=True, 2-D) or 200
    samples of the space.

    gp.noise is a scalar nugget or an ndarray nu with one finite value >= 0 per pool point (aligned with mcPoints): each
    subset's Gram then takes diag(nu) on that subset, K_AA + diag nu_A and K_S'S' + diag nu_S'.  space.noiseFunc is not
    used, as in the reference; a caller with a noise function passes gp.noise = noiseFunc(pool)."""

    def __init__(self, gaussianProcess, nInputs, space, nmc=None, mcpoints=None, square=False):
        costFunctionBase.__init__(self, nInputs, space)
        self.gaussianProcess = gaussianProcess
        if nmc is not None:
            pool = np.copy(mcpoints)
        elif space.dimension == 2 and square is True:
            axis = np.linspace(-1, 1, 10)
            pool = np.array(list(itertools.product(axis, axis)))
            nmc = len(pool)
        else:
            nmc = 200
            pool = space.sample((nmc, space.dimension))
        self.add_candidates(nmc, pool, _copy=False)

    def add_candidates(self, nCandidates, candidates, _copy=True):
        self.nMC = nCandidates
        self.mcPoints = copy.deepcopy(candidates) if _copy else candidates
        self.gaussianProcess.addNodesAndComputeCovariance(self.mcPoints)

    # the reference stores both at construction and never reads them again (:241-242); here they are produced on demand
    @property
    def cov(self):
        return self.gaussianProcess.covarianceMatrix

    @property
    def invcov(self):
        return self.gaussianProcess.precisionMatrix

    evaluate = _mi_evaluate


# ---- discrete greedy drivers ----------------------------------------------------------------------------------------------
def performGreedyMIExperimentalDesign(costFuncMI, nPoints, start=0, shard=None):
    """Greedy MI design over the cost function's pool (experimentalDesign.py:753-785).
    Returns the chosen POINTS (as the reference does); the indices are left in
    `costFuncMI.lastIndices`.  With `shard` (gpexp_b200.engine.Shard, every rank passing the same pool and the same
    gp.noise) the |V| x |V| factorisation is column-sharded over the ranks (ShardedMIEngine) -- required above |V| ~ 9e4.
    A per-point gp.noise works as in costFunctionGP_MI.evaluate (one finite value >= 0 per pool point, else ValueError)."""
    eng = _mi_new_engine(costFuncMI, nPoints, shard=shard)
    idx = eng.run(nPoints, start=start)
    costFuncMI.lastIndices = idx
    costFuncMI.lastEngine = eng
    return costFuncMI.mcPoints[idx, :]


def performGreedyVarExperimentalDesign(kernel, mcPoints, nPoints, dimension, weights=None, indKeepStart=[], shard=None):
    """Greedy maximum-posterior-variance design (experimentalDesign.py:787-845).

    Same contract as the reference: returns mcPoints[indKeep, :]; `indKeepStart` seeds the design and
    is extended in place (the reference mutates the caller's list, :808); selected points stay in the
    pool; the nugget is 0.0 (:825).  Extension: with `shard` (gpexp_b200.engine.Shard) every rank passes the full
    pool and works on its own contiguous block; all ranks return the same design.
    """
    indKeep = [] if indKeepStart == [] else indKeepStart
    dev = kernel._bind()
    lo, hi = 0, mcPoints.shape[0]
    if shard is not None:
        lo, hi = Shard.split(mcPoints.shape[0], shard.world, shard.rank)
    pool = dev.points(mcPoints[lo:hi])
    eng = GreedyVarEngine(dev, pool, max(nPoints, len(indKeep)), weights=None if weights is None else weights[lo:hi],
                          noise=0.0, shard=shard, index_offset=lo)
    for seed in list(indKeep):
        eng.force(int(seed))

    def progress(have):
        if VERBOSE and have % 10 == 0:
            print("Number of points we have ", have)

    idx = eng.run(nPoints, progress=progress)
    for i in idx[len(indKeep):]:
        indKeep.append(int(i))
    return mcPoints[indKeep, :]


def _checked_per_point(values, n, source, need_positive=False):
    """`values` as one float64 per point for n points (a nugget or an integration weight); `source` ("noise function
    returned", "gp.noise has", "mcWeights has") starts the message of the ValueError raised unless there is exactly one
    finite value >= 0 per point -- and, with need_positive, at least one value > 0."""
    v = np.asarray(values, dtype=np.float64).ravel()
    if v.size != n:
        raise ValueError(f"{source} {v.size} values for {n} points (one per point expected)")
    if not np.all(np.isfinite(v)):
        raise ValueError(f"{source} a value that is not finite")
    if np.any(v < 0.0):
        raise ValueError(f"{source} a negative value")
    if need_positive and not np.any(v > 0.0):
        raise ValueError(f"{source} no positive value (at least one must be > 0)")
    return v


def _noise_values(noiseFunc, points):
    """noiseFunc(points) as one float64 nugget per point; the noise function is user code, so its output is checked."""
    return _checked_per_point(noiseFunc(points), points.shape[0], "noise function returned")


def beginGreedyIVARExperimentalDesign(costFuncIVAR, candidates, nPoints, shard=None, resident=None):
    """The greedy-IVAR design as a steppable object (a gpexp_b200.engine.GreedyIVAREngine): `.run(n)` grows the design to n
    points (one C call for all steps), `.indices()`, `.pick_scores`, `.snapshot()` / `.restore()` re-time a step.

    candidates : (C, d) array.  With `shard` (a gpexp_b200.engine.Shard) every rank passes the FULL candidate array and
    scores its own contiguous block.
    resident : keep the M x C posterior covariance in HBM and update it by one rank-1 pass per step instead of
    re-contracting (identical picks, 16*M*C bytes per step instead of 2*M*n*C flop).  None = automatic: on when
    the matrix takes less than half of the free device memory.

    With a heteroscedastic `costFuncIVAR.space.noiseFunc`, the cost of design + [c] uses the nugget noiseFunc(design + [c])
    as costFunctionGP_IVAR.evaluate does, and gp.noise is not used.  The noise function must be pointwise and
    deterministic: it is evaluated once on this rank's candidates (the reference re-evaluates it on every design + [c]).
    It must return one finite value >= 0 per point, else ValueError.

    With `costFuncIVAR.mcWeights` the cost of design + [c] is the weighted sum over the integration points (see
    costFunctionGP_IVAR); the weights are replicated with the integration points, so every rank passes the same ones.

    With `costFuncIVAR.measure` the engine is a gpexp_b200.engine.MeasureIVAREngine (exact integral for a
    squared-exponential or Mehler kernel, `.run(n)`, `.indices()`, `.pick_scores`); shard and resident=True raise
    NotImplementedError there."""
    gp = costFuncIVAR.gaussianProcess
    meas = _ivar_measure(costFuncIVAR, "shard=" if shard is not None else "resident=True" if resident else None)
    weights = None if meas is not None else _ivar_weights(costFuncIVAR)
    lo, hi = 0, candidates.shape[0]
    if shard is not None:
        lo, hi = Shard.split(candidates.shape[0], shard.world, shard.rank)
    if costFuncIVAR.space.noiseFunc is not None:
        noise, cand_noise = 0.0, _noise_values(costFuncIVAR.space.noiseFunc, candidates[lo:hi])
    else:
        noise, cand_noise = _nugget_arg(gp.noise), None
        if isinstance(noise, np.ndarray):
            raise NotImplementedError("greedy IVAR needs a scalar noise")
        noise = float(noise)
    dev = gp.kernel._bind()
    fam, d, params = gp.kernel._gpx_spec()
    cand = dev.points(candidates[lo:hi])
    if meas is not None:
        return MeasureIVAREngine(dev, cand, nPoints, noise, (fam, d, params), meas, cand_noise=cand_noise)
    mc = _ivar_mc_points(costFuncIVAR, dev)
    if resident is None:
        import torch
        free, _ = torch.cuda.mem_get_info(dev.torch_device)
        resident = 8.0 * mc.n * cand.ld < 0.5 * free
        if shard is not None and shard.world > 1:  # every rank must take the same path
            flag = torch.tensor([1 if resident else 0], device=dev.torch_device)
            shard.dist.all_reduce(flag, op=shard.dist.ReduceOp.MIN, group=shard.group)
            resident = bool(flag.item())
    return GreedyIVAREngine(dev, cand, mc, nPoints, noise, prior_scale(fam, params), shard=shard, index_offset=lo,
                            resident=bool(resident), cand_noise=cand_noise, mc_weights=weights)


def performGreedyIVARExperimentalDesign(costFuncIVAR, candidates, nPoints, returnIndices=False, shard=None, resident=None):
    """Discrete greedy IVAR: at every step score `costFuncIVAR.evaluate(design + [c])` for every candidate
    c and add the arg-min -- what a loop over costFunctionGP_IVAR.evaluate (experimentalDesign.py:79-117)
    computes, restated with the Schur identity and run as one FP64 tensor-core contraction per step.
    Arguments as beginGreedyIVARExperimentalDesign.  Leaves lastIndices, lastScores (weighted costs when the cost function
    has mcWeights), lastPivots and illConditionedFrom (first step beyond which 1e-9 agreement with the reference's pinv
    arithmetic cannot be expected, or None) on the cost function."""
    eng = beginGreedyIVARExperimentalDesign(costFuncIVAR, candidates, nPoints, shard=shard, resident=resident)
    idx = eng.run(nPoints)
    costFuncIVAR.lastIndices = idx
    costFuncIVAR.lastScores = eng.pick_scores[: eng.n].cpu().numpy()
    costFuncIVAR.lastPivots = eng.pivots()
    costFuncIVAR.illConditionedFrom = eng.ill_conditioned_from(eng.zero_scale)
    if returnIndices:
        return idx
    return candidates[idx, :]


def refineGreedyIVARExperimentalDesign(costFuncIVAR, candidates, indices, maxSweeps=10, rtol=1e-8, returnIndices=False,
                                       shard=None, resident=None):
    """Improve a discrete IVAR design by exchange (Fedorov-type) passes over the candidate set.

    `indices` are candidate indices of the design (e.g. performGreedyIVARExperimentalDesign(..., returnIndices=True) or
    cf.lastIndices); duplicates are allowed as greedy allows them.  The engine is built as in
    beginGreedyIVARExperimentalDesign (noise function, mcWeights, every kernel family, both contraction cores, resident and
    sharded runs apply unchanged) and the given points are forced in order.  Then, as a queue, each step takes the oldest
    point out, scores every candidate c as the design of the other n-1 points plus c, and puts back the arg-min
    challenger (lowest index on ties) only if its cost is below (1 - rtol) x the removed point's own cost from the same
    pass; otherwise the removed point returns.  One sweep re-decides every point once; the pass stops after a sweep without
    a swap or after maxSweeps.  The cost never increases, and the result is 1-swap optimal up to rtol when the pass stops
    by itself.  rtol = 1e-8 lies well above the rounding of the scores, so the pass cannot cycle on ties.

    Returns the refined points (or indices with returnIndices) in factor order, the oldest first.  Leaves on the cost
    function: lastIndices, lastScores (design cost after every exchange step), lastSwaps (accepted swaps per sweep),
    lastCost (cost of the returned design: the mean posterior variance over mcPoints, or sum_m w_m var(x_m) with
    mcWeights) and illConditionedFrom (as performGreedyIVARExperimentalDesign, for the returned design).
    ValueError for indices that are not integers or lie outside the candidates, rtol < 0, maxSweeps < 0, and for a
    design whose factor has a non-finite entry (e.g. a repeated point under zero noise).  maxSweeps = 0 returns the
    input design.  NotImplementedError for a cost function with a `measure`."""
    _ivar_measure(costFuncIVAR, "exchange refinement")
    idx = _checked_exchange_args(indices, candidates.shape[0], maxSweeps, rtol, "candidate")
    n = idx.size
    eng = beginGreedyIVARExperimentalDesign(costFuncIVAR, candidates, n, shard=shard, resident=resident)
    for i in idx:
        eng.force(int(i))
    _require_finite_factor(eng.U, n)
    swaps = eng.exchange(int(maxSweeps), float(rtol))
    dev, mc = eng.dev, eng.mc
    total = dev.zeros(1)
    check(lib.gpx_sum_w(dev.h, ptr(eng.varM), ptr(eng.mc_weights), mc.n, ptr(total), dev.stream), "gpx_sum_w")
    cost = float(total.item())
    out = eng.indices()
    costFuncIVAR.lastIndices = out
    costFuncIVAR.lastScores = eng.exchange_costs.cpu().numpy()
    costFuncIVAR.lastSwaps = swaps
    costFuncIVAR.lastCost = abs(cost) if eng.mc_weights is not None else abs(cost / float(mc.n))
    costFuncIVAR.illConditionedFrom = eng.ill_conditioned_from(eng.zero_scale)
    if returnIndices:
        return out
    return candidates[out, :]


def _checked_exchange_args(indices, n_total, maxSweeps, rtol, what, unique=False):
    """The design of an exchange refinement as an int64 array, after the checks every refine driver makes (ValueError)."""
    idx = np.asarray(indices)
    if idx.ndim != 1 or idx.size == 0 or not np.issubdtype(idx.dtype, np.integer):
        raise ValueError(f"indices must be a non-empty 1-D sequence of integer {what} indices")
    if np.any(idx < 0) or np.any(idx >= n_total):
        raise ValueError(f"indices must lie in [0, {n_total})")
    if unique and np.unique(idx).size != idx.size:
        raise ValueError("indices must be distinct: a chosen point leaves the pool")
    if not rtol >= 0.0:
        raise ValueError(f"rtol must be >= 0, got {rtol}")
    if isinstance(maxSweeps, (bool, np.bool_)) or not isinstance(maxSweeps, (int, np.integer)) or maxSweeps < 0:
        raise ValueError(f"maxSweeps must be an integer >= 0, got {maxSweeps!r}")
    return idx.astype(np.int64)


def _require_finite_factor(U, n, strict=False):
    """ValueError unless the leading n x n block of the design factor U is finite (and, with strict, its diagonal > 0: the
    objectives take its logarithm)."""
    import torch
    u = U[:n, :n]
    ok = bool(torch.isfinite(u).all()) and (not strict or bool((torch.diagonal(u) > 0).all()))
    if not ok:
        raise ValueError("the design's Cholesky factor has a non-finite entry (a repeated or numerically dependent "
                         "point without noise): it cannot be refined")


def refineGreedyMIExperimentalDesign(costFuncMI, indices, maxSweeps=10, rtol=1e-8, returnIndices=False, shard=None):
    """Improve a discrete mutual-information design by exchange (Fedorov-type) passes over the cost function's pool.

    `indices` are distinct pool indices of the design (e.g. costFuncMI.lastIndices after
    performGreedyMIExperimentalDesign).  The engine is built as performGreedyMIExperimentalDesign builds it (scalar noise,
    per-point gp.noise and `shard` apply unchanged; the pool is factored once) and the given points are forced in order.
    Then, as a queue, each step takes the oldest point out of A (it returns to the pool S), scores every pool point y with
    the greedy's own score var(y | A) / var(y | S minus y) against the other n-1 points, and puts back the arg-max
    challenger (lowest index on ties) only if its score exceeds (1 + rtol) x the removed point's own score from the same
    pass; otherwise the removed point returns.  One sweep re-decides every point once; the pass stops after a sweep
    without a swap or after maxSweeps.

    The keep rule uses the greedy's score.  With zero noise a swap of j for c changes I(y_A; y_{V minus A}) by exactly
    1/2 log(score_c / score_j), so every accepted swap raises the mutual information.  With a nugget (scalar or per point)
    the score is not the exact gain and no monotone objective is claimed; maxSweeps bounds the pass.

    Returns the refined points (or indices with returnIndices) in factor order, the oldest first.  Leaves on the cost
    function: lastIndices, lastScores (the score of the point put back at every step), lastSwaps (accepted swaps per
    sweep) and lastMI (I(y_A; y_{V minus A}) in nats of the returned design, from its two Cholesky factors).
    ValueError for repeated, out-of-range or non-integer indices, rtol < 0, maxSweeps < 0 and a factor with a non-finite
    entry.  maxSweeps = 0 returns the input design."""
    idx = _checked_exchange_args(indices, len(costFuncMI.mcPoints), maxSweeps, rtol, "pool", unique=True)
    n = idx.size
    eng = _mi_new_engine(costFuncMI, n, shard=shard, keep_factors=True)
    for i in idx:
        eng.force(int(i))
    _require_finite_factor(eng.UA, n, strict=True)
    _require_finite_factor(eng.UQ, n, strict=True)
    swaps = eng.exchange(int(maxSweeps), float(rtol))
    out = eng.indices()
    costFuncMI.lastIndices = out
    costFuncMI.lastScores = eng.exchange_costs.cpu().numpy()
    costFuncMI.lastSwaps = swaps
    costFuncMI.lastMI = eng.mutual_information()
    if returnIndices:
        return out
    return costFuncMI.mcPoints[out, :]


def refineGreedyVarExperimentalDesign(kernel, mcPoints, indices, weights=None, nFixed=0, maxSweeps=10, rtol=1e-8,
                                      returnIndices=False, returnInfo=False, shard=None):
    """Improve a discrete maximum-variance (conditional entropy) design by exchange passes over the pool mcPoints.

    The nugget is 0.0 and `weights` (one finite value >= 0 per pool point, at least one > 0) scales the variances, as in
    performGreedyVarExperimentalDesign.  The first `nFixed` indices are fixed seeds (what indKeepStart holds there): they
    keep their place and are never removed.  The others are exchanged as a queue: each step takes the oldest exchangeable
    point out (position nFixed), scores every pool point by its posterior variance x weight given the other n-1 points,
    and appends the arg-max challenger (lowest index on ties) only if its score exceeds (1 + rtol) x the removed point's
    own score from the same pass; otherwise the removed point returns.  One sweep re-decides every exchangeable point
    once; the pass stops after a sweep without a swap or after maxSweeps.  Every accepted swap raises
    log det K_AA + sum_{i in A} log w_i by log(score_c / score_j) (without weights, log det K_AA: the D-optimal /
    maximum-entropy exchange).  With `shard` every rank passes the full pool and works on its own contiguous block.

    Returns the refined points (or indices with returnIndices) in factor order: the seeds, then the oldest first.  With
    returnInfo, (result, info) with info = {"indices", "scores" (score of the point put back at every step), "swaps"
    (accepted swaps per sweep), "logdet" (the objective above, of the returned design)}.  ValueError for repeated (their
    Gram without a nugget is singular), out-of-range or non-integer indices, nFixed outside [0, len(indices)], bad
    weights, rtol < 0, maxSweeps < 0 and a factor with a non-finite entry or a zero pivot.  maxSweeps = 0 returns the
    input design."""
    N = mcPoints.shape[0]
    idx = _checked_exchange_args(indices, N, maxSweeps, rtol, "pool", unique=True)
    n = idx.size
    if isinstance(nFixed, (bool, np.bool_)) or not isinstance(nFixed, (int, np.integer)) or not 0 <= nFixed <= n:
        raise ValueError(f"nFixed must be an integer in [0, {n}], got {nFixed!r}")
    w = None if weights is None else _checked_per_point(weights, N, "weights has", need_positive=True)
    dev = kernel._bind()
    lo, hi = 0, N
    if shard is not None:
        lo, hi = Shard.split(N, shard.world, shard.rank)
    eng = GreedyVarEngine(dev, dev.points(mcPoints[lo:hi]), n, weights=None if w is None else w[lo:hi], noise=0.0,
                          shard=shard, index_offset=lo, keep_factors=True)
    for i in idx:
        eng.force(int(i))
    _require_finite_factor(eng.U, n, strict=True)
    swaps = eng.exchange(int(maxSweeps), float(rtol), first=int(nFixed))
    out = eng.indices()
    total = dev.zeros(1)
    check(lib.gpx_logdet_chol(dev.h, ptr(eng.U), n, eng.U.shape[1], ptr(total), dev.stream), "gpx_logdet_chol")
    logdet = float(total.item())
    if w is not None:
        logdet += float(np.sum(np.log(w[out])))
    result = out if returnIndices else mcPoints[out, :]
    if returnInfo:
        return result, {"indices": out, "scores": eng.exchange_costs.cpu().numpy(), "swaps": swaps, "logdet": logdet}
    return result


def scoreCandidatesIVAR(costFuncIVAR, design, candidates, shard=None):
    """One stateless IVAR scoring pass from HOST buffers: cost of design + [c] for every candidate c.
    Returns (costs, argmin index).  With `shard` every rank passes the full candidate array, scores its own contiguous
    block and returns (costs of its block, GLOBAL arg-min index).  This is the end-to-end call bench.py times (`e2e`).
    A heteroscedastic `costFuncIVAR.space.noiseFunc` is honoured as in beginGreedyIVARExperimentalDesign: the design
    Gram gets the nugget noiseFunc(design) and candidate c the noise noiseFunc(c).  `costFuncIVAR.mcWeights` weights the
    integration points as in costFunctionGP_IVAR.evaluate; `costFuncIVAR.measure` makes the costs the exact integrals
    (shard= then raises NotImplementedError)."""
    gp = costFuncIVAR.gaussianProcess
    meas = _ivar_measure(costFuncIVAR, "shard=" if shard is not None else None)
    weights = None if meas is not None else _ivar_weights(costFuncIVAR)
    noiseFunc = costFuncIVAR.space.noiseFunc
    lo, hi = 0, candidates.shape[0]
    if shard is not None:
        lo, hi = Shard.split(candidates.shape[0], shard.world, shard.rank)
    n = design.shape[0]
    if noiseFunc is None:
        noise = nugget = float(_nugget_arg(gp.noise))
        cand_noise = None
    else:
        noise, cand_noise = 0.0, _noise_values(noiseFunc, candidates[lo:hi])
        nugget = _noise_values(noiseFunc, design) if n else None
    dev = gp.kernel._bind()
    fam, d, params = gp.kernel._gpx_spec()
    cand = dev.points(candidates[lo:hi])
    if meas is not None:
        eng = MeasureIVAREngine(dev, cand, max(n, 1), noise, (fam, d, params), meas, cand_noise=cand_noise)
    else:
        mc = dev.points(costFuncIVAR.mcPoints)
        eng = GreedyIVAREngine(dev, cand, mc, max(n, 1), noise, prior_scale(fam, params), cand_noise=cand_noise,
                               mc_weights=weights)
    if n:
        eng.load_design(DesignFactor(dev, dev.points(design), nugget))
    eng.score()
    costs = eng.scores[: cand.n].cpu().numpy()
    best = int(eng.idx.item())
    if shard is None or shard.world == 1:
        return costs, best
    import torch
    mine = torch.tensor([costs[best] if best >= 0 else np.inf, float(best + lo)], dtype=torch.float64, device=dev.torch_device)
    allb = torch.zeros(2 * shard.world, dtype=torch.float64, device=dev.torch_device)
    shard.all_gather(allb, mine)
    allb = allb.cpu().numpy().reshape(shard.world, 2)
    return costs, int(allb[np.lexsort((allb[:, 1], allb[:, 0]))[0], 1])


# what install_as_gpExp() rebinds on the reference's own module: class methods and module-level functions
DEVICE_METHODS = {
    "costFunctionGP_IVAR": {"evaluate": _ivar_evaluate, "derivative": _ivar_derivative},
    "costFunctionGP_MI": {"evaluate": _mi_evaluate},
}
DEVICE_FUNCTIONS = {
    "performGreedyVarExperimentalDesign": performGreedyVarExperimentalDesign,
    "performGreedyMIExperimentalDesign": performGreedyMIExperimentalDesign,
    "performGreedyIVARExperimentalDesign": performGreedyIVARExperimentalDesign,
    "beginGreedyIVARExperimentalDesign": beginGreedyIVARExperimentalDesign,
    "refineGreedyIVARExperimentalDesign": refineGreedyIVARExperimentalDesign,
    "refineGreedyMIExperimentalDesign": refineGreedyMIExperimentalDesign,
    "refineGreedyVarExperimentalDesign": refineGreedyVarExperimentalDesign,
    "scoreCandidatesIVAR": scoreCandidatesIVAR,
}
