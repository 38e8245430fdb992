"""Cost functions and discrete greedy design drivers behind the reference's names (gpExp/experimentalDesign.py), running on
the device-resident engines of gpexp_b200.engine.

    costFunctionGP_IVAR.evaluate / derivative   experimentalDesign.py:79-117, :148-179   (version 1, MC-integrated variance)
    costFunctionGP_MI.evaluate                  experimentalDesign.py:252-285
    performGreedyVarExperimentalDesign          experimentalDesign.py:787-845
    performGreedyMIExperimentalDesign           experimentalDesign.py:753-785
    performGreedyIVARExperimentalDesign,        NEW: the discrete greedy-IVAR driver the north star asks for; the
    beginGreedyIVARExperimentalDesign,          reference only has the per-design cost function (SURVEY.md 3.2 / 8c)
    scoreCandidatesIVAR

The continuous optimisers that CALL these cost functions (ExperimentalDesignDerivative / NoDerivative and the batch-greedy
wrappers, experimentalDesign.py:296-751) are deliberately not re-typed here: with the reference importable,
`gpexp_b200.install_as_gpExp()` rebinds the functions of `DEVICE_METHODS` / `DEVICE_FUNCTIONS` onto the reference's own
module, and its optimiser loops then drive the device path unchanged.
"""
import copy
import itertools

import numpy as np

from ._lib import check, lib
from .device import ptr
from .engine import (DesignFactor, GreedyIVAREngine, GreedyVarEngine, Shard, ShardedMIEngine, prior_scale)
from .gp_kernel_utilities import _nugget_arg

VERBOSE = True  # the reference prints its progress unconditionally (experimentalDesign.py:812-813)


# ---- costFunctionGP_IVAR --------------------------------------------------------------------------------------------------
def _ivar_mc_points(self, dev):
    """The Monte-Carlo integration points as a device point set, uploaded once per cost function."""
    cached = self.__dict__.get("_mc_dev")
    if cached is None or cached.dev is not dev or cached.n != len(self.mcPoints):
        cached = self.__dict__["_mc_dev"] = dev.points(self.mcPoints)
    return cached


def _ivar_evaluate(self, inputPoints):
    """|mean posterior variance over the MC points| for the design `inputPoints` (:79-117)."""
    assert inputPoints.shape == (self.numInputs, self.space.dimension), \
        ("inputPoints are the wrong size: ", inputPoints.shape)
    if self.version != 1:
        raise NotImplementedError("IVAR version 0 needs a kernel eigen-basis that no shipped kernel provides "
                                  "(experimentalDesign.py:119-146 is unreachable)")
    gp = self.gaussianProcess
    if self.space.noiseFunc is None:
        gp.addNodesAndComputeCovariance(inputPoints)
    else:
        gp.addNodesAndComputeCovariance(inputPoints, self.space.noiseFunc(inputPoints))
    f = gp._factor
    mc = _ivar_mc_points(self, f.dev)
    _, var = f.solve_gram(mc)
    total = f.dev.zeros(1)
    check(lib.gpx_sum(f.dev.h, ptr(var), mc.n, ptr(total), f.dev.stream), "gpx_sum")
    return np.abs(float(total.item()) / float(self.nMC))


def _ivar_derivative(self, inputPoints):
    """Gradient of the IVAR cost with respect to the design coordinates, shape (nPoints*dimension,)
    (:148-179, version 1): the row mean over the MC points of GP.evaluateVarianceDerivative, with the noise function's
    own derivative in the heteroscedastic case.  Squared-exponential kernels."""
    gp = self.gaussianProcess
    gp.kernel._require_derivative()
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
    check(lib.gpx_rowsum(f.dev.h, ptr(full), rows, mc.n, mc.ld, 1.0 / float(self.nMC), ptr(out), f.dev.stream), "gpx_rowsum")
    return out[:rows].cpu().numpy()


# ---- costFunctionGP_MI ----------------------------------------------------------------------------------------------------
def _mi_new_engine(self, n_max):
    gp = self.gaussianProcess
    noise = _nugget_arg(gp.noise)
    if isinstance(noise, np.ndarray):
        raise NotImplementedError("MI with per-point noise is not supported on the device path")
    # left-looking blocked set-up (measured faster than a right-looking dense engine on one GPU as well:
    # |V| = 40 000: 2.33 s vs 2.97 s)
    return ShardedMIEngine(gp.kernel._bind(), self.mcPoints, n_max, float(noise))


def _mi_evaluate(self, index, indexAdded):
    """MI ratio of candidate `index` given the already chosen `indexAdded` (:252-285); shape (1,).

    The reference pays two pseudo-inverses per call; here the O(|V|^3) factorisation of the pool is built once and kept
    (until the pool, the kernel or the noise changes), the chosen points are replayed only when `indexAdded` stops
    extending the previous call's list, and the scores of ALL candidates for that list are kept, so the reference's loop
    `for ind in options: evaluate(ind, indKeep)` (:776-777) costs one scoring pass per greedy step."""
    added = [int(i) for i in indexAdded]
    gp = self.gaussianProcess
    fam, _, params = gp.kernel._gpx_spec()
    key = (fam, tuple(np.ravel(params)), float(_nugget_arg(gp.noise)), id(self.mcPoints), len(self.mcPoints))
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
    version=1, mcPoints=...)  (:60-75).  Holds a shallow copy of the GP; without mcPoints, 10 000 samples of the space."""

    def __init__(self, gaussianProcess, nInputs, space, version=1, **kwargs):
        costFunctionBase.__init__(self, nInputs, space)
        self.gaussianProcess, self.version = copy.copy(gaussianProcess), version
        if version == 1:
            pts = kwargs['mcPoints'] if 'mcPoints' in kwargs else space.sample((10000, space.dimension))
            self.mcPoints, self.nMC = pts, len(pts)

    evaluate = _ivar_evaluate
    derivative = _ivar_derivative


class costFunctionGP_MI(costFunctionBase):
    """Krause-Guestrin mutual-information ratio var(y|A) / var(y|V minus A minus y) over a candidate pool (:223-285).
    The GP passed in is used directly, not copied (:227); pool = mcpoints[nmc], a 10 x 10 grid (square=True, 2-D) or 200
    samples of the space."""

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
    `costFuncMI.lastIndices`.  With `shard` (gpexp_b200.engine.Shard, every rank passing the same pool) the
    |V| x |V| factorisation is column-sharded over the ranks (ShardedMIEngine) -- required above |V| ~ 9e4."""
    if shard is not None:
        gp = costFuncMI.gaussianProcess
        noise = _nugget_arg(gp.noise)
        if isinstance(noise, np.ndarray):
            raise NotImplementedError("MI with per-point noise is not supported on the device path")
        eng = ShardedMIEngine(gp.kernel._bind(), costFuncMI.mcPoints, nPoints, float(noise), shard=shard)
    else:
        eng = _mi_new_engine(costFuncMI, nPoints)
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


def _noise_values(noiseFunc, points):
    """noiseFunc(points) as one float64 nugget per point; the noise function is user code, so its output is checked."""
    nu = np.asarray(noiseFunc(points), dtype=np.float64).ravel()
    if nu.size != points.shape[0]:
        raise ValueError(f"noise function returned {nu.size} values for {points.shape[0]} points (one per point expected)")
    if not np.all(np.isfinite(nu)):
        raise ValueError("noise function returned a value that is not finite")
    if np.any(nu < 0.0):
        raise ValueError("noise function returned a negative value")
    return nu


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
    It must return one finite value >= 0 per point, else ValueError."""
    gp = costFuncIVAR.gaussianProcess
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
                            resident=bool(resident), cand_noise=cand_noise)


def performGreedyIVARExperimentalDesign(costFuncIVAR, candidates, nPoints, returnIndices=False, shard=None, resident=None):
    """Discrete greedy IVAR: at every step score `costFuncIVAR.evaluate(design + [c])` for every candidate
    c and add the arg-min -- what a loop over costFunctionGP_IVAR.evaluate (experimentalDesign.py:79-117)
    computes, restated with the Schur identity and run as one FP64 tensor-core contraction per step.
    Arguments as beginGreedyIVARExperimentalDesign.  Leaves lastIndices, lastScores, lastPivots and illConditionedFrom
    (first step beyond which 1e-9 agreement with the reference's pinv arithmetic cannot be expected, or None) on the
    cost function."""
    eng = beginGreedyIVARExperimentalDesign(costFuncIVAR, candidates, nPoints, shard=shard, resident=resident)
    idx = eng.run(nPoints)
    costFuncIVAR.lastIndices = idx
    costFuncIVAR.lastScores = eng.pick_scores[: eng.n].cpu().numpy()
    costFuncIVAR.lastPivots = eng.pivots()
    costFuncIVAR.illConditionedFrom = eng.ill_conditioned_from(eng.zero_scale)
    if returnIndices:
        return idx
    return candidates[idx, :]


def scoreCandidatesIVAR(costFuncIVAR, design, candidates, shard=None):
    """One stateless IVAR scoring pass from HOST buffers: cost of design + [c] for every candidate c.
    Returns (costs, argmin index).  With `shard` every rank passes the full candidate array, scores its own contiguous
    block and returns (costs of its block, GLOBAL arg-min index).  This is the end-to-end call bench.py times (`e2e`).
    A heteroscedastic `costFuncIVAR.space.noiseFunc` is honoured as in beginGreedyIVARExperimentalDesign: the design
    Gram gets the nugget noiseFunc(design) and candidate c the noise noiseFunc(c)."""
    gp = costFuncIVAR.gaussianProcess
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
    mc = dev.points(costFuncIVAR.mcPoints)
    eng = GreedyIVAREngine(dev, cand, mc, max(n, 1), noise, prior_scale(fam, params), cand_noise=cand_noise)
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
    "scoreCandidatesIVAR": scoreCandidatesIVAR,
}
