"""Device-resident greedy design engines.

Every engine keeps its whole state in HBM (W factors, running variances, pivot records, picked
indices) and advances one greedy step with a fixed, host-sync-free sequence of C-ABI launches; the
host reads the picked indices back once at the end.  Layouts (all float64):

    X      d x ld        dimension-major coordinates of a point set (ld = roundup(n, 128))
    W      ncap x ld     row i = i-th row of L^-1 K(D, .) for every point of the set (K-major for DMMA)
    var    ld            running posterior variance of every point
    rec    19 + ncap     pivot record: score, global index, var_p + noise (or + nu(p)), x_p[16], W[0:n, p]

Candidates shard across ranks (one process per GPU): each rank owns a contiguous block of the pool,
the integration points are replicated, and the only exchange per step is one NCCL all-gather of the
ranks' pivot records followed by an identical on-device selection (lowest score/highest score, ties
to the lowest global index) -- so every rank appends bit-identical rows.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings

import numpy as np
import torch

from . import _lib
from ._lib import GpxError, check, lib
from .device import Device, PointSet, prologue_operands, ptr, roundup

HDR = _lib.GPX_PIVOT_HDR
ZERO_VAR_TOL = 1e-13
# A greedy step whose pivot var_D(p) + noise falls below this fraction of the prior variance means
# cond(K_DD + noise I) >~ 1e7: eps * cond exceeds the 1e-9 parity contract with the reference's pinv arithmetic
# (SURVEY.md section 7, demo.py:52-58 stress values).  The run continues; the step is reported.
PIVOT_WARN_RATIO = 1e-7


class GpxConditionWarning(RuntimeWarning):
    """The design Gram matrix became too ill conditioned for the 1e-9 parity contract (or was jittered to factor)."""


class Shard:
    """Position of this process in a candidate-sharded job (torch.distributed, NCCL on GPUs)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)

    @staticmethod
    def split(n_total: int, world: int, rank: int):
        """Contiguous block [lo, hi) of rank `rank` (remainder spread over the first ranks)."""
        base, rem = divmod(n_total, world)
        lo = rank * base + min(rank, rem)
        return lo, lo + base + (1 if rank < rem else 0)

    def all_gather(self, out: torch.Tensor, inp: torch.Tensor):
        self.dist.all_gather_into_tensor(out, inp, group=self.group)

    def native(self, dev: Device) -> bool:
        """Give the device handle its own NCCL communicator (gpx_comm_init) so that the C-side greedy loops can run
        the per-step exchange themselves.  The 128-byte id travels over torch.distributed once.  NCCL groups only."""
        if self.world == 1 or self.dist.get_backend(self.group) != "nccl":
            return False
        if int(lib.gpx_comm_size(dev.h)) == self.world:
            return True
        buf = (C.c_char * _lib.GPX_COMM_ID_BYTES)()
        if self.rank == 0:
            check(lib.gpx_comm_unique_id(buf, _lib.GPX_COMM_ID_BYTES), "gpx_comm_unique_id")
        t = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).to(dev.torch_device)
        self.dist.broadcast(t, src=self.dist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
        raw = bytes(t.cpu().numpy().tobytes())
        torch.cuda.current_stream(dev.torch_device).synchronize()
        check(lib.gpx_comm_init(dev.h, raw, self.rank, self.world), "gpx_comm_init")
        return True


def prior_scale(family: int, params) -> float:
    """k(0,0): the magnitude against which 'numerically zero variance' is judged."""
    params = np.asarray(params, dtype=np.float64)
    if family == _lib.SE:
        return float(abs(params[-1]))
    if family == _lib.MATERN32:
        return float(abs(params[1]))
    return float(np.prod((1.0 - params ** 2.0) ** -0.5))


class _Pivoting:
    """Shared pivot plumbing: gather the local best, exchange across ranks, keep the history."""

    def _init_pivot(self, dev: Device, ncap: int, n_max: int, shard, index_offset: int):
        self.dev = dev
        self.ncap = ncap
        self.n_max = n_max
        self.n = 0
        self.shard = shard
        self.index_offset = index_offset
        self.reclen = HDR + ncap
        self.rec = dev.zeros(self.reclen)
        self.best = dev.zeros(1)
        self.idx = dev.zeros(1, dtype=torch.int64)
        self.picks = dev.zeros(max(n_max, 1), dtype=torch.int64)
        self.pick_scores = dev.zeros(max(n_max, 1))
        self.pick_pivots = dev.zeros(max(n_max, 1))
        if shard is not None and shard.world > 1:
            self.rec_all = dev.zeros(shard.world * self.reclen)
            self.rec_win = dev.zeros(self.reclen)
        else:
            self.rec_all = None
            self.rec_win = self.rec

    def _gather(self, W, ld, var, X: PointSet, noise: float, minimize: bool):
        dev = self.dev
        check(lib.gpx_gather_pivot(dev.h, ptr(W), ld, self.n, ptr(var), ptr(X.X), X.ld, ptr(self.best), ptr(self.idx),
                                   self.index_offset, ptr(getattr(self, "index_map", None)), noise, ptr(self.rec), dev.stream),
              "gpx_gather_pivot")
        if self.rec_all is not None:
            self.shard.all_gather(self.rec_all, self.rec)
            check(lib.gpx_select_pivot(dev.h, ptr(self.rec_all), self.shard.world, self.reclen, self.n,
                                       1 if minimize else 0, ptr(self.rec_win), dev.stream), "gpx_select_pivot")

    def _local_of(self, global_index: int) -> int:
        local = global_index - self.index_offset
        return local if 0 <= local < self._local_count() else -1

    def _force_local(self, global_index: int):
        """Make `global_index` the pivot of this step (seeds / given designs): owner rank points at it."""
        local = self._local_of(global_index)
        self.idx.fill_(local)
        self.best.zero_()

    def _record(self, U=None, ldu=0):
        dev = self.dev
        check(lib.gpx_store_pivot(dev.h, ptr(self.rec_win), self.n, ptr(U), ldu, ptr(self.picks), ptr(self.pick_scores),
                                  ptr(self.pick_pivots), dev.stream), "gpx_store_pivot")

    def indices(self) -> np.ndarray:
        return self.picks[: self.n].cpu().numpy()

    def pivots(self) -> np.ndarray:
        """var_D(p) + noise of the pick, for every pick in pick order (noise = nu(p) for a per-candidate noise)."""
        return self.pick_pivots[: self.n].cpu().numpy()

    def ill_conditioned_from(self, scale: float):
        """First step whose pivot fell below PIVOT_WARN_RATIO * scale (None if none did); warns once."""
        piv = self.pivots()
        bad = np.nonzero(~(piv > PIVOT_WARN_RATIO * scale))[0]
        if bad.size == 0:
            return None
        step = int(bad[0])
        warnings.warn(f"greedy design: pivot {piv[step]:.3e} at step {step} is below {PIVOT_WARN_RATIO:g} x the prior "
                      f"variance: the design Gram matrix is too ill conditioned for 1e-9 agreement with a pinv-based "
                      f"evaluation from this step on (add noise or shorten the design)", GpxConditionWarning, stacklevel=3)
        return step

    def _native_ready(self) -> bool:
        """The C-side loop can run this engine: single rank, or an NCCL shard whose ranks all hold candidates."""
        if self.shard is None or self.shard.world == 1:
            return True
        if getattr(self, "_native", None) is None:
            ok = self.shard.native(self.dev) and self._local_count() > 0
            flag = torch.tensor([1 if ok else 0], device=self.dev.torch_device)
            self.shard.dist.all_reduce(flag, op=self.shard.dist.ReduceOp.MIN, group=self.shard.group)
            self._native = bool(flag.item())
        return self._native


class GreedyVarEngine(_Pivoting):
    """Greedy maximum posterior variance (conditional entropy), experimentalDesign.py:787-845, as an
    incremental diagonally-pivoted Cholesky of K_CC: per step one arg-max and one HBM-bound row append."""

    def __init__(self, dev: Device, pool: PointSet, n_max: int, weights=None, noise: float = 0.0, shard=None,
                 index_offset: int = 0):
        self.pool = pool
        self.noise = float(noise)
        ncap = max(int(n_max), 1)
        self._init_pivot(dev, ncap, n_max, shard, index_offset)
        self.W = dev.zeros(ncap, pool.ld)
        self.var = dev.zeros(pool.ld)
        check(lib.gpx_prior_diag(dev.h, ptr(pool.X), pool.n, pool.ld, ptr(self.var), dev.stream), "gpx_prior_diag")
        self.weights = None if weights is None else dev.upload(np.asarray(weights, dtype=np.float64))
        self.score_trace = None

    def _local_count(self):
        return self.pool.n

    def select(self):
        dev = self.dev
        check(lib.gpx_argreduce(dev.h, ptr(self.var), ptr(self.weights), None, self.pool.n, 0, ptr(self.best),
                                ptr(self.idx), dev.stream), "gpx_argreduce")

    def append(self):
        dev, pool = self.dev, self.pool
        self._gather(self.W, pool.ld, self.var, pool, self.noise, minimize=False)
        check(lib.gpx_append_row(dev.h, _lib.ROW_KERNEL, ptr(self.rec_win), None, ptr(pool.X), pool.n, pool.ld,
                                 ptr(self.W), pool.ld, self.n, ptr(self.var), dev.stream), "gpx_append_row")
        self._record()
        self.n += 1

    def force(self, global_index: int):
        self._force_local(int(global_index))
        self.append()

    def step(self):
        if self.score_trace is not None:
            v = self.var[: self.pool.n]
            self.score_trace.append((v * self.weights if self.weights is not None else v).cpu().numpy().copy())
        self.select()
        self.append()

    def _state(self):
        st = _lib.VarState()
        pool = self.pool
        st.X, st.C, st.ld, st.W, st.var, st.weights = ptr(pool.X), pool.n, pool.ld, ptr(self.W), ptr(self.var), ptr(self.weights)
        st.ncap, st.index_offset, st.noise = self.ncap, self.index_offset, self.noise
        st.best, st.idx, st.rec = ptr(self.best), ptr(self.idx), ptr(self.rec)
        st.rec_all = ptr(self.rec_all)
        st.rec_win = ptr(self.rec_win) if self.rec_all is not None else None
        st.picks, st.pick_scores, st.pick_pivots = ptr(self.picks), ptr(self.pick_scores), ptr(self.pick_pivots)
        return st

    def run(self, n_points: int, progress=None, chunk: int = 10):
        """Grow the design to n_points.  Without a score trace the steps are issued by the C-side loop
        (gpx_var_greedy_run) in chunks of `chunk`, between which `progress(n)` is called (the reference prints every
        10 points, experimentalDesign.py:812-813)."""
        if self.score_trace is not None or not self._native_ready():
            while self.n < n_points:
                if progress is not None:
                    progress(self.n)
                self.step()
            return self.indices()
        st = self._state()
        while self.n < n_points:
            if progress is not None:
                progress(self.n)
            stop = min(n_points, (self.n // chunk + 1) * chunk) if progress is not None else n_points
            check(lib.gpx_var_greedy_run(self.dev.h, C.byref(st), self.n, stop, self.dev.stream), "gpx_var_greedy_run")
            self.n = stop
        return self.indices()


class DesignFactor:
    """Cholesky factor of a given design's Gram matrix and the solves built on it (GP class backend):
    K(D,D) + diag(nugget) = U^T U  (K1 + K2), W = U^-T K(D, X) and posterior variances (K1+K3+K4)."""

    def __init__(self, dev: Device, design: PointSet, nugget):
        self.dev, self.design = dev, design
        n = design.n
        self.n = n
        self.ldu = design.ld
        self.U = dev.zeros(max(n, 1), self.ldu)
        self.info = dev.zeros(1, dtype=torch.int32)
        nug_vec = None
        nug = 0.0
        if isinstance(nugget, np.ndarray):
            nug_vec = dev.upload(nugget.astype(np.float64).ravel())
        else:
            nug = float(nugget)
        self.jitter = 0.0
        if n:
            check(lib.gpx_gram(dev.h, ptr(design.X), n, design.ld, ptr(design.X), n, design.ld, ptr(self.U), self.ldu, 1,
                               ptr(nug_vec), nug, dev.stream), "gpx_gram")
            self._cov = self.U.clone()
            check(lib.gpx_potrf(dev.h, ptr(self.U), n, self.ldu, ptr(self.info), dev.stream), "gpx_potrf")
            bad = int(self.info.item())
            scale = float(torch.diagonal(self._cov[:n, :n]).abs().max().item())
            if not bad:
                # a pivot that survives only as round-off (U_ii^2 <= 1e-13 x the largest diagonal entry) is a numerically
                # singular Gram as well: cond >~ 1e13, everything solved against this factor would be noise
                piv = torch.diagonal(self.U[:n, :n]) ** 2
                if not bool(torch.isfinite(piv).all()) or float(piv.min().item()) <= 1e-13 * scale:
                    bad = int(torch.argmin(torch.nan_to_num(piv, nan=-1.0)).item()) + 1
            if bad:
                # The reference pseudo-inverts (np.linalg.pinv, gp.py:181) and so tolerates numerically singular Grams
                # (noise 0 with duplicate or nearly dependent nodes); a Cholesky factor does not exist there.  Retry once
                # with a jitter at the level of pinv's own cut-off region, loudly; fail if that is not enough.
                self.jitter = 1e-10 * scale
                warnings.warn(f"Gram matrix is not numerically positive definite (pivot {bad - 1} of {n}); factoring "
                              f"K + {self.jitter:.3e} I instead -- results near the null directions differ from a "
                              f"pseudo-inverse", GpxConditionWarning, stacklevel=3)
                self.U.copy_(self._cov)
                self.U[:n, :n].diagonal().add_(self.jitter)
                check(lib.gpx_potrf(dev.h, ptr(self.U), n, self.ldu, ptr(self.info), dev.stream), "gpx_potrf")
                bad = int(self.info.item())
                if bad:
                    raise GpxError(f"Gram matrix is not positive definite even with jitter {self.jitter:.3e}: "
                                   f"failing pivot {bad - 1} of {n}")
        else:
            self._cov = self.U.clone()
        self._Ut = None

    def covariance(self) -> np.ndarray:
        return self._cov[: self.n, : self.n].cpu().numpy()

    def pivot_failure(self) -> int:
        return int(self.info.item())

    def Ut(self):
        if self._Ut is None:
            dev = self.dev
            self._Ut = dev.zeros(max(self.n, 1), self.ldu)
            check(lib.gpx_transpose(dev.h, ptr(self.U), self.n, self.n, self.ldu, ptr(self._Ut), self.ldu, dev.stream),
                  "gpx_transpose")
        return self._Ut

    def solve_gram(self, X: PointSet, W=None, want_var=True):
        """W = U^-T K(D, X) (n x X.ld) and var = k(x,x) - colsumsq(W)."""
        dev, D = self.dev, self.design
        if W is None:
            W = dev.zeros(max(self.n, 1), X.ld)
        var = dev.zeros(X.ld) if want_var else None
        check(lib.gpx_trsm_gram(dev.h, ptr(self.U), self.n, self.ldu, ptr(D.X), D.ld, ptr(X.X), X.n, X.ld, ptr(W), X.ld,
                                ptr(var), dev.stream), "gpx_trsm_gram")
        return W, var

    def solve_vector(self, y: np.ndarray) -> np.ndarray:
        """(U^T U)^-1 y : GP.train coefficients, gp.py:101."""
        dev = self.dev
        B = dev.zeros(max(self.n, 1), 2)
        B[: self.n, 0] = dev.upload(np.asarray(y, dtype=np.float64))
        check(lib.gpx_trsm(dev.h, ptr(self.U), self.n, self.ldu, ptr(B), 1, 2, dev.stream), "gpx_trsm")
        check(lib.gpx_trsm_back(dev.h, ptr(self.Ut()), self.n, self.ldu, ptr(B), 1, 2, dev.stream), "gpx_trsm_back")
        return B[: self.n, 0].cpu().numpy()

    def logdet(self) -> float:
        """log det(K + nugget) = 2 sum log U_ii."""
        dev = self.dev
        out = dev.zeros(1)
        check(lib.gpx_logdet_chol(dev.h, ptr(self.U), self.n, self.ldu, ptr(out), dev.stream), "gpx_logdet_chol")
        return float(out.item())

    def whitened_norm2(self, y: np.ndarray) -> float:
        """|U^-T y|^2 = y^T (K + nugget)^-1 y."""
        dev = self.dev
        B = dev.zeros(max(self.n, 1), 2)
        B[: self.n, 0] = dev.upload(np.asarray(y, dtype=np.float64))
        check(lib.gpx_trsm(dev.h, ptr(self.U), self.n, self.ldu, ptr(B), 1, 2, dev.stream), "gpx_trsm")
        out = dev.zeros(2)
        check(lib.gpx_colsumsq(dev.h, ptr(B), self.n, 1, 2, None, ptr(out), dev.stream), "gpx_colsumsq")
        return float(out[0].item())

    def variance_gradient(self, X: PointSet, noise_grad=None, same_location=None):
        """(n*d) x X.ld device matrix  out[j*d+k, m] = d var(x_m) / d design[j,k]  as GP.evaluateVarianceDerivative
        (gp.py:282-341) defines it.  Squared-exponential kernels only.

        Heteroscedastic branch (gp.py:314-318): noise_grad[j,k] = d noise(p_j)/d p_j[k] enters the derivative of the
        design Gram at every pair of coincident design points -- same_location[z,j] true where p_z == p_j (the diagonal
        for distinct points) -- i.e. E[z, j*d+k] = same[z,j] * noise_grad[j,k] is added to dK/dp before the contraction and
        the doubly counted diagonal is taken out again inside gpx_se_var_grad."""
        dev, D = self.dev, self.design
        n, d = self.n, D.d
        W, _ = self.solve_gram(X, want_var=False)
        check(lib.gpx_trsm_back(dev.h, ptr(self.Ut()), n, self.ldu, ptr(W), X.n, X.ld, dev.stream), "gpx_trsm_back")  # At = P K(D,X)
        ldn = roundup(n * d)
        dct = dev.zeros(max(n, 1), ldn)
        check(lib.gpx_se_dgram(dev.h, ptr(D.X), n, D.ld, ptr(D.X), n, D.ld, ptr(dct), ldn, dev.stream), "gpx_se_dgram")
        diag = None
        if noise_grad is not None:
            ng = np.asarray(noise_grad, dtype=np.float64).reshape(n, d)
            same = np.eye(n, dtype=bool) if same_location is None else np.asarray(same_location, dtype=bool)
            E = np.zeros((n, ldn))
            E[:, : n * d] = (same[:, :, None] * ng[None, :, :]).reshape(n, n * d)
            check(lib.gpx_axpby(dev.h, n * ldn, 1.0, ptr(dev.upload(E)), 1.0, ptr(dct), dev.stream), "gpx_axpby")
            diag = dev.upload(ng.reshape(n * d))
        qneg = dev.zeros(max(n * d, 1), X.ld)
        check(lib.gpx_dgemm_tn_sub(dev.h, ptr(dct), ldn, ptr(W), X.ld, ptr(qneg), X.ld, n * d, X.n, n, 0, dev.stream),
              "gpx_dgemm_tn_sub")
        out = dev.zeros(max(n * d, 1), X.ld)
        check(lib.gpx_se_var_grad(dev.h, ptr(D.X), n, D.ld, ptr(X.X), X.n, X.ld, ptr(W), ptr(qneg), ptr(diag), ptr(out),
                                  dev.stream), "gpx_se_var_grad")
        return out

    def precision_device(self):
        """(U^T U)^-1 as a dense n x roundup(n) device matrix: U^-1 (U^-T I)."""
        dev, n = self.dev, self.n
        ld = roundup(n)
        Y = dev.zeros(max(n, 1), ld)
        check(lib.gpx_trtri_t(dev.h, ptr(self.U), n, self.ldu, ptr(Y), ld, dev.stream), "gpx_trtri_t")
        check(lib.gpx_trsm_back(dev.h, ptr(self.Ut()), n, self.ldu, ptr(Y), n, ld, dev.stream), "gpx_trsm_back")
        return Y

    def precision(self) -> np.ndarray:
        return self.precision_device()[: self.n, : self.n].cpu().numpy()

    def loglike_gradient(self, y: np.ndarray) -> np.ndarray:
        """1/2 tr((alpha alpha^T - P) dK/dtheta) for theta = cl_0..cl_{d-1}, signalSize, noise (bare trace for the
        noise entry), squared-exponential kernels (gp.py:447-468)."""
        dev, D, n = self.dev, self.design, self.n
        P = self.precision_device()
        alpha = dev.upload(self.solve_vector(y))
        ws = dev.zeros(max(int(lib.gpx_se_loglike_grad_workspace(n, D.d)), 1))
        out = dev.zeros(D.d + 2)
        check(lib.gpx_se_loglike_grad(dev.h, ptr(D.X), n, D.ld, ptr(P), P.shape[1], ptr(alpha), ptr(ws), ptr(out), dev.stream),
              "gpx_se_loglike_grad")
        return out.cpu().numpy()


class FitcFactor:
    """FITC sparse-GP covariance and precision of a design (gp_kernel_utilities.py:70-104, gp.py:182-208), all on the
    device:  Q = K_fu K_uu^-1 K_uf,  G = diag(K_ff + noise - Q),  cov = Q + G,
             precision = G^-1 - G^-1 K_fu (K_uu + K_uf G^-1 K_fu)^-1 K_uf G^-1      (Woodbury).
    The reference pseudo-inverts K_uu and inverts the inner matrix; here both are Cholesky factors (K_uu carries the
    noise on its diagonal, gp.py:193)."""

    def __init__(self, dev: Device, design: PointSet, inducing: PointSet, noise: float):
        self.dev, self.design, self.inducing = dev, design, inducing
        n, nu, st = design.n, inducing.n, dev.stream
        self.n = n
        ld = design.ld
        self.ld = ld
        uu = DesignFactor(dev, inducing, float(noise))          # K_uu + noise I = U_u^T U_u
        if uu.jitter:
            warnings.warn("FITC: inducing-point Gram was jittered", GpxConditionWarning, stacklevel=3)
        # A = U_u^-T K_uf   (nu x n): Q = A^T A, diag(Q) = column sums of squares
        A = dev.zeros(max(nu, 1), ld)
        check(lib.gpx_gram(dev.h, ptr(inducing.X), nu, inducing.ld, ptr(design.X), n, ld, ptr(A), ld, 0, None, 0.0, st), "gpx_gram")
        Kuf = A.clone()
        check(lib.gpx_trsm(dev.h, ptr(uu.U), nu, uu.ldu, ptr(A), n, ld, st), "gpx_trsm")
        g = dev.zeros(ld)
        check(lib.gpx_prior_diag(dev.h, ptr(design.X), n, ld, ptr(g), st), "gpx_prior_diag")
        check(lib.gpx_colsumsq(dev.h, ptr(A), nu, n, ld, ptr(g), ptr(g), st), "gpx_colsumsq")     # k(x,x) - Q_ii
        gh = g[:n].cpu().numpy() + float(noise)                                                  # + noise (gp.py:203-204)
        g = dev.upload(np.concatenate([gh, np.ones(ld - n)]))
        ginv = dev.upload(np.concatenate([1.0 / (gh + 1e-12), np.zeros(ld - n)]))                # gp.py:207
        # cov = Q + G = A^T A + diag(g)
        cov = dev.zeros(max(n, 1), ld)
        check(lib.gpx_dgemm_tn_sub(dev.h, ptr(A), ld, ptr(A), ld, ptr(cov), ld, n, n, nu, 0, st), "gpx_dgemm_tn_sub")
        check(lib.gpx_scale_rows_cols(dev.h, ptr(cov), n, n, ld, None, None, -1.0, ptr(cov), ld, st), "gpx_scale_rows_cols")
        check(lib.gpx_diag_update(dev.h, ptr(cov), n, ld, 1.0, ptr(g), 0.0, st), "gpx_diag_update")
        self._cov = cov
        # S = K_uu + K_uf G^-1 K_fu   (nu x nu), contraction index = design points (K-major operands: K_fu rows)
        ldu = inducing.ld
        Kfu = dev.zeros(max(n, 1), ldu)
        check(lib.gpx_gram(dev.h, ptr(design.X), n, ld, ptr(inducing.X), nu, ldu, ptr(Kfu), ldu, 0, None, 0.0, st), "gpx_gram")
        Kfu_s = dev.zeros(max(n, 1), ldu)
        check(lib.gpx_scale_rows_cols(dev.h, ptr(Kfu), n, nu, ldu, ptr(ginv), None, -1.0, ptr(Kfu_s), ldu, st), "gpx_scale_rows_cols")
        S = uu._cov.clone()
        check(lib.gpx_dgemm_tn_sub(dev.h, ptr(Kfu_s), ldu, ptr(Kfu), ldu, ptr(S), uu.ldu, nu, nu, n, 0, st), "gpx_dgemm_tn_sub")
        info = dev.zeros(1, dtype=torch.int32)
        check(lib.gpx_potrf(dev.h, ptr(S), nu, uu.ldu, ptr(info), st), "gpx_potrf")
        if int(info.item()):
            raise GpxError(f"FITC: inner Woodbury matrix is not positive definite (pivot {int(info.item()) - 1})")
        # T = U_s^-T (K_uf G^-1)  ;  precision = G^-1 - T^T T
        T = dev.zeros(max(nu, 1), ld)
        check(lib.gpx_scale_rows_cols(dev.h, ptr(Kuf), nu, n, ld, None, ptr(ginv), 1.0, ptr(T), ld, st), "gpx_scale_rows_cols")
        check(lib.gpx_trsm(dev.h, ptr(S), nu, uu.ldu, ptr(T), n, ld, st), "gpx_trsm")
        P = dev.zeros(max(n, 1), ld)
        check(lib.gpx_diag_update(dev.h, ptr(P), n, ld, 0.0, ptr(ginv), 0.0, st), "gpx_diag_update")
        check(lib.gpx_dgemm_tn_sub(dev.h, ptr(T), ld, ptr(T), ld, ptr(P), ld, n, n, nu, 0, st), "gpx_dgemm_tn_sub")
        self.P = P
        self.jitter = 0.0

    def covariance(self) -> np.ndarray:
        return self._cov[: self.n, : self.n].cpu().numpy()

    def precision(self) -> np.ndarray:
        return self.P[: self.n, : self.n].cpu().numpy()

    def cross_gram(self, X: PointSet):
        dev, D = self.dev, self.design
        Kx = dev.zeros(max(self.n, 1), X.ld)
        check(lib.gpx_gram(dev.h, ptr(D.X), self.n, D.ld, ptr(X.X), X.n, X.ld, ptr(Kx), X.ld, 0, None, 0.0, dev.stream), "gpx_gram")
        return Kx

    def apply_precision(self, B, ncols: int, ldb: int):
        """Z = P B for a device matrix B (n x ldb); P is symmetric, so it is its own K-major operand."""
        dev = self.dev
        Z = dev.zeros(max(self.n, 1), ldb)
        check(lib.gpx_dgemm_tn_sub(dev.h, ptr(self.P), self.ld, ptr(B), ldb, ptr(Z), ldb, self.n, ncols, self.n, 0, dev.stream),
              "gpx_dgemm_tn_sub")
        check(lib.gpx_scale_rows_cols(dev.h, ptr(Z), self.n, ncols, ldb, None, None, -1.0, ptr(Z), ldb, dev.stream),
              "gpx_scale_rows_cols")
        return Z

    def solve_gram(self, X: PointSet, W=None, want_var=True):
        """(K(D,X), var) with var = k(x,x) - k^T P k  (gp.py:246-256 with the FITC precision)."""
        dev = self.dev
        Kx = self.cross_gram(X)
        var = None
        if want_var:
            Z = self.apply_precision(Kx, X.n, X.ld)
            var = dev.zeros(X.ld)
            check(lib.gpx_prior_diag(dev.h, ptr(X.X), X.n, X.ld, ptr(var), dev.stream), "gpx_prior_diag")
            check(lib.gpx_coldot(dev.h, ptr(Kx), ptr(Z), self.n, X.n, X.ld, ptr(var), ptr(var), dev.stream), "gpx_coldot")
        return Kx, var

    def solve_vector(self, y: np.ndarray) -> np.ndarray:
        """P y  (GP.train coefficients, gp.py:101)."""
        dev = self.dev
        B = dev.zeros(max(self.n, 1), 2)
        B[: self.n, 0] = dev.upload(np.asarray(y, dtype=np.float64))
        return self.apply_precision(B, 1, 2)[: self.n, 0].cpu().numpy()

    def logdet(self) -> float:
        """log det(Q + G) through a Cholesky factor of the dense FITC covariance (np.linalg.slogdet, gp.py:432)."""
        dev, n = self.dev, self.n
        C = self._cov.clone()
        info = dev.zeros(1, dtype=torch.int32)
        check(lib.gpx_potrf(dev.h, ptr(C), n, self.ld, ptr(info), dev.stream), "gpx_potrf")
        if int(info.item()):
            raise GpxError("FITC covariance is not positive definite")
        out = dev.zeros(1)
        check(lib.gpx_logdet_chol(dev.h, ptr(C), n, self.ld, ptr(out), dev.stream), "gpx_logdet_chol")
        return float(out.item())

    def quad_form(self, y: np.ndarray) -> float:
        return float(np.dot(np.asarray(y, dtype=np.float64), self.solve_vector(y)))


class GreedyIVAREngine(_Pivoting):
    """Discrete greedy IVAR (SURVEY.md 3.2 / 8c): every step scores all candidates with the FP64 DMMA
    contraction (K5), takes the arg-min, and appends one row to W_C and W_M."""

    # resident problems up to this many (integration point, candidate) pairs run their whole loop as ONE cooperative
    # kernel (gpx_ivar_greedy_small): 256 MB of covariance, roughly what stays close to the 126 MB L2.
    # GPX_ONE_KERNEL_PAIRS overrides (0 = always the multi-launch loop).
    ONE_KERNEL_DEFAULT = 32_000_000
    ONE_KERNEL_PAIRS = int(os.environ.get("GPX_ONE_KERNEL_PAIRS", ONE_KERNEL_DEFAULT))

    def __init__(self, dev: Device, cand: PointSet, mc: PointSet, n_max: int, noise: float, zero_scale: float,
                 shard=None, index_offset: int = 0, resident: bool = False, cand_noise=None):
        """resident=True keeps the posterior covariance cov_D(m, c) (8*M*C bytes) in HBM and replaces the per-step
        O(M n C) contraction by one rank-1 update pass (16*M*C bytes of traffic per step, independent of n) -- the
        better algorithm for a greedy LOOP whenever the matrix fits; scoring a GIVEN design still takes the contraction.

        cand_noise: host vector nu of a heteroscedastic noise function at the local candidates (noise must be 0.0 then).
        The candidate running variance is then kept noise-inclusive, varC[c] = var_D(c) + nu(c): every kernel sees the
        noise only as varC + noise, the append's (var + nu) - w^2 is the same update, and the pivot var_D(p) + nu(p)
        makes U the factor of K_DD + diag(nu(D)).  Integration points carry no noise."""
        self.cand, self.mc = cand, mc
        self.resident = bool(resident)
        self.noise = float(noise)
        self.cand_noise = None
        if cand_noise is not None:
            nu = np.asarray(cand_noise, dtype=np.float64).ravel()
            if self.noise != 0.0:
                raise ValueError("cand_noise replaces the scalar noise: pass noise=0.0 with it")
            if nu.size != cand.n:
                raise ValueError(f"cand_noise has {nu.size} values for {cand.n} candidates")
            self.cand_noise = dev.upload(nu)
        self.zero_tol = ZERO_VAR_TOL * float(zero_scale)
        ncap = max(int(n_max), 1)
        self._init_pivot(dev, ncap, n_max, shard, index_offset)
        self.Wc = dev.zeros(ncap, cand.ld)
        self.Wm = dev.zeros(ncap, mc.ld)
        self.varC = dev.zeros(cand.ld)
        self.varM = dev.zeros(mc.ld)
        self.U = dev.zeros(ncap, roundup(ncap))
        check(lib.gpx_prior_diag(dev.h, ptr(cand.X), cand.n, cand.ld, ptr(self.varC), dev.stream), "gpx_prior_diag")
        self._add_cand_noise()
        check(lib.gpx_prior_diag(dev.h, ptr(mc.X), mc.n, mc.ld, ptr(self.varM), dev.stream), "gpx_prior_diag")
        self.nseg = int(lib.gpx_cov_segments(mc.n, cand.n))
        self.ldp = (cand.n + 1) & ~1
        # partial column sums: M-splits of the contraction, or row segments of the resident update
        ws = max(int(lib.gpx_score_ivar_workspace(dev.h, mc.n, cand.n)), self.nseg * self.ldp)
        self.workspace = dev.zeros(max(ws, 1))
        if not self.resident and ncap <= _lib.GPX_I8_MAX_N:  # only the contraction of the INT8 core reads it
            dev.reserve_ivar_scratch(mc.n, cand.n, ncap)
        self.scores = dev.zeros(cand.ld)
        self.score_trace = None
        self.cov = None
        self.zero_scale = float(zero_scale)
        if self.resident:
            self.cov = dev.empty(mc.n, cand.ld)
            # cov_0 = K(mc, cand), then the column sums of squares for the first scoring
            check(lib.gpx_gram(dev.h, ptr(mc.X), mc.n, mc.ld, ptr(cand.X), cand.n, cand.ld, ptr(self.cov), cand.ld, 0, None,
                               0.0, dev.stream), "gpx_gram")
            self._cov_pass(None, None)

    def _local_count(self):
        return self.cand.n

    def _add_cand_noise(self):
        """varC += nu: called wherever varC is (re)built from the prior or from a factor."""
        if self.cand_noise is not None:
            check(lib.gpx_axpby(self.dev.h, self.cand.n, 1.0, ptr(self.cand_noise), 1.0, ptr(self.varC), self.dev.stream),
                  "gpx_axpby")

    def _cov_pass(self, a, b):
        dev, cand, mc = self.dev, self.cand, self.mc
        check(lib.gpx_cov_update(dev.h, ptr(self.cov), cand.ld, mc.n, cand.n, ptr(a), ptr(b), ptr(self.workspace), self.ldp,
                                 dev.stream), "gpx_cov_update")

    def prologue(self):
        """(mode, rows of the integration points, rows of the candidates) for the contraction's covariance prologue.
        The centre of the expanded form is the mid-range of the integration points."""
        self.dev.set_center(self.mc.midrange())
        return prologue_operands(self.mc, self.cand)

    def score(self, contraction: bool = False):
        """Score every candidate and arg-min.  contraction=True forces the DMMA contraction even in resident mode
        (cross-check of the two paths on the same state)."""
        dev, cand, mc = self.dev, self.cand, self.mc
        if self.resident and not contraction:
            check(lib.gpx_score_ivar_partials(dev.h, ptr(self.workspace), self.nseg, self.ldp, ptr(self.varM), mc.n,
                                              ptr(self.varC), cand.n, self.noise, self.zero_tol, None, ptr(self.scores),
                                              ptr(self.best), ptr(self.idx), dev.stream), "gpx_score_ivar_partials")
            return
        mode, ma_rows, cb_rows = self.prologue()
        ws = self.workspace
        if self.resident:  # keep the resident column sums intact: the contraction gets its own scratch
            if getattr(self, "_ws2", None) is None:
                self._ws2 = dev.zeros(self.workspace.numel())
            ws = self._ws2
        check(lib.gpx_score_ivar(dev.h, mode, ptr(self.Wm), mc.ld, ptr(self.varM), ptr(ma_rows), mc.n, ptr(self.Wc), cand.ld,
                                 ptr(self.varC), ptr(cb_rows), cand.n, self.n, self.noise, self.zero_tol, None, ptr(ws),
                                 ptr(self.scores), ptr(self.best), ptr(self.idx), dev.stream), "gpx_score_ivar")

    def append(self):
        dev, cand, mc = self.dev, self.cand, self.mc
        self._gather(self.Wc, cand.ld, self.varC, cand, self.noise, minimize=True)
        check(lib.gpx_append_row(dev.h, _lib.ROW_KERNEL, ptr(self.rec_win), None, ptr(cand.X), cand.n, cand.ld,
                                 ptr(self.Wc), cand.ld, self.n, ptr(self.varC), dev.stream), "gpx_append_row")
        check(lib.gpx_append_row(dev.h, _lib.ROW_KERNEL, ptr(self.rec_win), None, ptr(mc.X), mc.n, mc.ld,
                                 ptr(self.Wm), mc.ld, self.n, ptr(self.varM), dev.stream), "gpx_append_row")
        self._record(self.U, self.U.shape[1])
        if self.resident:
            # cov -= w_M[n] w_C[n]^T and the next step's column sums of squares, one pass over the resident matrix
            self._cov_pass(self.Wm[self.n], self.Wc[self.n])
        self.n += 1

    def force(self, global_index: int):
        self._force_local(int(global_index))
        self.append()

    def snapshot(self):
        """Cheap save point (running variances + design size); rows >= n of W are never read.
        Not available in resident mode (the covariance matrix is updated in place)."""
        assert not self.resident, "resident mode cannot be rolled back"
        return (self.n, self.varC.clone(), self.varM.clone())

    def restore(self, snap):
        self.n = snap[0]
        self.varC.copy_(snap[1])
        self.varM.copy_(snap[2])

    def rollback(self, n_keep: int):
        """Forget the rows appended after n_keep (bench.py re-times the same step)."""
        assert 0 <= n_keep <= self.n
        if n_keep == self.n:
            return
        dev, cand, mc = self.dev, self.cand, self.mc
        self.Wc[n_keep: self.n].zero_()
        self.Wm[n_keep: self.n].zero_()
        self.n = n_keep
        prior = dev.zeros(cand.ld)
        check(lib.gpx_prior_diag(dev.h, ptr(cand.X), cand.n, cand.ld, ptr(prior), dev.stream), "gpx_prior_diag")
        check(lib.gpx_colsumsq(dev.h, ptr(self.Wc), self.n, cand.n, cand.ld, ptr(prior), ptr(self.varC), dev.stream), "colsumsq")
        self._add_cand_noise()
        prior = dev.zeros(mc.ld)
        check(lib.gpx_prior_diag(dev.h, ptr(mc.X), mc.n, mc.ld, ptr(prior), dev.stream), "gpx_prior_diag")
        check(lib.gpx_colsumsq(dev.h, ptr(self.Wm), self.n, mc.n, mc.ld, ptr(prior), ptr(self.varM), dev.stream), "colsumsq")

    def load_design(self, factor: DesignFactor):
        """State for a GIVEN design (not grown greedily): W_C, W_M via the fused Gram+TRSM, var via K4."""
        assert factor.n <= self.ncap
        self.n = factor.n
        _, vC = factor.solve_gram(self.cand, W=self.Wc)
        _, vM = factor.solve_gram(self.mc, W=self.Wm)
        self.varC.copy_(vC)
        self._add_cand_noise()
        self.varM.copy_(vM)
        if self.resident:
            dev, cand, mc = self.dev, self.cand, self.mc
            mode, ma_rows, cb_rows = self.prologue()
            check(lib.gpx_cov_from_factors(dev.h, mode, ptr(self.Wm), mc.ld, ptr(ma_rows), mc.n, ptr(self.Wc), cand.ld,
                                           ptr(cb_rows), cand.n, self.n, ptr(self.cov), cand.ld, dev.stream),
                  "gpx_cov_from_factors")
            self._cov_pass(None, None)

    def step(self):
        self.score()
        if self.score_trace is not None:
            self.score_trace.append(self.scores[: self.cand.n].cpu().numpy().copy())
        self.append()

    def _state(self):
        st = _lib.IvarState()
        cand, mc = self.cand, self.mc
        mode, ma_rows, cb_rows = (_lib.PRO_DIFF, mc.X, cand.X) if self.resident else self.prologue()
        self._state_keep = (ma_rows, cb_rows)
        st.Xm, st.M, st.ldm, st.Wm, st.varM, st.Ma_rows = ptr(mc.X), mc.n, mc.ld, ptr(self.Wm), ptr(self.varM), ptr(ma_rows)
        st.Xc, st.C, st.ldc, st.Wc, st.varC, st.Cb_rows = ptr(cand.X), cand.n, cand.ld, ptr(self.Wc), ptr(self.varC), ptr(cb_rows)
        st.ncap, st.index_offset, st.prologue, st.nseg = self.ncap, self.index_offset, mode, self.nseg
        st.noise, st.zero_tol = self.noise, self.zero_tol
        st.workspace, st.scores, st.best, st.idx = ptr(self.workspace), ptr(self.scores), ptr(self.best), ptr(self.idx)
        st.rec, st.rec_all = ptr(self.rec), ptr(self.rec_all)
        st.rec_win = ptr(self.rec_win) if self.rec_all is not None else None
        st.U, st.ldu = ptr(self.U), self.U.shape[1]
        st.picks, st.pick_scores, st.pick_pivots = ptr(self.picks), ptr(self.pick_scores), ptr(self.pick_pivots)
        st.cov, st.ldcov, st.ldp = ptr(self.cov), cand.ld, self.ldp
        return st

    def run(self, n_points: int, progress=None, chunk: int = 10):
        """Grow the design to n_points: the whole loop is issued by gpx_ivar_greedy_run (one C call, no host round trip
        per step) unless per-step score vectors are being traced."""
        if self.score_trace is not None or not self._native_ready():
            while self.n < n_points:
                if progress is not None:
                    progress(self.n)
                self.step()
            return self.indices()
        st = self._state()
        # small resident problems on one GPU: the whole loop as one cooperative kernel (no per-launch issue cost)
        one_kernel = (self.resident and (self.shard is None or self.shard.world == 1) and n_points <= 1024 and
                      self.mc.n * self.cand.n <= self.ONE_KERNEL_PAIRS)
        run = lib.gpx_ivar_greedy_small if one_kernel else lib.gpx_ivar_greedy_run
        while self.n < n_points:
            if progress is not None:
                progress(self.n)
            stop = min(n_points, (self.n // chunk + 1) * chunk) if progress is not None else n_points
            check(run(self.dev.h, C.byref(st), self.n, stop, self.dev.stream), "gpx_ivar_greedy_run")
            self.n = stop
        return self.indices()


class GreedyMIEngine(_Pivoting):
    """Greedy mutual information (experimentalDesign.py:753-785 with :252-285 restated):
    numerator = running posterior variance given A (nugget = noise); denominator from the diagonal of
    the precision of V minus A, kept current by lazy rank-1 downdates."""

    def __init__(self, dev: Device, pool: PointSet, n_max: int, noise: float):
        self.pool = pool
        self.noise = float(noise)
        ncap = max(int(n_max), 1)
        self._init_pivot(dev, ncap, n_max, None, 0)
        v, ld = pool.n, pool.ld
        self.W = dev.zeros(ncap, ld)          # numerator factor rows
        self.num = dev.zeros(ld)
        check(lib.gpx_prior_diag(dev.h, ptr(pool.X), v, ld, ptr(self.num), dev.stream), "gpx_prior_diag")
        # set-up: K_VV + noise I = U^T U ; Y = U^-T ; pd = diag(P) = colsumsq(Y)
        K = dev.zeros(v, ld)
        info = dev.zeros(1, dtype=torch.int32)
        check(lib.gpx_gram(dev.h, ptr(pool.X), v, ld, ptr(pool.X), v, ld, ptr(K), ld, 1, None, self.noise, dev.stream), "gpx_gram")
        self.cov = K.clone()
        check(lib.gpx_potrf(dev.h, ptr(K), v, ld, ptr(info), dev.stream), "gpx_potrf")
        self.U = K
        self.Y = dev.zeros(v, ld)
        check(lib.gpx_trtri_t(dev.h, ptr(K), v, ld, ptr(self.Y), ld, dev.stream), "gpx_trtri_t")
        self.pd = dev.zeros(ld)
        check(lib.gpx_colsumsq(dev.h, ptr(self.Y), v, v, ld, None, ptr(self.pd), dev.stream), "gpx_colsumsq")
        self.info = info
        self.Us = dev.zeros(ncap, ld)         # downdate vectors u_s
        self.pcol = dev.zeros(ld)
        self.pws = dev.zeros(max(int(lib.gpx_mi_prec_column_workspace(v, ld)), 1))
        self.rec2 = dev.zeros(self.reclen)
        self.mask = dev.zeros(ld, dtype=torch.uint8)
        self.scores = dev.zeros(ld)
        self.score_trace = None

    def _local_count(self):
        return self.pool.n

    def take(self):
        """Move the point in self.idx from S = V minus A into A."""
        dev, pool = self.dev, self.pool
        v, ld = pool.n, pool.ld
        self._gather(self.W, ld, self.num, pool, self.noise, minimize=False)
        check(lib.gpx_append_row(dev.h, _lib.ROW_KERNEL, ptr(self.rec), None, ptr(pool.X), v, ld, ptr(self.W), ld, self.n,
                                 ptr(self.num), dev.stream), "gpx_append_row")
        check(lib.gpx_mi_prec_column(dev.h, ptr(self.Y), v, v, ld, 0, 0, 1, ptr(self.idx), None, ptr(self.pws), ptr(self.pcol),
                                     dev.stream), "gpx_mi_prec_column")
        check(lib.gpx_gather_pivot(dev.h, ptr(self.Us), ld, self.n, ptr(self.pd), ptr(pool.X), ld, None, ptr(self.idx), 0, None,
                                   0.0, ptr(self.rec2), dev.stream), "gpx_gather_pivot")
        check(lib.gpx_append_row(dev.h, _lib.ROW_MATRIX, ptr(self.rec2), ptr(self.pcol), None, v, ld, ptr(self.Us), ld, self.n,
                                 ptr(self.pd), dev.stream), "gpx_append_row")
        check(lib.gpx_set_mask(dev.h, ptr(self.mask), ptr(self.idx), 1, dev.stream), "gpx_set_mask")
        self._record()
        self.n += 1

    def force(self, index: int):
        self._force_local(int(index))
        self.take()

    def score(self):
        dev = self.dev
        check(lib.gpx_score_mi(dev.h, ptr(self.num), ptr(self.pd), self.noise, ptr(self.mask), self.pool.n, ptr(self.scores),
                               ptr(self.best), ptr(self.idx), dev.stream), "gpx_score_mi")

    def step(self):
        self.score()
        if self.score_trace is not None:
            self.score_trace.append(self.scores[: self.pool.n].cpu().numpy().copy())
        self.take()

    def run(self, n_points: int, start: int = 0):
        if self.n == 0:
            self.force(start)
        while self.n < n_points:
            self.step()
        return self.indices()


class ShardedMIEngine(_Pivoting):
    """Greedy mutual information with the |V| x |V| matrices sharded by COLUMN BLOCKS over the ranks
    (cfg-4 at full size: 200 000^2 doubles do not fit one GPU).

    Distribution: block-cyclic -- global column block g (BLK columns) lives on rank g % world as its local block g // world,
    so every rank owns the same share of every part of both triangles and each elimination step is balanced.

    Set-up, left-looking in BLK-row blocks, every rank holding its columns of both matrices:
        panel  P = U[0:kb, kb:kb+BLK]                 broadcast from the owner of column block kb / BLK
        U[kb blk, my cols >= kb]    = U_kk^-T (A[kb blk, .] - P^T U[0:kb, .])     DMMA update + forward substitution
        Y[kb blk, my cols < kb+BLK] = U_kk^-T (I[kb blk, .] - P^T Y[0:kb, .])     (Y = U^-T, lower triangular: the rows of a
                                                                                   column tile above its own global column
                                                                                   are zero and skipped inside the kernel)
    so that K_VV + noise I = U^T U and (K_VV + noise I)^-1 = Y^T Y without any rank ever holding a full matrix.  Executed
    work: V^3/3 (U) + V^3/3 (Y) flop, the useful amount.
    Per greedy step: one all_gather of numerator pivot records, one all_reduce that carries column p of Y (and of the
    downdate vectors) from its owner to everybody, then purely local kernels.
    """

    # columns per distribution block = rows per elimination block (GPX_MI_BLK overrides; power of two >= 256).
    # 2 GPUs, |V| = 80 000: 512 -> 5.81 s, 1024 -> 5.64 s (round 1, contiguous ranges, no zero skipping: 10.65 s)
    BLK = 1024

    def __init__(self, dev: Device, pool_host: np.ndarray, n_max: int, noise: float, shard=None):
        import os
        self.BLK = int(os.environ.get("GPX_MI_BLK", self.BLK))
        if self.BLK < 256 or self.BLK & (self.BLK - 1):
            # tiles of the TMA update kernel (128 columns) and of the precision-column kernel (256) must not straddle blocks
            raise ValueError(f"GPX_MI_BLK must be a power of two >= 256, got {self.BLK}")
        import torch.distributed as dist
        self.dist = dist
        self.noise = float(noise)
        world = shard.world if shard is not None else 1
        rank = shard.rank if shard is not None else 0
        self.world, self.rank = world, rank
        V = pool_host.shape[0]
        self.V = V
        # keep a few elimination blocks per rank on small pools
        while self.BLK > 256 and (V + self.BLK - 1) // self.BLK < 4 * world:
            self.BLK //= 2
        B = self.BLK
        nblk = (V + B - 1) // B
        gcols = self.cyclic_columns(V, B, world, rank)
        self.gcols = gcols                                           # global column of every local column
        nloc = int(gcols.size)
        self.nloc = nloc
        self.ncols_per_rank = [sum(min((g + 1) * B, V) - g * B for g in range(r, nblk, world)) for r in range(world)]
        ncap = max(int(n_max), 1)
        self._init_pivot(dev, ncap, n_max, shard, 0)
        self.pool = dev.points(pool_host[gcols]) if nloc else dev.points(pool_host[:0])
        allpts = dev.points(pool_host)
        ld = self.pool.ld
        self.ld = ld
        self.index_map = dev.upload(self.gcols, dtype=torch.int64) if nloc else dev.zeros(1, dtype=torch.int64)
        st = dev.stream
        # ---- local columns of K_VV + noise I and of the identity (all V rows: only rows <= column are read)
        A = dev.zeros(V, ld)
        Y = dev.zeros(V, ld)
        if nloc > 0:
            check(lib.gpx_gram(dev.h, ptr(allpts.X), V, allpts.ld, ptr(self.pool.X), nloc, ld, ptr(A), ld, 0, None, 0.0, st), "gpx_gram")
            check(lib.gpx_add_at_rows(dev.h, ptr(A), ld, ptr(self.index_map), nloc, self.noise, st), "gpx_add_at_rows")
            check(lib.gpx_add_at_rows(dev.h, ptr(Y), ld, ptr(self.index_map), nloc, 1.0, st), "gpx_add_at_rows")
        del allpts
        panel = dev.zeros(V, B)
        diag = dev.zeros(B, B)  # the factored diagonal block travels as a dense BLK x BLK matrix
        info = dev.zeros(1, dtype=torch.int32)
        bad = dev.zeros(1, dtype=torch.int32)
        group = shard.group if shard is not None else None

        def first_local_block_at_or_after(g):  # smallest local block j with global block rank + j*world >= g
            return max(0, -(-(g - rank) // world))

        for g in range(nblk):
            kb = g * B
            b = min(B, V - kb)
            owner = g % world
            own = rank == owner
            jl = g // world                     # local block index on the owner
            if kb > 0:
                if own:
                    panel[:kb, :b].copy_(A[:kb, jl * B: jl * B + b])
                if world > 1:
                    dist.broadcast(panel[:kb], src=owner, group=group)
                # U: my columns in global blocks >= g (a suffix of the local columns)
                cu = min(first_local_block_at_or_after(g) * B, nloc)
                if nloc - cu > 0:
                    # panel, A and Y are allocated in whole 128-wide tiles: the TMA update kernel may read full tiles
                    check(lib.gpx_dgemm_tn_sub_padded(dev.h, ptr(panel), B, ptr(A) + 8 * cu, ld, ptr(A) + 8 * (kb * ld + cu), ld,
                                                      b, nloc - cu, kb, 0, st), "gpx_dgemm_tn_sub_padded")
                # Y: my columns in global blocks <= g (a prefix); rows above each tile's own column are skipped in-kernel
                ny = min(first_local_block_at_or_after(g + 1) * B, nloc)
                if ny > 0:
                    check(lib.gpx_dgemm_tn_sub_lower(dev.h, ptr(panel), B, ptr(Y), ld, ptr(Y) + 8 * kb * ld, ld, b, ny, kb, B,
                                                     world, rank, st), "gpx_dgemm_tn_sub_lower")
            if own:
                check(lib.gpx_potrf(dev.h, ptr(A) + 8 * (kb * ld + jl * B), b, ld, ptr(info), st), "gpx_potrf")
                bad.copy_(torch.maximum(bad, torch.where(info > 0, info + kb, info)))
                diag[:b, :b].copy_(A[kb: kb + b, jl * B: jl * B + b])
            if world > 1:
                dist.broadcast(diag, src=owner, group=group)
            cs = min(first_local_block_at_or_after(g + 1) * B, nloc)   # my columns in global blocks > g
            if nloc - cs > 0:
                check(lib.gpx_trsm(dev.h, ptr(diag), b, B, ptr(A) + 8 * (kb * ld + cs), nloc - cs, ld, st), "gpx_trsm")
            ny = cs                                                      # ... and in global blocks <= g
            if ny > 0:
                check(lib.gpx_trsm(dev.h, ptr(diag), b, B, ptr(Y) + 8 * kb * ld, ny, ld, st), "gpx_trsm")
        if world > 1:
            dist.all_reduce(bad, op=dist.ReduceOp.MAX, group=group)
        self.info = bad
        self.Y = Y
        del A, panel
        self._init_greedy(n_max)

    @staticmethod
    def cyclic_columns(V: int, B: int, world: int, rank: int) -> np.ndarray:
        """Global columns owned by `rank`, in local order: blocks rank, rank + world, ... of B columns."""
        blocks = range(rank, (V + B - 1) // B, world)
        parts = [np.arange(g * B, min((g + 1) * B, V), dtype=np.int64) for g in blocks]
        return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)

    @staticmethod
    def cyclic_local(g: int, V: int, B: int, world: int, rank: int) -> int:
        if not (0 <= g < V) or (g // B) % world != rank:
            return -1
        return ((g // B) // world) * B + g % B

    def _init_greedy(self, n_max: int):
        """(Re)start the greedy state on the factorisation already held: nothing chosen, denominators from diag(Y^T Y)."""
        dev, ld, V = self.dev, self.ld, self.V
        nloc = self.nloc
        st = dev.stream
        ncap = max(int(n_max), 1)
        self._init_pivot(dev, ncap, n_max, self.shard, 0)
        self.pd = dev.zeros(ld)
        if nloc > 0:
            check(lib.gpx_colsumsq(dev.h, ptr(self.Y), V, nloc, ld, None, ptr(self.pd), st), "gpx_colsumsq")
        self.W = dev.zeros(ncap, ld)
        self.num = dev.zeros(ld)
        check(lib.gpx_prior_diag(dev.h, ptr(self.pool.X), nloc, ld, ptr(self.num), st), "gpx_prior_diag")
        self.Us = dev.zeros(ncap, ld)
        self.pcol = dev.zeros(ld)
        self.pws = dev.zeros(max(int(lib.gpx_mi_prec_column_workspace(V, ld)), 1))
        self.bufY_len = HDR + V
        self.buf = dev.zeros(self.bufY_len + HDR + ncap)
        self.loc2 = dev.zeros(2, dtype=torch.int64)
        self.mask = dev.zeros(ld, dtype=torch.uint8)
        self.scores = dev.zeros(ld)
        self.score_trace = None

    def reset(self, n_max: int):
        """Forget the chosen points but keep the O(|V|^3) factorisation (costFunctionGP_MI.evaluate is called once per
        candidate with a growing `indexAdded`, experimentalDesign.py:776-777)."""
        self._init_greedy(n_max)

    def _local_count(self):
        return self.nloc

    def _local_of(self, global_index: int) -> int:
        return self.cyclic_local(int(global_index), self.V, self.BLK, self.world, self.rank)

    def global_scores(self) -> np.ndarray:
        """This rank's scores scattered to global candidate positions (NaN where another rank owns the candidate)."""
        out = np.full(self.V, np.nan)
        out[self.gcols] = self.scores[: self.nloc].cpu().numpy()
        return out

    def score(self):
        dev = self.dev
        nloc = self.nloc
        if nloc == 0:  # a rank without columns (more ranks than blocks) only takes part in the exchanges
            self.idx.fill_(-1)
            self.best.zero_()
            return
        check(lib.gpx_score_mi(dev.h, ptr(self.num), ptr(self.pd), self.noise, ptr(self.mask), nloc, ptr(self.scores),
                               ptr(self.best), ptr(self.idx), dev.stream), "gpx_score_mi")

    def take(self):
        dev, pool, ld, V = self.dev, self.pool, self.ld, self.V
        nloc = self.nloc
        st = dev.stream
        self._gather(self.W, ld, self.num, pool, self.noise, minimize=False)
        check(lib.gpx_append_row(dev.h, _lib.ROW_KERNEL, ptr(self.rec_win), None, ptr(pool.X), nloc, ld, ptr(self.W), ld,
                                 self.n, ptr(self.num), st), "gpx_append_row")
        check(lib.gpx_local_index_cyclic(dev.h, ptr(self.rec_win), self.BLK, self.world, self.rank, nloc, ptr(self.loc2), st),
              "gpx_local_index_cyclic")
        self.buf.zero_()
        bufY, bufU = self.buf[: self.bufY_len], self.buf[self.bufY_len:]
        if nloc > 0:
            check(lib.gpx_gather_column(dev.h, ptr(self.Y), ld, V, ptr(self.pd), ptr(self.loc2), ptr(bufY), st),
                  "gpx_gather_column")
            check(lib.gpx_gather_column(dev.h, ptr(self.Us), ld, self.n, ptr(self.pd), ptr(self.loc2), ptr(bufU), st),
                  "gpx_gather_column")
        if self.rec_all is not None:
            self.dist.all_reduce(self.buf, op=self.dist.ReduceOp.SUM, group=self.shard.group)
        if nloc > 0:
            check(lib.gpx_mi_prec_column(dev.h, ptr(self.Y), V, nloc, ld, self.rank, self.BLK, self.world, ptr(self.loc2) + 8,
                                         ptr(bufY) + 8 * HDR, ptr(self.pws), ptr(self.pcol), st), "gpx_mi_prec_column")
            check(lib.gpx_append_row(dev.h, _lib.ROW_MATRIX, ptr(bufU), ptr(self.pcol), None, nloc, ld, ptr(self.Us), ld,
                                     self.n, ptr(self.pd), st), "gpx_append_row")
            check(lib.gpx_set_mask(dev.h, ptr(self.mask), ptr(self.loc2), 1, st), "gpx_set_mask")
        self._record()
        self.n += 1

    def force(self, index: int):
        self._force_local(int(index))
        self.take()

    def step(self):
        self.score()
        if self.score_trace is not None:
            self.score_trace.append(self.global_scores())
        self.take()

    def run(self, n_points: int, start: int = 0):
        if self.n == 0:
            self.force(start)
        while self.n < n_points:
            self.step()
        return self.indices()
