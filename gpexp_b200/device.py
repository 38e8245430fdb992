"""Device-side plumbing: one gpx handle per CUDA device, device buffers (torch tensors used only as
allocations), and thin typed wrappers over the C ABI.  No arithmetic happens in this file."""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from ._lib import GpxError, check, lib

F64 = torch.float64
PAD = 128  # leading dimensions are multiples of the tensor-core tile (also keeps every row 16-byte aligned)


def roundup(n: int, m: int = PAD) -> int:
    return max(m, (int(n) + m - 1) // m * m)


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


# The expanded-form prologue k = f(alpha_i + beta_j + sum u v) loses eps * (max|alpha| + max|beta|) to cancellation
# (relative error of k for the exponential families).  Above this bound the difference form is used instead.
EXPANDED_FORM_TOL = 1e-11
_EPS = float(np.finfo(np.float64).eps)


class PointSet:
    """A set of points resident on the device, dimension-major: X[i, j] = coordinate i of point j."""

    def __init__(self, dev: "Device", X: torch.Tensor, n: int, d: int, lo=None, hi=None):
        self.dev, self.X, self.n, self.d, self.ld = dev, X, n, d, X.shape[1]
        self.lo, self.hi = lo, hi  # per-dimension bounding box (host), for the centre of the expanded form
        self._sides = {}

    def midrange(self):
        if self.lo is None or self.n == 0:
            return np.zeros(max(self.d, 1))
        return 0.5 * (self.lo + self.hi)

    def side(self, which: int):
        """Prepared operand for the GPX_PRO_EXPANDED prologue and its max |alpha| (or |beta|): (rows, maxabs);
        cached per kernel / centre epoch."""
        key = (which, self.dev.kernel_epoch)
        if key not in self._sides:
            rows = torch.empty((_lib.GPX_KROWS, self.ld), dtype=F64, device=self.dev.torch_device)
            mx = torch.zeros((1,), dtype=F64, device=self.dev.torch_device)
            check(lib.gpx_prep_side(self.dev.h, which, ptr(self.X), self.n, self.ld, ptr(rows), self.ld, ptr(mx),
                                    self.dev.stream), "gpx_prep_side")
            self._sides = {k: v for k, v in self._sides.items() if k[1] == self.dev.kernel_epoch}
            self._sides[key] = (rows, float(mx.item()))
        return self._sides[key]


def prologue_operands(a: PointSet, b: PointSet):
    """(mode, rows_a, rows_b) for a contraction whose covariance prologue pairs point set `a` (side A) with `b`
    (side B): the expanded form on the tensor pipe when its cancellation error stays below EXPANDED_FORM_TOL (and the
    d + 2 rows fit a prepared side), else the difference form on the raw coordinates."""
    dev = a.dev
    if a.d + 2 <= _lib.GPX_KROWS and not dev.force_diff_form:
        ra, ma = a.side(_lib.SIDE_A)
        rb, mb = b.side(_lib.SIDE_B)
        if _EPS * (ma + mb) <= EXPANDED_FORM_TOL:
            return _lib.PRO_EXPANDED, ra, rb
    return _lib.PRO_DIFF, a.X, b.X


class Device:
    """Owns the gpx handle of one CUDA device."""

    _instances = {}
    _lock = threading.Lock()

    @classmethod
    def get(cls, index=None) -> "Device":
        if not torch.cuda.is_available():
            raise GpxError("gpexp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if index is None:
            index = torch.cuda.current_device()
        with cls._lock:
            if index not in cls._instances:
                cls._instances[index] = cls(index)
            return cls._instances[index]

    def __init__(self, index: int):
        self.index = index
        self.torch_device = torch.device("cuda", index)
        torch.cuda.set_device(index)
        h = C.c_void_p()
        check(lib.gpx_create(index, C.byref(h)), "gpx_create")
        self.h = h
        self.kernel_epoch = 0
        self._kernel_key = None
        self._center = None
        self.force_diff_form = False  # tests / A-B runs: never use the expanded-form prologue
        self._ivar_scratch = None

    def reserve_ivar_scratch(self, M: int, C: int, n_max: int) -> None:
        """Grow the handle's scratch for the INT8 IVAR core to cover M integration points, C candidates and designs of
        up to n_max points.  The device keeps the buffer for its lifetime, so every engine on the handle can use it."""
        need = int(lib.gpx_ivar_scratch_bytes(self.h, M, C, n_max))
        if self._ivar_scratch is not None and self._ivar_scratch.numel() >= need:
            return
        self._ivar_scratch = torch.empty(need, dtype=torch.uint8, device=self.torch_device)
        check(lib.gpx_set_ivar_scratch(self.h, self._ivar_scratch.data_ptr(), need), "gpx_set_ivar_scratch")

    @property
    def launches(self) -> int:
        """Kernels launched by libgpexp_b200.so so far (counted inside the library, process-wide)."""
        return int(lib.gpx_launch_count())

    # ---- stream / kernel -------------------------------------------------------------------------
    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.torch_device).cuda_stream

    def set_kernel(self, family: int, d: int, params) -> None:
        params = np.ascontiguousarray(params, dtype=np.float64)
        key = (family, d, params.tobytes())
        if key == self._kernel_key:
            return
        check(lib.gpx_set_kernel(self.h, family, d, params.ctypes.data_as(C.POINTER(C.c_double)), params.size),
              "gpx_set_kernel")
        self._kernel_key = key
        self._center = None
        self.kernel_epoch += 1

    def set_center(self, center) -> None:
        """Centre of the expanded-form prologue (stationary kernels): both sides of a contraction are prepared under the
        current centre; changing it invalidates the cached sides."""
        c = np.zeros(_lib.GPX_MAX_DIM)
        center = np.asarray(center, dtype=np.float64).ravel()
        c[: center.size] = center
        if self._center is not None and np.array_equal(c, self._center):
            return
        check(lib.gpx_set_center(self.h, c.ctypes.data_as(C.POINTER(C.c_double))), "gpx_set_center")
        self._center = c
        self.kernel_epoch += 1

    # ---- buffers ---------------------------------------------------------------------------------
    def zeros(self, *shape, dtype=F64) -> torch.Tensor:
        return torch.zeros(shape, dtype=dtype, device=self.torch_device)

    def empty(self, *shape, dtype=F64) -> torch.Tensor:
        return torch.empty(shape, dtype=dtype, device=self.torch_device)

    def upload(self, a: np.ndarray, dtype=F64) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a))
        if t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.torch_device, non_blocking=False)

    def points(self, pts: np.ndarray) -> PointSet:
        """Upload row-major (n, d) host points and lay them out dimension-major on the device."""
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        assert pts.ndim == 2, "points must be an (n, d) array"
        n, d = pts.shape
        if d > _lib.GPX_MAX_DIM:
            raise GpxError(f"dimension {d} exceeds GPX_MAX_DIM={_lib.GPX_MAX_DIM}")
        ld = roundup(n)
        X = self.zeros(max(d, 1), ld)
        lo = hi = None
        if n:
            raw = self.upload(pts)
            check(lib.gpx_transpose(self.h, ptr(raw), n, d, d, ptr(X), ld, self.stream), "gpx_transpose")
            if n * d >= 50_000:
                # the bounding box from the device copy (numpy's axis-0 reduction of an (n, small d) array costs
                # milliseconds at 1e5 points): two row reductions and one 2*d-double read-back
                lo_hi = torch.stack(torch.aminmax(X[:d, :n], dim=1)).cpu().numpy()
                lo, hi = lo_hi[0], lo_hi[1]
            else:
                lo = np.array([pts[:, q].min() for q in range(d)])
                hi = np.array([pts[:, q].max() for q in range(d)])
        return PointSet(self, X, n, d, lo, hi)

    def sync(self) -> None:
        torch.cuda.current_stream(self.torch_device).synchronize()
