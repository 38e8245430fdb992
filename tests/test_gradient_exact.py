"""The squared-exponential gradient layer (gpx_se_dgram, gpx_se_var_grad, gpx_se_loglike_grad, gpx_rowsum) against
exact arithmetic, term by term and at every dimension D = 1 .. 16 of GPX_DISPATCH_DIM.

References are evaluated by mpmath at 50 digits from the same float64 coordinates, At, Qneg, diag, P and alpha the kernel
reads, and by fractions where a sum is exact.  They are pinned to the CPU oracle (and the log-likelihood gradient to
central differences of the log-likelihood) on the CPU, so the formulas in include/gpexp_b200.h are the reference's,
signalSize^2 in the derivative Gram and the bare trace in the noise entry included.

Error bounds (u = 2^-53, eps = 2^-52, DENORM = 2^-1074; A = sum_k a_k (x - y)_k^2 with a_k = cl_k^-2, e = exp(-A/2)):
  dgram     out = -s^2 d_k a_k e, per element:
                |got - ref| <= (C0 + C1(D) A) eps |ref| + 8 DENORM (1 + s |d_k| a_k (1 + s)).
            C1(D) = (D + 6) / 4: the exponent is accumulated from D fma terms of one sign; each term carries the rounding
            of the difference (its square doubles it), of a_k (gpx_set_kernel's host pow, <= 1 ulp) and of the fma,
            i.e. <= (D + 5) u A in all, and exp turns A/2 of that into the same relative error of e.  C0 = 10 covers
            libdevice exp (<= 1 ulp, CUDA Math API; ~2u relative), s e, the three products and the rounding of d_k and
            a_k.  The absolute term is gradual underflow: a subnormal e (A/2 > 708.4) or s e is off by at most a few
            DENORM, and that error is multiplied by what follows it (s, then s |d_k| a_k) -- with s = 2^40 a subnormal e
            still gives a normal result, so the allowance cannot be tied to |ref| alone.
  var_grad  out = 2 At (D - Qneg) - At^2 diag, per element, in terms of the operands and not of |ref| (D - Qneg may
            cancel to nothing):
                |got - ref| <= 2 |At| B_dgram(D) + 4 u (2 |At| (|D| + |Qneg|) + At^2 |diag|) + 4 DENORM
            (one rounding of D - Qneg, one of the product, one of At^2 and one of the final sum, with or without fma).
  loglike   out[q] = 1/2 sum_ij T_ij,q;  T = t k d_q^2 / cl_q^3, t e, t [i = j]  with t = alpha_i alpha_j - P_ij.
            Pair by pair (alpha = 0, one symmetric pair of P): the two terms are bitwise equal and the halving is exact,
            so out[q] is one computed term:  |got - ref| <= (C0 + C1(D) A) eps |ref| + abs (a^(3/2) = a sqrt(a) adds two
            roundings, within C0).  Random cases: with M_ij,q = (|alpha_i alpha_j| + |P_ij|) |dK_ij / dtheta_q| (t itself
            is rounded once, or twice without fma),
                |got - ref| <= 1/2 (sum M (C0 + C1 A) eps + gamma_k 1.01 sum M) + abs,
            gamma_k = k u / (1 - k u), k = 5 + 8 + ceil(nblocks / 256) + 5 + 8: each term is one thread's value, a
            5-level warp butterfly and 8 warp partials in sequence per block, then ceil(nblocks / 256) strided adds, the
            butterfly and the 8 warp partials of grad_reduce_kernel.
  rowsum    integer A, scale 2^-k: every partial sum is an integer below 2^53, so the result is exact.
None of these bounds depends on whether nvcc contracts a*b + c into an fma: both kernel twins (numpy restatements in the
kernels' own operation order, one with a correctly rounded fma and one without) pass the very checkers the GPU tests
use, and twins with one deliberate defect each fail them.  That is the CPU half; the GPU half runs the checkers on the
device at the shapes where the kernels' block indexing has edges (255 / 256 / 257 and ragged last blocks, padding with
sentinels the kernels must not write and NaN where they must not read), then the public entry points end to end against
the CPU oracle with a tolerance per gradient row.  Each checker prints its worst error / bound ratio ("RATIO ...").
"""
import math
from fractions import Fraction

import mpmath
import numpy as np
import pytest

from oracle import gpexp_oracle as orc

mpmath.mp.dps = 50
U_RND = 2.0 ** -53
EPS = 2.0 ** -52
DENORM = 2.0 ** -1074
C0 = 10.0
GPX_OK, GPX_EINVAL = 0, -1
DIMS = list(range(1, 17))
SIGNALS = [2.0 ** -40, 0.3, 1.0, 1.7, 2.0 ** 40]
# A/2 of the value probes: the list of test_covariance_domain.py up to 1e3 (e is subnormal past 708.4, 0 past 745.1)
HALF_EXPONENTS = [0.0, 1e-300, 1e-17, 1e-8, 1.0, 700.0, 707.5, 707.9, 708.2, 708.39, 708.4, 709.0, 745.0, 746.0, 1e3]
TWIN_DIMS = [1, 3, 16]   # the CPU twins are loops over D; these cover the shortest, an odd and the longest


def c1(D):
    return (D + 6) / 4.0


def cls(D):
    """Length-scales 0.55 .. 2.3, none equal to 1 (a defect scaling by cl must show)."""
    return np.array([0.55]) if D == 1 else np.linspace(0.55, 2.3, D)


def a_of(cl):
    return np.array([float(c) ** -2.0 for c in cl])  # pow(cl, -2.0), as gpx_set_kernel computes it


def mpf(x):
    return mpmath.mpf(float(x))


def sentinels(rows, ld):
    return -(1000.0 + np.arange(rows * ld, dtype=np.float64).reshape(rows, ld))


def same_bits(got, want):
    got, want = np.asarray(got, dtype=np.float64) + 0.0, np.asarray(want, dtype=np.float64) + 0.0
    return got.shape == want.shape and np.array_equal(got.view(np.int64), want.view(np.int64))


def edges(n, b=256, extra=3, seed=0):
    """Indices at every block edge (b - 1, b, b + 1, ...), both ends, and a few random ones."""
    s = {0, 1, n - 1, n - 2} | {e for k in range(b, n + 1, b) for e in (k - 1, k, k + 1)}
    s |= set(np.random.default_rng(seed + n).integers(0, n, extra).tolist())
    return sorted(i for i in s if 0 <= i < n)


def note(kernel, D, ratio):
    """The worst error / bound ratio of a check (visible with pytest -s): how much headroom the bound leaves."""
    print(f"RATIO {kernel} D={D} {ratio:.3g}")


# ------------------------------------------------------------------------------------------------
# exact references
# ------------------------------------------------------------------------------------------------
def _mp_pair(x, y, cl):
    dl = [mpf(b) - mpf(a) for a, b in zip(x, y)]
    ai = [1 / mpf(c) ** 2 for c in cl]
    A = mpmath.fsum(ak * dk * dk for ak, dk in zip(ai, dl))
    return dl, ai, A, mpmath.exp(-A / 2)


def mp_dgram(x, y, cl, s):
    """D(y, x)[k] = -s (y - x)_k / cl_k^2 * s e^{-A/2} for all k; also A."""
    dl, ai, A, e = _mp_pair(x, y, cl)
    s = mpf(s)
    return [-s * dk * ak * s * e for dk, ak in zip(dl, ai)], float(A)


def mp_var_grad_entry(p, x, cl, s, at, qneg, diag):
    """2 At (D(x, p)_k - Qneg_k) - At^2 diag_k for every k (diag None: no term); also D(x, p) and A."""
    dk, A = mp_dgram(p, x, cl, s)
    at = mpf(at)
    out = [2 * at * (d - mpf(q)) for d, q in zip(dk, qneg)]
    if diag is not None:
        out = [o - at * at * mpf(g) for o, g in zip(out, diag)]
    return out, dk, A


def mp_loglike_terms(xi, xj, cl, s, t, diagonal):
    """The d + 2 terms (alpha_i alpha_j - P_ij) dK_ij / dtheta_q, theta = cl_0 .. cl_{d-1}, signalSize, noise; also A."""
    dl, _, A, e = _mp_pair(xi, xj, cl)
    s = mpf(s)
    return ([t * s * e * dk * dk / mpf(c) ** 3 for dk, c in zip(dl, cl)] + [t * e, t if diagonal else mpmath.mpf(0)],
            float(A))


def mp_rowsum(row, scale):
    return float(Fraction(float(scale)) * sum(Fraction(float(v)) for v in row))


def dgram_bound(ref_abs, A, s, dfa, D):
    return (C0 + c1(D) * A) * EPS * ref_abs + 8 * DENORM * (1 + s * dfa * (1 + s))


def var_grad_bound(at, dk_abs, q_abs, diag_abs, A, s, dfa, D):
    at = np.abs(at)
    return (2 * at * dgram_bound(dk_abs, A, s, dfa, D) + 4 * U_RND * (2 * at * (dk_abs + q_abs) + at * at * diag_abs)
            + 4 * DENORM)


def ll_abs(t, s, df2, a):
    return 8 * DENORM * (1 + (1 + abs(t)) * (1 + s) * (1 + df2) * (1 + a) ** 2)


# ------------------------------------------------------------------------------------------------
# kernel twins: the kernels' arithmetic in their own operation order, on the host
# ------------------------------------------------------------------------------------------------
def _split(a):
    c = 134217729.0 * a
    hi = c - (c - a)
    return hi, a - hi


def two_product(a, b):
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def fma(x, y, z):
    """Correctly rounded x * y + z, elementwise (Boldo and Melquiond, IEEE TC 57(4), 2008: RN(th + RO(tl + ul))).
    Exact wherever the low part of x * y does not underflow."""
    x, y, z = np.broadcast_arrays(np.asarray(x, np.float64), np.asarray(y, np.float64), np.asarray(z, np.float64))
    with np.errstate(all="ignore"):
        uh, ul = two_product(x, y)
        th, tl = _two_sum(z, uh)
        vh, vl = _two_sum(tl, ul)
        even = (np.atleast_1d(vh).view(np.int64) & 1) == 0
        vh = np.where((vl != 0) & even.reshape(np.shape(vh)), np.nextafter(vh, np.where(vl > 0, np.inf, -np.inf)), vh)
        r = th + vh
        # z + x*y with a non-finite or overflowing operand: the plain expression has the fma's value
        bad = ~np.isfinite(uh) | ~np.isfinite(z) | ~np.isfinite(r)
        return np.where(bad, x * y + z, r)


def madd(x, y, z, use_fma):
    return fma(x, y, z) if use_fma else np.asarray(x) * np.asarray(y) + np.asarray(z)


_EXP = np.frompyfunc(math.exp, 1, 1)


def exp64(x, mut):
    e = np.asarray(_EXP(np.asarray(x, dtype=np.float64)), dtype=np.float64)
    return e + 64 * np.spacing(e) if mut == "exp64" else e


def butterfly(v):
    """Lane 0 of the 5-level __shfl_xor_sync butterfly over the last-but-one axis (32 lanes)."""
    lanes = np.arange(32)
    for off in (16, 8, 4, 2, 1):
        v = v + v[..., lanes ^ off, :]
    return v[..., 0, :]


def block_sum(v):
    """v (..., 256, q): butterfly per warp, then the 8 warp partials added in order from 0."""
    w = butterfly(v.reshape(v.shape[:-2] + (8, 32, v.shape[-1])))
    s = np.zeros(w.shape[:-2] + w.shape[-1:])
    for k in range(8):
        s = s + w[..., k, :]
    return s


class Twin:
    """Host restatement of the four kernels; `fma` picks contracted or separate multiply-adds, `mut` one defect."""

    def __init__(self, use_fma, mut=None):
        self.fma, self.mut = use_fma, mut

    def dgram(self, X, Y, cl, s, ld, out0):
        nx, D = X.shape
        ny = Y.shape[0]
        a = a_of(cl)
        out = out0.copy()
        df = Y[None, :, :] - X[:, None, :]
        acc = np.zeros((nx, ny))
        for q in range(D):
            acc = madd(df[..., q] * df[..., q], a[q], acc, True)    # explicit fma() in the kernel
        kv = s * exp64(-0.5 * acc, self.mut)
        sig = 1.0 if self.mut == "signal_once" else s
        shift = (np.arange(ny) >= 256).astype(int) if self.mut == "colshift" else np.zeros(ny, int)
        for q in range(D):
            v = ((-sig * df[..., q]) * a[q]) * kv
            out[:, np.arange(ny) * D + q + shift] = v
        return out

    def var_grad(self, P, X, cl, s, At, Qneg, diag, out0):
        n, D = P.shape
        M = X.shape[0]
        a = a_of(cl)
        out = out0.copy()
        df = X[None, :, :] - P[:, None, :]
        acc = np.zeros((n, M))
        for q in range(D):
            acc = madd(df[..., q] * df[..., q], a[q], acc, True)
        kv = s * exp64(-0.5 * acc, self.mut)
        at = At[:n, :M]
        a2 = 2.0 * at
        sig = 1.0 if self.mut == "signal_once" else s
        cols = np.arange(M) + ((np.arange(M) >= 256) if self.mut == "colshift" else 0)
        for q in range(D):
            rows = np.arange(n) * D + q
            dk = ((-sig * df[..., q]) * a[q]) * kv
            v = a2 * (dk - Qneg[rows][:, :M])
            if diag is not None:
                sq = at * at if self.mut == "diag_sign" else -at * at
                v = madd(sq, diag[rows][:, None], v, self.fma)
            out[rows[:, None], cols[None, :]] = v
        return out

    def loglike(self, X, P, alpha, cl, s):
        n, D = X.shape
        a = a_of(cl)
        nb = (n + 255) // 256
        t = madd(alpha[:, None], alpha[None, :], -P[:n, :n], self.fma)
        key = (X.tobytes(), a.tobytes())
        if getattr(self, "_geometry", (None,))[0] != key:   # the pair-by-pair runs reuse one X with many P
            acc = np.zeros((n, n))
            df2 = []
            for q in range(D):
                df = X[:, None, q] - X[None, :, q]
                df2.append(df * df)
                acc = madd(df2[q], a[q], acc, True)
            self._geometry = (key, df2, exp64(-0.5 * acc, self.mut))
        _, df2, e = self._geometry
        kv = s * e
        g = np.zeros((n, nb * 256, D + 2))
        for q in range(D):
            g[:, :n, q] = t * kv * df2[q] * a[q] if self.mut == "a_not_a32" else t * kv * df2[q] * a[q] * np.sqrt(a[q])
        g[:, :n, D] = t * kv if self.mut == "e_to_k" else t * e
        g[:, :n, D + 1] = np.where(np.eye(n, dtype=bool), t, 0.0)
        part = block_sum(g.reshape(n, nb, 256, D + 2)).reshape(n * nb, D + 2)   # part[(by * gx + bx) * (D + 2) + q]
        if self.mut == "drop_block":
            part = part[:-1]
        elif self.mut == "double_block":
            part = np.concatenate([part, part[-1:]])
        nblk = part.shape[0]
        strides = (nblk + 255) // 256
        padded = np.zeros((strides * 256, D + 2))
        padded[:nblk] = part
        s_t = np.zeros((256, D + 2))
        for k in range(strides):
            s_t = s_t + padded[k * 256:(k + 1) * 256]
        out = 0.5 * block_sum(s_t)
        if self.mut == "noise_no_half":
            out[D + 1] *= 2.0
        return out

    def rowsum(self, A, rows, cols, scale, w=None):
        strides = max((cols + 255) // 256, 1)
        pad = np.zeros((rows, strides * 256))
        pad[:, :cols] = A[:rows, :cols]
        s = np.zeros((rows, 256))
        for k in range(strides):
            blk = pad[:, k * 256:(k + 1) * 256]
            if w is None:
                s = s + blk
            else:
                wp = np.zeros(strides * 256)
                wp[:cols] = w
                s = fma(wp[k * 256:(k + 1) * 256][None, :], blk, s)
        return scale * block_sum(s[:, :, None])[:, 0]


# ------------------------------------------------------------------------------------------------
# the device, behind the same interface
# ------------------------------------------------------------------------------------------------
def dim_major(pts, ld, fill=np.nan):
    n, d = pts.shape
    buf = np.full((d, ld), fill)
    buf[:, :n] = pts.T
    return buf


class Gpu:
    def __init__(self, gx):
        self.gx, self.dev, self.lib, self.ptr = gx, gx.dev, gx.lib, gx.ptr

    def _kernel(self, cl, s):
        self.dev.set_kernel(0, len(cl), list(np.asarray(cl, dtype=np.float64)) + [float(s)])

    def dgram(self, X, Y, cl, s, ld, out0):
        self._kernel(cl, s)
        dev = self.dev
        nx, ny = X.shape[0], Y.shape[0]
        ldx, ldy = nx + 5, ny + 7
        Xd, Yd, Od = dev.upload(dim_major(X, ldx)), dev.upload(dim_major(Y, ldy)), dev.upload(out0)
        rc = self.lib.gpx_se_dgram(dev.h, self.ptr(Xd), nx, ldx, self.ptr(Yd), ny, ldy, self.ptr(Od), ld, dev.stream)
        assert rc == GPX_OK, self.gx._lib.lib.gpx_last_error()
        return Od.cpu().numpy()

    def var_grad(self, P, X, cl, s, At, Qneg, diag, out0):
        self._kernel(cl, s)
        dev, ptr = self.dev, self.ptr
        n, M, ldx = P.shape[0], X.shape[0], out0.shape[1]
        ldp = n + 3
        Pd, Xd = dev.upload(dim_major(P, ldp)), dev.upload(dim_major(X, ldx))
        Ad, Qd, Od = dev.upload(At), dev.upload(Qneg), dev.upload(out0)
        gd = None if diag is None else dev.upload(diag)
        rc = self.lib.gpx_se_var_grad(dev.h, ptr(Pd), n, ldp, ptr(Xd), M, ldx, ptr(Ad), ptr(Qd), ptr(gd), ptr(Od),
                                      dev.stream)
        assert rc == GPX_OK, self.gx._lib.lib.gpx_last_error()
        return Od.cpu().numpy()

    def loglike_setup(self, X, cl, s):
        """Device X (NaN padding), workspace and output; returns a function (Pd, ldp, alphad) -> out[:D + 2]."""
        self._kernel(cl, s)
        dev, ptr = self.dev, self.ptr
        n, D = X.shape
        ldx = n + 3
        Xd = dev.upload(dim_major(X, ldx))
        ws = dev.zeros(int(self.lib.gpx_se_loglike_grad_workspace(n, D)))

        def run(Pd, ldp, alphad):
            out = dev.empty(D + 3).fill_(-3.25)
            rc = self.lib.gpx_se_loglike_grad(dev.h, ptr(Xd), n, ldx, ptr(Pd), ldp, ptr(alphad), ptr(ws), ptr(out),
                                              dev.stream)
            assert rc == GPX_OK, self.gx._lib.lib.gpx_last_error()
            o = out.cpu().numpy()
            assert o[D + 2] == -3.25
            return o[:D + 2]
        return run

    def loglike(self, X, P, alpha, cl, s):
        n = X.shape[0]
        Pb = np.full((n, n + 1), np.nan)
        Pb[:, :n] = P
        return self.loglike_setup(X, cl, s)(self.dev.upload(Pb), n + 1, self.dev.upload(alpha))

    def rowsum(self, A, rows, cols, scale, w=None):
        dev, ptr = self.dev, self.ptr
        Ad = dev.upload(A)
        out = dev.empty(rows + 1).fill_(-3.25)
        if w is None:
            rc = self.lib.gpx_rowsum(dev.h, ptr(Ad), rows, cols, A.shape[1], float(scale), ptr(out), dev.stream)
        else:
            rc = self.lib.gpx_rowsum_w(dev.h, ptr(Ad), rows, cols, A.shape[1], ptr(dev.upload(w)), ptr(out), dev.stream)
        assert rc == GPX_OK
        o = out.cpu().numpy()
        assert o[rows] == -3.25
        return o[:rows]


# ------------------------------------------------------------------------------------------------
# the checkers, shared by the twins (CPU) and the device (GPU)
# ------------------------------------------------------------------------------------------------
def value_probe(D, seed=0):
    """X: 3 points; Y: one point per A/2 in HALF_EXPONENTS from X[0] along a random direction, A/2 exact up to the
    rounding of the coordinates."""
    rng = np.random.default_rng(100 + D + seed)
    cl = cls(D)
    x0 = np.zeros(D) if D == 1 else 0.1 * np.cos(np.arange(D))
    X = np.vstack([x0, x0 + 0.3 * rng.standard_normal(D) * cl, x0 - 0.05 * cl])
    Y = []
    for E in HALF_EXPONENTS:
        u = rng.standard_normal(D)
        u /= np.linalg.norm(u)
        w = np.sqrt(np.sum((u / cl) ** 2))
        Y.append(x0 + u * (np.sqrt(2.0 * E) / w))
    return X, np.array(Y)


def check_dgram(run, D, s, X, Y, rows=None, cols=None, ld=None):
    """All of: padding columns keep their sentinels bit for bit, no NaN, and every sampled (i, j) within the bound of
    the module docstring against mp_dgram.  Returns the worst error / bound ratio."""
    cl = cls(D)
    nx, ny = X.shape[0], Y.shape[0]
    ld = ny * D + 3 if ld is None else ld
    out0 = sentinels(nx, ld)
    got = run.dgram(X, Y, cl, s, ld, out0)
    assert same_bits(got[:, ny * D:], out0[:, ny * D:]), "dgram wrote into the padding columns"
    assert not np.isnan(got[:, :ny * D]).any(), "dgram produced NaN"
    rows = range(nx) if rows is None else rows
    cols = range(ny) if cols is None else cols
    a = a_of(cl)
    worst, bad = 0.0, []
    for i in rows:
        for j in cols:
            ref, A = mp_dgram(X[i], Y[j], cl, s)
            for k in range(D):
                b = dgram_bound(float(abs(ref[k])), A, s, abs(Y[j, k] - X[i, k]) * a[k], D)
                err = float(abs(mpf(got[i, j * D + k]) - ref[k]))
                worst = max(worst, err / b)
                if not err <= b:
                    bad.append((i, j, k, got[i, j * D + k], float(ref[k]), err / b))
    assert not bad, f"dgram D={D} s={s:g}: {len(bad)} entries out of bound, first {bad[:3]}"
    return worst


def var_grad_case(D, n, M, seed):
    """(P, X, At, Qneg, near, diag): At (magnitudes 1e-3 .. 10), Qneg and diag arbitrary, NaN in the padding; `near`
    marks the half of the entries where the caller makes Qneg cancel D."""
    rng = np.random.default_rng(seed)
    cl = cls(D)
    P = rng.uniform(-1, 1, (n, D)) * cl
    X = rng.uniform(-1, 1, (M, D)) * cl
    ldx = M + 3
    At = np.full((n, ldx), np.nan)
    At[:, :M] = rng.standard_normal((n, M)) * 10.0 ** rng.uniform(-3, 1, (n, M))
    Qneg = np.full((n * D, ldx), np.nan)
    Qneg[:, :M] = rng.standard_normal((n * D, M))
    near = rng.random((n * D, M)) < 0.5
    diag = rng.standard_normal(n * D)
    return P, X, At, Qneg, near, diag


def check_var_grad(run, D, n, M, s, with_diag, seed=0):
    cl = cls(D)
    P, X, At, Qneg, near, diag = var_grad_case(D, n, M, seed + 1000 * D + 10 * n + M)
    # the cancelling half: Qneg = D(x, p) (1 + 2^-k) computed from the float64 formula, k in 10 .. 50
    plain = Twin(False).var_grad(P, X, cl, s, np.full_like(At, 0.5), np.zeros_like(Qneg), None, np.zeros_like(Qneg))
    rng = np.random.default_rng(seed + 7)
    Qneg[:, :M] = np.where(near, plain[:, :M] * (1 + 2.0 ** -rng.integers(10, 50, (n * D, M))), Qneg[:, :M])
    dg = diag if with_diag else None
    ldx = M + 3
    out0 = sentinels(n * D, ldx)
    got = run.var_grad(P, X, cl, s, At, Qneg, dg, out0)
    assert same_bits(got[:, M:], out0[:, M:]), "var_grad wrote into the padding columns"
    assert not np.isnan(got[:, :M]).any(), "var_grad produced NaN"
    a = a_of(cl)
    worst, bad = 0.0, []
    for j in edges(n, 256, 1, seed):
        for m in edges(M, 256, 3, seed):
            ref, dk, A = mp_var_grad_entry(P[j], X[m], cl, s, At[j, m], Qneg[j * D:(j + 1) * D, m],
                                           None if dg is None else dg[j * D:(j + 1) * D])
            for k in range(D):
                r = j * D + k
                b = var_grad_bound(At[j, m], float(abs(dk[k])), abs(Qneg[r, m]), 0.0 if dg is None else abs(dg[r]), A, s,
                                   abs(X[m, k] - P[j, k]) * a[k], D)
                err = float(abs(mpf(got[r, m]) - ref[k]))
                worst = max(worst, err / b)
                if not err <= b:
                    bad.append((j, m, k, got[r, m], float(ref[k]), err / b))
    assert not bad, f"var_grad D={D} n={n} M={M}: {len(bad)} entries out of bound, first {bad[:3]}"
    return worst


LL_N = [1, 2, 255, 256, 257, 600]


def ll_pairs(n):
    """(i, j): the diagonal at both ends, the ends of a 256-column block, and the last ragged block."""
    c = {(0, 0), (n - 1, n - 1), (0, min(1, n - 1)), (n - 1, 0)}
    for e in (255, 256, 257, 511, 512):
        if e < n:
            c |= {(0, e), (e, e), (n - 1, e), (e, n - 1)}
    return sorted(c)


def ll_points(D, n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, (n, D)) * cls(D) * 0.8


def check_loglike_pairs(run_factory, D, n, s=1.7):
    """alpha = 0 and P with one symmetric pair (i, j): out[q] is one computed term, against mp."""
    cl = cls(D)
    X = ll_points(D, n, 50 + D + n)
    run = run_factory(X, cl, s)
    a = a_of(cl)
    worst, bad = 0.0, []
    for idx, (i, j) in enumerate(ll_pairs(n)):
        p = float(1.25 + idx)
        got = run(i, j, p)
        ref, A = mp_loglike_terms(X[i], X[j], cl, s, mpf(-p), i == j)
        ref = [r / 2 for r in ref] if i == j else ref
        for q in range(D + 2):
            df2 = float((X[i, q] - X[j, q]) ** 2) if q < D else 0.0
            b = (C0 + c1(D) * A) * EPS * float(abs(ref[q])) + ll_abs(p, s, df2, a[q] if q < D else 1.0)
            err = float(abs(mpf(got[q]) - ref[q]))
            worst = max(worst, err / b)
            if not err <= b:
                bad.append(((i, j), q, got[q], float(ref[q]), err / b))
    assert not bad, f"loglike pairs D={D} n={n}: {bad[:3]}"
    return worst


def check_loglike_reduction(run, D, n):
    """Identical points: e = 1, the cl entries are 0, out[d] = -sum P / 2 and out[d + 1] = -tr P / 2 exactly."""
    X = np.tile(np.linspace(-0.3, 0.4, D), (n, 1))
    P = (np.arange(n * n, dtype=np.float64).reshape(n, n) + 1.0)   # distinct integers, all sums below 2^53
    got = run(X, P, np.zeros(n), cls(D), 1.7)
    want = np.zeros(D + 2)
    want[D] = -float(P.sum()) / 2
    want[D + 1] = -float(np.trace(P)) / 2
    assert same_bits(got, want), f"loglike reduction D={D} n={n}: got {got[D:]} want {want[D:]}"


def check_loglike_random(run, D, n, seed=0):
    rng = np.random.default_rng(seed + 31 * D + n)
    cl, s = cls(D), 0.7
    X = ll_points(D, n, seed + 3 * n + D)
    alpha = rng.standard_normal(n)
    Pm = rng.standard_normal((n, n))
    Pm = Pm + Pm.T
    got = run(X, Pm, alpha, cl, s)
    a = a_of(cl)
    nb = (n + 255) // 256
    k = 5 + 8 + (n * nb + 255) // 256 + 5 + 8
    gam = k * U_RND / (1 - k * U_RND)
    ref = [mpmath.mpf(0)] * (D + 2)
    mag_rel = np.zeros(D + 2)
    mag = np.zeros(D + 2)
    absb = 0.0
    for i in range(n):
        for j in range(i, n):
            t = mpf(alpha[i]) * mpf(alpha[j]) - mpf(Pm[i, j])
            terms, A = mp_loglike_terms(X[i], X[j], cl, s, t, i == j)
            tm = abs(alpha[i] * alpha[j]) + abs(Pm[i, j])
            mult = 1 if i == j else 2
            for q in range(D + 2):
                ref[q] += mult * terms[q]
                m = float(abs(terms[q] / t)) * tm if t != 0 else float(abs(terms[q])) + tm
                mag[q] += mult * m
                mag_rel[q] += mult * m * (C0 + c1(D) * A) * EPS
            absb += mult * ll_abs(tm, s, float(np.max((X[i] - X[j]) ** 2)), float(a.max()))
    worst, bad = 0.0, []
    for q in range(D + 2):
        r = ref[q] / 2
        b = 0.5 * (mag_rel[q] + gam * 1.01 * mag[q]) + absb
        err = float(abs(mpf(got[q]) - r))
        worst = max(worst, err / b)
        if not err <= b:
            bad.append((q, got[q], float(r), err / b))
    assert not bad, f"loglike random D={D} n={n}: {bad[:3]}"
    return worst


ROWSUM_COLS = [1, 255, 256, 257, 5000]


def check_rowsum(run, cols, seed=0):
    rng = np.random.default_rng(seed + cols)
    rows, ld = 5, cols + 3
    A = np.full((rows, ld), np.nan)
    A[:, :cols] = rng.integers(-2 ** 20, 2 ** 20, (rows, cols))
    for k in (0, 3, 12):
        got = run.rowsum(A, rows, cols, 2.0 ** -k)
        want = np.array([mp_rowsum(A[r, :cols], 2.0 ** -k) for r in range(rows)])
        assert same_bits(got, want), (cols, k, got, want)


# ------------------------------------------------------------------------------------------------
# 1. CPU half: the references against the oracle, the twins against the checkers, the mutants rejected
# ------------------------------------------------------------------------------------------------
def test_fma_emulation_is_correctly_rounded():
    rng = np.random.default_rng(3)
    x = rng.standard_normal(3000) * np.ldexp(1.0, rng.integers(-30, 30, 3000))
    y = rng.standard_normal(3000) * np.ldexp(1.0, rng.integers(-30, 30, 3000))
    z = -(x * y) * (1 + rng.integers(-4, 5, 3000) * EPS)     # heavy cancellation
    z[::3] = rng.standard_normal(1000)
    got = fma(x, y, z)
    for a, b, c, g in zip(x, y, z, got):
        assert g == float(Fraction(a) * Fraction(b) + Fraction(c))
    assert fma(1.0 + 2.0 ** -30, 1.0 - 2.0 ** -30, -1.0) == -(2.0 ** -60)


@pytest.mark.parametrize("D", [1, 2, 5, 16])
def test_mp_dgram_matches_oracle(D):
    rng = np.random.default_rng(D)
    cl = cls(D)
    for s in (0.3, 1.7):
        ks = orc.KernelSpec.se(list(cl), s, D)
        X, Y = rng.uniform(-1, 1, (3, D)), rng.uniform(-1, 1, (6, D))
        for i in range(3):
            want = orc.se_derivative(ks, Y, X[i:i + 1])     # [j, k] = D(y_j, x_i)[k]
            for j in range(6):
                ref, _ = mp_dgram(X[i], Y[j], cl, s)
                assert np.allclose([float(r) for r in ref], want[j], rtol=1e-13, atol=1e-300)


@pytest.mark.parametrize("D", [1, 3])
def test_mp_var_grad_matches_oracle(D):
    """At = P K(D, X) and Qneg = -(dK/dp)^T At from float64 algebra, then mp_var_grad_entry against
    orc.fast_variance_derivative (gp.py:282-341 restated)."""
    rng = np.random.default_rng(10 + D)
    cl, s, noise = cls(D), 1.7, 1e-3
    ks = orc.KernelSpec.se(list(cl), s, D)
    n, M = 5, 7
    design, X = rng.uniform(-1, 1, (n, D)), rng.uniform(-1, 1, (M, D))
    At = np.linalg.solve(ks.gram(design, design) + noise * np.eye(n), ks.gram(design, X))
    dct = np.zeros((n, n * D))                             # gpx_se_dgram(X = design, Y = design)
    for z in range(n):
        for j in range(n):
            dct[z, j * D:(j + 1) * D] = [float(v) for v in mp_dgram(design[z], design[j], cl, s)[0]]
    Qneg = -dct.T @ At
    want = orc.fast_variance_derivative(ks, design, X, noise)
    for j in range(n):
        for m in range(M):
            ref, _, _ = mp_var_grad_entry(design[j], X[m], cl, s, At[j, m], Qneg[j * D:(j + 1) * D, m], None)
            for k in range(D):
                scale = np.max(np.abs(want[j * D + k]))
                assert abs(float(ref[k]) - want[j * D + k, m]) <= 1e-11 * scale


def mp_loglike_gradient(ks, pts, y, noise):
    n, D = pts.shape
    prec = np.linalg.inv(ks.gram(pts, pts) + noise * np.eye(n))
    alpha = prec @ y
    out = [mpmath.mpf(0)] * (D + 2)
    for i in range(n):
        for j in range(n):
            t = mpf(alpha[i]) * mpf(alpha[j]) - mpf(prec[i, j])
            terms, _ = mp_loglike_terms(pts[i], pts[j], ks.cl, ks.signal, t, i == j)
            out = [o + v for o, v in zip(out, terms)]
    return [float(o / 2) for o in out]


@pytest.mark.parametrize("D", [1, 2, 3])
def test_mp_loglike_terms_match_oracle_and_differences(D):
    """The d + 2 entries: against orc.fast_loglike_gradient (whose noise entry is the bare trace times 2 noise) and
    against central differences of the log-likelihood in cl_q, signalSize and noise."""
    rng = np.random.default_rng(20 + D)
    cl, s, noise = cls(D), 1.7, 1e-3
    ks = orc.KernelSpec.se(list(cl), s, D)
    pts = rng.uniform(-1, 1, (9, D))
    y = np.sin(3 * pts).sum(axis=1)
    g = mp_loglike_gradient(ks, pts, y, noise)
    want = orc.fast_loglike_gradient(ks, pts, y, noise)
    scale = max(abs(v) for v in g)
    for q in range(D):
        assert abs(g[q] - want["cl%d" % q]) <= 1e-9 * scale
    assert abs(g[D] - want["signalSize"]) <= 1e-9 * scale
    assert abs(g[D + 1] * 2 * noise - want["noise"]) <= 1e-9 * abs(want["noise"])
    h = 1e-6
    for q in range(D):
        up, dn = cl.copy(), cl.copy()
        up[q] += h
        dn[q] -= h
        fd = (orc.fast_loglike(orc.KernelSpec.se(list(up), s, D), pts, y, noise) -
              orc.fast_loglike(orc.KernelSpec.se(list(dn), s, D), pts, y, noise)) / (2 * h)
        assert abs(fd - g[q]) <= 1e-5 * max(1.0, abs(fd)), q
    fd = (orc.fast_loglike(orc.KernelSpec.se(list(cl), s + h, D), pts, y, noise) -
          orc.fast_loglike(orc.KernelSpec.se(list(cl), s - h, D), pts, y, noise)) / (2 * h)
    assert abs(fd - g[D]) <= 1e-5 * max(1.0, abs(fd))
    hn = 1e-8
    fd = (orc.fast_loglike(ks, pts, y, noise + hn) - orc.fast_loglike(ks, pts, y, noise - hn)) / (2 * hn)
    assert abs(fd - g[D + 1]) <= 1e-4 * max(1.0, abs(fd))    # d loglike / d noise is the bare 1/2 trace


def test_mp_rowsum_matches_fsum():
    rng = np.random.default_rng(4)
    row = rng.standard_normal(1000) * np.ldexp(1.0, rng.integers(-20, 20, 1000))
    assert mp_rowsum(row, 0.25) == math.fsum(row.tolist()) * 0.25


class TwinLoglikePairs:
    """The pair-by-pair runner over a twin: P dense with one symmetric pair, alpha = 0."""

    def __init__(self, twin):
        self.twin = twin

    def __call__(self, X, cl, s):
        n = X.shape[0]

        def run(i, j, p):
            P = np.zeros((n, n))
            P[i, j] = P[j, i] = p
            return self.twin.loglike(X, P, np.zeros(n), cl, s)
        return run


def twin_suite(twin, kernels, D):
    """The GPU tests' checkers, run on a twin; returns the worst ratio per kernel."""
    worst = {}
    if "dgram" in kernels:
        X, Y = value_probe(D)
        worst["dgram"] = max(check_dgram(twin, D, s, X, Y) for s in SIGNALS)
        rng = np.random.default_rng(D)
        for nx in (1, 3, 300):
            for ny in (1, 255, 256, 257, 513):
                Xl, Yl = rng.uniform(-1, 1, (nx, D)) * cls(D), rng.uniform(-1, 1, (ny, D)) * cls(D)
                worst["dgram"] = max(worst["dgram"], check_dgram(twin, D, 1.7, Xl, Yl, edges(nx, 256, 1), edges(ny)))
    if "var_grad" in kernels:
        worst["var_grad"] = max(check_var_grad(twin, D, n, M, s, diag)
                                for n in (1, 2, 40) for M in (1, 255, 256, 257, 1000) for s, diag in ((1.7, True), (0.3, False)))
    if "loglike" in kernels:
        worst["loglike"] = max(check_loglike_pairs(TwinLoglikePairs(twin), D, n) for n in LL_N)
        for n in LL_N:
            check_loglike_reduction(twin.loglike, D, n)
        worst["loglike"] = max(worst["loglike"], max(check_loglike_random(twin.loglike, D, n) for n in (1, 2, 40)))
    return worst


@pytest.mark.parametrize("use_fma", [True, False], ids=["fma", "no_fma"])
@pytest.mark.parametrize("D", TWIN_DIMS)
def test_twins_meet_the_bounds(D, use_fma):
    worst = twin_suite(Twin(use_fma), ("dgram", "var_grad", "loglike"), D)
    for k, v in worst.items():
        note(f"twin_{'fma' if use_fma else 'nofma'}_{k}", D, v)
    for cols in ROWSUM_COLS:
        check_rowsum(Twin(use_fma), cols)


MUTANTS = {
    "signal_once": ("dgram", "var_grad"),
    "a_not_a32": ("loglike",),
    "e_to_k": ("loglike",),
    "noise_no_half": ("loglike",),
    "drop_block": ("loglike",),
    "double_block": ("loglike",),
    "colshift": ("dgram", "var_grad"),
    "diag_sign": ("var_grad",),
    "exp64": ("dgram", "var_grad", "loglike"),
}


@pytest.mark.parametrize("mut", list(MUTANTS))
def test_mutants_are_rejected(mut):
    """Each defect, in each kernel it applies to, fails that kernel's checker (with fma and without)."""
    for use_fma in (True, False):
        for kernel in MUTANTS[mut]:
            with pytest.raises(AssertionError):
                twin_suite(Twin(use_fma, mut), (kernel,), 3)


# ------------------------------------------------------------------------------------------------
# 2. GPU half, kernel by kernel
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    ed.VERBOSE = False
    from gpexp_b200 import _lib, device
    from gpexp_b200 import gp as gpmod
    from gpexp_b200 import kernels as K
    from gpexp_b200.approximation import Space

    class NS:
        pass
    ns = NS()
    ns.torch, ns.lib, ns._lib, ns.device, ns.ed, ns.gp, ns.K, ns.Space = torch, _lib.lib, _lib, device, ed, gpmod, K, Space
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    return ns


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_dgram_values_over_the_exponent_range(gx, D):
    X, Y = value_probe(D)
    note("gpx_se_dgram values", D, max(check_dgram(Gpu(gx), D, s, X, Y) for s in SIGNALS))


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_dgram_block_edges_and_padding(gx, D):
    """nx in {1, 3, 300} x ny in {1, 255, 256, 257, 513}, ld = ny d + 3, NaN in the padding of X and Y: edge rows and
    columns against mp, every other element against the host twin within twice the bound."""
    rng = np.random.default_rng(D)
    gpu, twin = Gpu(gx), Twin(True)
    cl, s = cls(D), 1.7
    a = a_of(cl)
    worst = 0.0
    for nx in (1, 3, 300):
        for ny in (1, 255, 256, 257, 513):
            X, Y = rng.uniform(-1, 1, (nx, D)) * cl, rng.uniform(-1, 1, (ny, D)) * cl
            worst = max(worst, check_dgram(gpu, D, s, X, Y, edges(nx, 256, 1), edges(ny)))
            ld = ny * D + 3
            got = gpu.dgram(X, Y, cl, s, ld, sentinels(nx, ld))[:, :ny * D]
            ref = twin.dgram(X, Y, cl, s, ld, sentinels(nx, ld))[:, :ny * D]
            df = (Y[None, :, :] - X[:, None, :]).reshape(nx, ny * D)
            A = np.repeat(np.sum((Y[None, :, :] - X[:, None, :]) ** 2 * a, axis=2), D, axis=1)
            b = 2 * dgram_bound(np.abs(ref), A, s, np.abs(df) * np.tile(a, ny), D)
            assert np.all(np.abs(got - ref) <= b), (nx, ny, np.argwhere(np.abs(got - ref) > b)[:4])
    note("gpx_se_dgram edges", D, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_dgram_antisymmetry_and_dyadic_shift(gx, D):
    """dgram(X, Y)[i, j d + k] = -dgram(Y, X)[j, i d + k] bit for bit (the difference flips sign exactly, its square
    and the exponent do not change), and adding 32 to every coordinate of dyadic points (multiples of 2^-20 in
    [-1, 1]) keeps every difference, so every bit of the output."""
    rng = np.random.default_rng(D)
    gpu, cl = Gpu(gx), cls(D)
    nx, ny = 300, 257
    X = rng.integers(-2 ** 20, 2 ** 20, (nx, D)) * 2.0 ** -20
    Y = rng.integers(-2 ** 20, 2 ** 20, (ny, D)) * 2.0 ** -20
    for s in (0.3, 1.7):
        f = gpu.dgram(X, Y, cl, s, ny * D, np.zeros((nx, ny * D))).reshape(nx, ny, D)
        b = gpu.dgram(Y, X, cl, s, nx * D, np.zeros((ny, nx * D))).reshape(ny, nx, D)
        assert same_bits(f, -b.transpose(1, 0, 2))
        sh = gpu.dgram(X + 32.0, Y + 32.0, cl, s, ny * D, np.zeros((nx, ny * D))).reshape(nx, ny, D)
        assert same_bits(sh, f)


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_var_grad_entries(gx, D):
    """M in {1, 255, 256, 257, 1000} x n in {1, 2, 40}, ldx = M + 3 with NaN in the padding of X, At and Qneg and
    sentinels in that of out, diag NULL and given; Qneg cancels D to 10 .. 50 bits in half the entries."""
    gpu, worst = Gpu(gx), 0.0
    for n in (1, 2, 40):
        for M in (1, 255, 256, 257, 1000):
            for s, with_diag in ((1.7, True), (0.3, False), (2.0 ** 40, True)):
                worst = max(worst, check_var_grad(gpu, D, n, M, s, with_diag))
    note("gpx_se_var_grad", D, worst)


class GpuLoglikePairs:
    def __init__(self, gx):
        self.gpu = Gpu(gx)

    def __call__(self, X, cl, s):
        gpu, dev = self.gpu, self.gpu.dev
        n = X.shape[0]
        run = gpu.loglike_setup(X, cl, s)
        ldp = n + 1
        Pd = dev.zeros(n, ldp)
        Pd[:, n] = float("nan")
        alphad = dev.zeros(n)

        def pair(i, j, p):
            Pd[i, j] = Pd[j, i] = p
            try:
                return run(Pd, ldp, alphad)
            finally:
                Pd[i, j] = Pd[j, i] = 0.0
        return pair


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_loglike_grad_pair_by_pair(gx, D):
    note("gpx_se_loglike_grad pairs", D, max(check_loglike_pairs(GpuLoglikePairs(gx), D, n) for n in LL_N))


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_loglike_grad_reduction_is_exact(gx, D):
    """n in {1, 2, 255, 256, 257, 600}: nblocks = ceil(n / 256) n is 514 and 1800 (not multiples of 256) at the last
    two, where grad_reduce_kernel's threads stride over several partials."""
    gpu = Gpu(gx)
    for n in LL_N:
        check_loglike_reduction(gpu.loglike, D, n)


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_se_loglike_grad_random(gx, D):
    gpu = Gpu(gx)
    note("gpx_se_loglike_grad random", D, max(check_loglike_random(gpu.loglike, D, n) for n in (1, 2, 40, 100)))


@pytest.mark.gpu
@pytest.mark.parametrize("cols", ROWSUM_COLS)
def test_rowsum_is_exact(gx, cols):
    check_rowsum(Gpu(gx), cols)


@pytest.mark.gpu
def test_loglike_grad_and_rowsum_repeat_bit_for_bit(gx):
    gpu = Gpu(gx)
    for D in (1, 7, 16):
        rng = np.random.default_rng(D)
        n = 300
        X = ll_points(D, n, D)
        P = rng.standard_normal((n, n))
        alpha = rng.standard_normal(n)
        first = gpu.loglike(X, P, alpha, cls(D), 0.7)
        assert same_bits(gpu.loglike(X, P, alpha, cls(D), 0.7), first)
    A = rng.standard_normal((7, 5003))
    w = rng.random(5001)
    assert same_bits(gpu.rowsum(A, 7, 5001, 1 / 5001), gpu.rowsum(A, 7, 5001, 1 / 5001))
    assert same_bits(gpu.rowsum(A, 7, 5001, 1.0, w), gpu.rowsum(A, 7, 5001, 1.0, w))


@pytest.mark.gpu
def test_argument_contract(gx):
    """Refusals return before any launch; zero sizes return GPX_OK and write nothing.  Every buffer is sized for the
    call as made, so none of these could fault even if a check were missing."""
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    st = dev.stream
    buf = dev.zeros(64)
    out = dev.empty(64).fill_(-3.25)
    ws = dev.zeros(64)

    def untouched():
        return bool((out == -3.25).all())
    for family, params in ((1, [0.7, 1.0]), (2, [0.5, 0.3]), (3, [0.7, 1.0]), (4, [0.7, 1.0])):
        dev.set_kernel(family, 2 if family == 2 else 1, params)
        assert lib.gpx_se_dgram(dev.h, ptr(buf), 2, 2, ptr(buf), 2, 2, ptr(out), 4, st) == GPX_EINVAL
        assert lib.gpx_se_var_grad(dev.h, ptr(buf), 2, 2, ptr(buf), 2, 2, ptr(buf), ptr(buf), None, ptr(out), st) == GPX_EINVAL
        assert lib.gpx_se_loglike_grad(dev.h, ptr(buf), 2, 2, ptr(buf), 2, ptr(buf), ptr(ws), ptr(out), st) == GPX_EINVAL
        assert untouched()
    dev.set_kernel(0, 1, [0.7, 1.3])
    big = dev.zeros(65536)
    bigo = dev.empty(65536).fill_(-3.25)
    assert lib.gpx_se_dgram(dev.h, ptr(big), 65536, 65536, ptr(buf), 1, 1, ptr(bigo), 1, st) == GPX_EINVAL
    assert lib.gpx_se_var_grad(dev.h, ptr(big), 65536, 65536, ptr(buf), 1, 1, ptr(big), ptr(big), None, ptr(bigo),
                               st) == GPX_EINVAL
    assert bool((bigo == -3.25).all())
    dev.set_kernel(0, 2, [0.7, 1.1, 1.3])
    assert lib.gpx_se_dgram(dev.h, ptr(buf), 2, 2, ptr(buf), 3, 3, ptr(out), 5, st) == GPX_EINVAL   # ld < ny d
    # ldp < n: a 3 x 3 precision handed over as if its rows were 2 apart
    assert lib.gpx_se_loglike_grad(dev.h, ptr(buf), 3, 3, ptr(buf), 2, ptr(buf), ptr(ws), ptr(out), st) == GPX_EINVAL
    assert lib.gpx_se_loglike_grad(dev.h, ptr(buf), 0, 1, ptr(buf), 1, ptr(buf), ptr(ws), ptr(out), st) == GPX_EINVAL
    for nx, ny in ((0, 3), (3, 0), (0, 0)):
        assert lib.gpx_se_dgram(dev.h, ptr(buf), nx, 3, ptr(buf), ny, 3, ptr(out), 6, st) == GPX_OK
    for n, M in ((0, 3), (3, 0)):
        assert lib.gpx_se_var_grad(dev.h, ptr(buf), n, 3, ptr(buf), M, 3, ptr(buf), ptr(buf), None, ptr(out), st) == GPX_OK
    assert lib.gpx_rowsum(dev.h, ptr(buf), 0, 5, 5, 1.0, ptr(out), st) == GPX_OK
    assert lib.gpx_rowsum_w(dev.h, ptr(buf), 0, 5, 5, ptr(buf), ptr(out), st) == GPX_OK
    dev.sync()
    assert untouched()


# ------------------------------------------------------------------------------------------------
# 3. GPU half, end to end at the new shapes
# ------------------------------------------------------------------------------------------------
E2E_NOISE = 1e-5


def e2e_case(D, n, M, seed):
    rng = np.random.default_rng(seed)
    cl, s = cls(D), 1.3
    return cl, s, rng.uniform(-1, 1, (n, D)) * cl, rng.uniform(-1, 1, (M, D)) * cl


def row_sensitivity(ks, design, X, nug, noise_grad=None):
    """S[r, m] = 2 max_z|At[z, m]| (|D_rm| + sum_z |dK(p_j, p_z)/dp_j,k| max_z|At[z, m]|), r = j d + k: the change of
    entry (r, m) under a perturbation of At of relative size 1 in each column -- what the cond eps error of the two
    solves (Cholesky on the device, LU in the oracle) is multiplied by.  A noise derivative adds |noise_grad[j, k]| per
    design point coincident with p_j to the sum.  Also cond(K)."""
    n, D = design.shape
    K = ks.gram(design, design) + np.diag(np.broadcast_to(nug, (n,)))
    At = np.linalg.solve(K, ks.gram(design, X))
    amax = np.max(np.abs(At), axis=0)
    S = np.zeros((n * D, X.shape[0]))
    for j in range(n):
        Dx = np.abs(orc.se_derivative(ks, X, design[j:j + 1]))          # (M, D)
        dc = np.abs(orc.se_derivative(ks, design, design[j:j + 1]))     # (n, D)
        if noise_grad is not None:
            same = np.linalg.norm(design - design[j], axis=1) < 1e-10
            dc = dc + same[:, None] * np.abs(noise_grad[j])[None, :]
        for k in range(D):
            S[j * D + k] = 2 * amax * (Dx[:, k] + dc[:, k].sum() * amax)
    return S, np.linalg.cond(K)


def check_rows(got, ref, S, cond, what, weights=None):
    """Per gradient row r: |got - ref| <= 1e-9 max|ref_r| + 100 cond eps max S_r (matrix), or with the row reduction
    (weights w, sum over m): 1e-9 sum w |ref_r| + 100 cond eps sum w S_r."""
    if weights is None:
        tol = 1e-9 * np.max(np.abs(ref), axis=1, keepdims=True) + 100 * cond * EPS * np.max(S, axis=1, keepdims=True)
    else:
        tol = 1e-9 * (np.abs(ref) @ weights) + 100 * cond * EPS * (S @ weights)
        ref = ref @ weights
    err = np.abs(got - ref)
    assert np.all(err <= tol), f"{what}: rows {np.unique(np.argwhere(err > tol)[:, 0])[:6]}, worst {np.max(err / tol):.3g}"


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_variance_and_ivar_gradient_end_to_end(gx, D):
    """GP.evaluateVarianceDerivative and costFunctionGP_IVAR.derivative (uniform and mcWeights) against
    orc.fast_variance_derivative, row by row."""
    for n, M in ((1, 255), (7, 257), (40, 1000)):
        cl, s, design, mc = e2e_case(D, n, M, 1000 * D + n)
        ks = orc.KernelSpec.se(list(cl), s, D)
        k = gx.K.KernelSquaredExponential(list(cl), s, D)
        ref = orc.fast_variance_derivative(ks, design, mc, E2E_NOISE)
        S, cond = row_sensitivity(ks, design, mc, E2E_NOISE)
        g = gx.gp.GP(k, E2E_NOISE)
        g.addNodesAndComputeCovariance(design)
        got = g.evaluateVarianceDerivative(mc)
        assert got.shape == ref.shape == (n * D, M)
        check_rows(got, ref, S, cond, f"evaluateVarianceDerivative D={D} n={n} M={M}")
        cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, E2E_NOISE), n, gx.Space(D, None, None), mcPoints=mc)
        check_rows(cf.derivative(design), ref, S, cond, f"IVAR derivative D={D} n={n} M={M}", np.full(M, 1.0 / M))
        w = np.random.default_rng(D + n).random(M)
        cfw = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, E2E_NOISE), n, gx.Space(D, None, None), mcPoints=mc, mcWeights=w)
        check_rows(cfw.derivative(design), ref, S, cond, f"weighted IVAR derivative D={D} n={n} M={M}", w)


@pytest.mark.gpu
@pytest.mark.parametrize("D", DIMS)
def test_loglike_gradient_end_to_end(gx, D):
    """GP.loglikeParams(returnDeriv=1) against orc.fast_loglike_gradient, entry by entry: 1e-9 of the entry's own sum
    of |terms| plus 100 cond eps times its terms' sensitivity to the solves, sum (|alpha_i alpha_j| + max|P|) |dK_q|."""
    for n in (1, 40, 300):
        cl, s, pts, _ = e2e_case(D, n, 1, 2000 * D + n)
        ks = orc.KernelSpec.se(list(cl), s, D)
        y = np.sin(2 * pts).sum(axis=1)
        _, grad = gx.gp.GP(gx.K.KernelSquaredExponential(list(cl), s, D), E2E_NOISE).loglikeParams(pts, y, returnDeriv=1)
        ref = orc.fast_loglike_gradient(ks, pts, y, E2E_NOISE)
        Kn = ks.gram(pts, pts) + E2E_NOISE * np.eye(n)
        cond = np.linalg.cond(Kn)
        prec = np.linalg.inv(Kn)
        alpha = prec @ y
        kmat = ks.gram(pts, pts)
        sens = np.abs(np.outer(alpha, alpha)) + np.max(np.abs(prec))
        term = np.abs(np.outer(alpha, alpha) - prec)
        for q, key in enumerate(list(ref)):
            if q < D:
                dk = kmat * (pts[:, None, q] - pts[None, :, q]) ** 2 / cl[q] ** 3
            elif q == D:
                dk = kmat / s
            else:
                dk = np.eye(n) * 2 * E2E_NOISE
            tol = 0.5 * (1e-9 * np.sum(term * dk) + 100 * cond * EPS * np.sum(sens * dk))
            assert abs(grad[key] - ref[key]) <= tol, (D, n, key, grad[key], ref[key], tol)


class QuadNoise:
    """noise(p) = 1e-4 + 1e-3 p_0^2 and its derivative (the heteroscedastic noise function of the golden vectors)."""

    def __call__(self, p):
        return 1e-4 + 1e-3 * p[:, 0] ** 2

    def deriv(self, p):
        out = np.zeros(p.shape)
        out[:, 0] = 2e-3 * p[:, 0]
        return out


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2, 3, 16])
def test_heteroscedastic_gradient_with_coincident_design_points(gx, D):
    """Two copies of one design point under a noise function: the noise derivative enters the design-Gram derivative at
    every coincident pair (gp.py:314-318), here off the diagonal too.  One integration point sits on a design point,
    which the reference allows (its degenerate-query test is the norm of the whole difference matrix)."""
    nf = QuadNoise()
    cl, s, design, mc = e2e_case(D, 6, 257, 3000 + D)
    design[4] = design[1]
    mc[0] = design[2]
    ks = orc.KernelSpec.se(list(cl), s, D)
    k = gx.K.KernelSquaredExponential(list(cl), s, D)
    nug = nf(design)
    ref = orc.ref_variance_derivative_hetero(ks, design, mc, nug, nf.deriv(design))
    S, cond = row_sensitivity(ks, design, mc, nug, nf.deriv(design))
    g = gx.gp.GP(k, 1e-6)
    g.addNodesAndComputeCovariance(design, noiseIn=nug)
    got = g.evaluateVarianceDerivative(mc, noiseFunc=nf)
    check_rows(got, ref, S, cond, f"hetero evaluateVarianceDerivative D={D}")
    cf = gx.ed.costFunctionGP_IVAR(gx.gp.GP(k, 1e-6), 6, gx.Space(D, None, None, noise=nf), mcPoints=mc)
    check_rows(cf.derivative(design), ref, S, cond, f"hetero IVAR derivative D={D}", np.full(len(mc), 1.0 / len(mc)))
