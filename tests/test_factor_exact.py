"""The factor layer (K2 / K3) against exact arithmetic.

Three kinds of check:
  1. Exact integer factors.  U upper-triangular with off-diagonals in {-2 .. 2} and powers of two 1 .. 8 on the
     diagonal: A = U^T U is an integer matrix, every pivot is 4^e, every division is by 2^e, and every partial sum of
     any summation order is an integer far below 2^53 (asserted as max(|U|^T |U|) < 2^52).  So any Cholesky returns U
     bit for bit, and the solves of U^T X and U X with integer X return X.  U = D (I + N) with N strictly upper and
     N^2 = 0 (N[i, j] != 0 only for i in S, j not in S) has the dyadic inverse U^-T = D^-1 (I - N^T), and
     Y^T Y = A^-1 is dyadic too.  No tolerance anywhere: results equal the exact ones (a zero may carry either sign).
  2. Where `info` lands and what gpx_potrf leaves alone: zero, negative and NaN pivots at the 32-column sub-panel
     edges, the 128-block edges and inside the ragged last block; sentinels in the strictly-lower triangle and the
     padding columns, which the factorisation must neither read nor write.
  3. Rounding where rounding happens: Grams from gpx_gram with nuggets 1e-2 .. 1e-12 (cond up to ~1e14), where a
     forward-error comparison says nothing and only backward-error bounds are valid tests (Higham, Accuracy and Stability
     of Numerical Algorithms, 2nd ed., Thm 8.5 and 10.3).  The residuals are computed exactly (TwoProduct by Veltkamp
     splitting, then math.fsum) for a sample of entries; exact scaling by powers of two and run-to-run
     reproducibility pin what rounding cannot change.
"""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

U_RND = 2.0 ** -53     # unit roundoff
TINY = 2.0 ** -1074    # absolute allowance per operation for gradual underflow (Higham's eta)


def roundup(n, m=128):
    return max(m, (int(n) + m - 1) // m * m)


def same(got, want):
    """Bit-identical up to the sign of zero (+ 0.0 maps -0.0 to +0.0 and keeps every other pattern, NaN included)."""
    got, want = np.asarray(got, dtype=np.float64) + 0.0, np.asarray(want, dtype=np.float64) + 0.0
    return got.shape == want.shape and np.array_equal(got.view(np.int64), want.view(np.int64))


def sentinels(rows, ld):
    """Distinct values -(1000 + flat index): a value that moves, or is overwritten, changes its bit pattern."""
    return -(1000.0 + np.arange(rows * ld, dtype=np.float64).reshape(rows, ld))


# ------------------------------------------------------------------------------------------------
# exact integer factors
# ------------------------------------------------------------------------------------------------
def int_factor(n, seed):
    """Upper-triangular U: off-diagonals in {-2, -1, 1, 2} at 25 % density, diagonal 2^e with e in 0 .. 3."""
    rng = np.random.default_rng(seed)
    U = np.triu(rng.choice(np.array([-2.0, -1.0, 1.0, 2.0]), (n, n)) * (rng.random((n, n)) < 0.25), 1)
    U[np.diag_indices(n)] = 2.0 ** rng.integers(0, 4, n)
    return U + 0.0  # no -0.0 from the products with the density mask


def exact_product(X, Y):
    """X^T Y by float64 BLAS, asserting that it is exact: every partial sum of |X|^T |Y| is an integer below 2^52."""
    assert float((np.abs(X).T @ np.abs(Y)).max(initial=0.0)) < 2.0 ** 52
    return X.T @ Y + 0.0


@functools.lru_cache(maxsize=3)
def int_case(n):
    """(U, A = U^T U) of the integer construction."""
    U = int_factor(n, 1000 + n)
    return U, exact_product(U, U)


def nilpotent_factor(n, seed):
    """(U, Y): U = D (I + N) with N^2 = 0, and its exact inverse transpose Y = U^-T = D^-1 (I - N^T)."""
    rng = np.random.default_rng(seed)
    in_s = rng.random(n) < 0.5
    N = np.triu(rng.choice(np.array([-2.0, -1.0, 1.0, 2.0]), (n, n)) * (rng.random((n, n)) < 0.25), 1)
    N[~in_s, :] = 0.0
    N[:, in_s] = 0.0
    d = 2.0 ** rng.integers(0, 4, n)
    eye = np.eye(n)
    return d[:, None] * (eye + N) + 0.0, (eye - N.T) / d[:, None] + 0.0


def int_rhs(n, ncols, seed):
    """Small integers Z (n x 257); the right-hand side X[:, j] = Z[:, j % 257] with a marker row holding j."""
    rng = np.random.default_rng(seed)
    return rng.integers(-3, 4, (n, min(ncols, 257))).astype(np.float64)


def test_integer_construction_is_exact_under_lapack():
    """The generator itself: LAPACK's Cholesky and triangular solves reproduce U, X and U^-T bit for bit."""
    from scipy.linalg import cholesky, solve_triangular
    for n in (129, 1024, 4097):
        U, A = int_case(n)
        assert np.all(np.diag(U) > 0) and set(np.unique(np.diag(U))) <= {1.0, 2.0, 4.0, 8.0}
        assert same(cholesky(A, lower=False), U)
        X = int_rhs(n, 100, n)
        assert same(solve_triangular(U, exact_product(U, X), trans="T", lower=False), X)
        assert same(solve_triangular(U, exact_product(U.T, X), lower=False), X)
        Un, Y = nilpotent_factor(n, n)
        assert same(Y @ Un.T, np.eye(n))
        assert same(solve_triangular(Un, np.eye(n), trans="T", lower=False), Y)
        An = exact_product(Un, Un)
        assert same(cholesky(An, lower=False), Un)
        assert same(exact_product(Y, Y) @ An, np.eye(n))   # Y^T Y = A^-1, exactly


# ------------------------------------------------------------------------------------------------
# exact residuals
# ------------------------------------------------------------------------------------------------
def _split(a):
    c = 134217729.0 * a  # 2^27 + 1
    hi = c - (c - a)
    return hi, a - hi


def two_product(a, b):
    """(p, e) with p + e = a * b exactly, elementwise (Dekker; no FMA, |a|, |b| < 2^996, no underflow in e)."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def exact_residuals(t, X, Y):
    """r[c] = t[c] - sum_k X[c, k] Y[c, k], computed exactly and rounded once; also sum_k |X[c, k] Y[c, k]|."""
    X, Y = np.atleast_2d(np.asarray(X, dtype=np.float64)), np.atleast_2d(np.asarray(Y, dtype=np.float64))
    p, e = two_product(X, Y)
    mag = np.abs(X * Y).sum(axis=1)
    r = np.array([math.fsum([float(t[c])] + (-p[c]).tolist() + (-e[c]).tolist()) for c in range(X.shape[0])])
    return r, mag


def test_exact_residuals_against_fractions():
    rng = np.random.default_rng(5)
    for trial in range(40):
        L = int(rng.integers(1, 300))
        X = rng.standard_normal((3, L)) * np.ldexp(1.0, rng.integers(-40, 40, (3, L)))
        Y = rng.standard_normal((3, L)) * np.ldexp(1.0, rng.integers(-40, 40, (3, L)))
        t = np.array([float(np.dot(X[0], Y[0])), float(sum(Fraction(a) * Fraction(b) for a, b in zip(X[1], Y[1]))),
                      rng.standard_normal()])
        if trial % 2:  # cancelling: a sum of pairs that cancel exactly but for their rounding error
            X[2] = np.repeat(X[2][: (L + 1) // 2], 2)[:L]
            Y[2] = np.repeat(Y[2][: (L + 1) // 2], 2)[:L] * np.resize([1.0, -1.0], L)
            Y[2][0] *= 1.0 + 2.0 ** -52
        r, mag = exact_residuals(t, X, Y)
        for c in range(3):
            want = Fraction(float(t[c])) - sum(Fraction(a) * Fraction(b) for a, b in zip(X[c], Y[c]))
            assert r[c] == float(want), (trial, c)
            assert abs(mag[c] - float(sum(abs(Fraction(a) * Fraction(b)) for a, b in zip(X[c], Y[c])))) <= 1e-12 * mag[c]
    assert exact_residuals([1.0], [[1.0 + 2.0 ** -30]], [[1.0 - 2.0 ** -30]])[0][0] == 2.0 ** -60


# ------------------------------------------------------------------------------------------------
# device plumbing
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gx():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    from gpexp_b200 import _lib, device

    class NS:
        pass
    ns = NS()
    ns.torch, ns.lib, ns._lib, ns.device = torch, _lib.lib, _lib, device
    ns.dev = device.Device.get(0)
    ns.ptr = device.ptr
    ns.check = _lib.check
    ns.grams = {}
    return ns


def put(gx, M, rows=None, ld=None, fill=0.0):
    """Device rows x ld buffer holding M in its leading block and `fill` (a scalar or a rows x ld array) elsewhere."""
    M = np.asarray(M, dtype=np.float64)
    rows = M.shape[0] if rows is None else rows
    buf = np.array(fill, dtype=np.float64) if np.ndim(fill) else np.full((rows, ld), fill)
    buf[: M.shape[0], : M.shape[1]] = M
    return gx.dev.upload(buf)


def get(t):
    return t.cpu().numpy()


def info_buf(gx, value=0):
    return gx.dev.upload(np.array([value], dtype=np.int32), dtype=gx.torch.int32)


def potrf(gx, Ad, n, ld, info_init=0):
    info = info_buf(gx, info_init)
    gx.check(gx.lib.gpx_potrf(gx.dev.h, gx.ptr(Ad), n, ld, gx.ptr(info), gx.dev.stream), "gpx_potrf")
    return int(info.item())


def wave_columns():
    """Columns tri_solve_kernel covers in one wave: 3 CTAs of 128 threads per SM."""
    import torch
    return 3 * 128 * torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------
# 1. exact integer factors
# ------------------------------------------------------------------------------------------------
POTRF_N = [1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 1000, 2049, 4096, 4097]


def potrf_lds(n):
    return sorted({roundup(n), n + (n & 1)})  # whole tiles, and even but not a multiple of 128


@pytest.mark.gpu
@pytest.mark.parametrize("n", POTRF_N)
def test_potrf_returns_the_integer_factor(gx, n):
    U, A = int_case(n)
    for ld in potrf_lds(n):
        Ad = put(gx, A, ld=ld)
        assert potrf(gx, Ad, n, ld, info_init=3) == 0
        assert same(np.triu(get(Ad)[:, :n]), U), ld


@pytest.mark.gpu
@pytest.mark.parametrize("n", POTRF_N)
def test_potrf_leaves_lower_triangle_and_padding_untouched(gx, n):
    """The header's promise (LAPACK's potrf contract): upper triangle read, U written in place, the strictly-lower part
    and the padding columns neither read nor written.  Sentinels there must survive bit for bit, and U must still be
    exact, so they were not read either."""
    U, A = int_case(n)
    upper = np.triu(np.ones((n, n), dtype=bool))
    for ld in potrf_lds(n):
        M = sentinels(n, ld)
        M[:, :n][upper] = A[upper]
        want = M.copy()
        want[:, :n][upper] = U[upper]
        Ad = gx.dev.upload(M)
        assert potrf(gx, Ad, n, ld) == 0
        got = get(Ad) + 0.0
        bad = np.argwhere(got.view(np.int64) != want.view(np.int64))
        assert bad.size == 0, f"ld {ld}: {len(bad)} entries changed, first {bad[:4].tolist()}"


TRSM_N = [33, 129, 300, 1025]


def trsm_ncols(wave):
    return [1, 2, 77, 128, 129, wave - 1, wave, wave + 1, 100_003]


def solve_case(gx, U, ncols, back, seed):
    """Device (X, B) with B = U^T X (forward) or U X (back), X integer and every column distinct: X[:, j] is
    Z[:, j % 257] except in a marker row that holds j (row 0 for U^T, whose row 0 couples it into every entry of B;
    row n-1 for U, whose column n-1 does).  B is formed on the device from the exact n x 257 product and the marker's
    rank-1 term, both integers: one product and one sum per entry, exact."""
    torch, dev = gx.torch, gx.dev
    n = U.shape[0]
    Z = int_rhs(n, ncols, seed)
    P = Z.shape[1]
    mr = n - 1 if back else 0
    T = U if back else U.T                                  # B = T X
    BZ = exact_product(T.T, Z)
    assert float(np.abs(T[:, mr]).max()) * ncols + float((np.abs(T) @ np.abs(Z)).max()) < 2.0 ** 52
    idx = torch.arange(ncols, device=dev.torch_device) % P
    jcol = torch.arange(ncols, device=dev.torch_device, dtype=torch.float64)
    Zd, BZd = dev.upload(Z), dev.upload(BZ)
    X = Zd[:, idx]
    delta = jcol - X[mr]
    X[mr] = jcol
    B = BZd[:, idx] + dev.upload(T[:, mr].copy())[:, None] * delta[None, :]
    return X, B


@pytest.mark.gpu
@pytest.mark.parametrize("n", TRSM_N)
def test_trsm_and_trsm_back_return_the_integer_solution(gx, n):
    """gpx_trsm (U^-T B) and gpx_trsm_back (U^-1 B, with U^T from gpx_transpose as DesignFactor.Ut makes it), around
    the one-wave limit of tri_solve_kernel's grid: past it every CTA walks several column chunks."""
    torch, dev, lib, ptr = gx.torch, gx.dev, gx.lib, gx.ptr
    U, _ = int_case(n)
    ldu = roundup(n)
    Ud = put(gx, U, ld=ldu)
    Utd = dev.zeros(n, ldu)
    gx.check(lib.gpx_transpose(dev.h, ptr(Ud), n, n, ldu, ptr(Utd), ldu, dev.stream))
    for ncols in trsm_ncols(wave_columns()):
        ldb = ncols + (ncols & 1)
        for back in (False, True):
            X, B = solve_case(gx, U, ncols, back, seed=n + ncols)
            Bd = torch.full((n, ldb), -7.5, dtype=torch.float64, device=dev.torch_device)
            Bd[:, :ncols] = B
            if back:
                gx.check(lib.gpx_trsm_back(dev.h, ptr(Utd), n, ldu, ptr(Bd), ncols, ldb, dev.stream))
            else:
                gx.check(lib.gpx_trsm(dev.h, ptr(Ud), n, ldu, ptr(Bd), ncols, ldb, dev.stream))
            wrong = (Bd[:, :ncols] != X).any(dim=0).nonzero().flatten()
            assert wrong.numel() == 0, (ncols, back, wrong[:8].tolist())
            assert bool((Bd[:, ncols:] == -7.5).all()), (ncols, back)   # the odd column count's padding


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 128, 129, 515, 2049])
def test_trtri_t_returns_the_dyadic_inverse(gx, n):
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    U, Y = nilpotent_factor(n, 300 + n)
    ld = roundup(n)
    Ud = put(gx, U, ld=ld)
    Yd = dev.empty(n, ld).fill_(np.nan)
    gx.check(lib.gpx_trtri_t(dev.h, ptr(Ud), n, ld, ptr(Yd), ld, dev.stream))
    assert same(get(Yd)[:, :n], Y)   # exact zeros above the diagonal included


def mi_column(gx, Yd, nrows, ncols, ldy, p, rank=0, blk=0, world=1, ycol=None):
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    pd = dev.upload(np.array([p], dtype=np.int64), dtype=gx.torch.int64)
    ws = dev.zeros(max(int(lib.gpx_mi_prec_column_workspace(nrows, ldy)), 1))
    out = dev.empty(ncols + 1).fill_(-3.25)
    gx.check(lib.gpx_mi_prec_column(dev.h, ptr(Yd), nrows, ncols, ldy, rank, blk, world, ptr(pd), ptr(ycol), ptr(ws),
                                    ptr(out), dev.stream))
    o = get(out)
    assert o[ncols] == -3.25
    return o[:ncols]


def mi_pivots(n):
    return sorted({p for p in (0, 255, 256, 511, 512, 1023, 1024, n - 1) if 0 <= p < n})


@pytest.mark.gpu
@pytest.mark.parametrize("nrows", [1, 255, 256, 257, 1000])
def test_mi_prec_column_dense_is_exact(gx, nrows):
    _, Y = nilpotent_factor(nrows, 500 + nrows)
    P = exact_product(Y, Y)
    for ldy in sorted({roundup(nrows), nrows + (nrows & 1)}):
        Yd = put(gx, Y, ld=ldy)
        for p in mi_pivots(nrows):
            assert same(mi_column(gx, Yd, nrows, nrows, ldy, p), P[:, p]), (ldy, p)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_mi_prec_column_block_cyclic_is_exact(gx, world):
    """Each rank's block-cyclic column slice (blk = 256, ragged last block) with the pivot column passed as a vector
    returns the same global columns of Y^T Y."""
    from gpexp_b200.engine import ShardedMIEngine
    V, blk = 256 * 5 + 77, 256
    _, Y = nilpotent_factor(V, 700 + world)
    P = exact_product(Y, Y)
    for rank in range(world):
        g = ShardedMIEngine.cyclic_columns(V, blk, world, rank)
        nloc = g.size
        ldy = roundup(nloc)
        Yd = put(gx, Y[:, g], ld=ldy)
        for p in mi_pivots(V):
            ycol = gx.dev.upload(Y[:, p].copy())
            assert same(mi_column(gx, Yd, V, nloc, ldy, p, rank, blk, world, ycol), P[g, p]), (rank, p)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 1000])
def test_potrf_trtri_mi_chain_gives_exact_inverse_columns(gx, n):
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    U, Y = nilpotent_factor(n, 900 + n)
    A = exact_product(U, U)
    Ainv = exact_product(Y, Y)
    assert same(Ainv @ A, np.eye(n))
    ld = roundup(n)
    Ad = put(gx, A, ld=ld)
    assert potrf(gx, Ad, n, ld) == 0
    Yd = dev.zeros(n, ld)
    gx.check(lib.gpx_trtri_t(dev.h, ptr(Ad), n, ld, ptr(Yd), ld, dev.stream))
    for p in mi_pivots(n):
        assert same(mi_column(gx, Yd, n, n, ld, p), Ainv[:, p]), p


def append_call(gx, Ud, n, ld, knew, kpp, info_init=0):
    info = info_buf(gx, info_init)
    gx.check(gx.lib.gpx_chol_append(gx.dev.h, gx.ptr(Ud), n, ld, gx.ptr(knew), float(kpp), gx.ptr(info),
                                    gx.dev.stream), "gpx_chol_append")
    return int(info.item())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 1024, 6112, 6113, 6143, 6144, 6145])
def test_chol_append_is_exact(gx, n):
    """Column n of U and U[n, n] from knew = U^T u and kpp = |u|^2 + U[n, n]^2.  From n = 6113 on, the n doubles of x
    plus the kernel's 32-double reduction buffer exceed the 48 KB a launch gets without opting in.  Nothing else in U
    changes."""
    Uf = int_factor(n + 1, 2000 + n)
    u = Uf[:n, n].copy()
    knew = exact_product(Uf[:n, :n], u[:, None])[:, 0]
    kpp = float(u @ u) + Uf[n, n] ** 2
    ld = roundup(n + 1)
    start = Uf.copy()
    start[: n + 1, n] = -99.0
    Ud = put(gx, start, ld=ld)
    knew_d = gx.dev.upload(np.concatenate([knew, [0.0]]))
    assert append_call(gx, Ud, n, ld, knew_d, kpp, info_init=5) == 0
    got = get(Ud)
    assert same(got[:, n], Uf[:, n]), np.flatnonzero(got[:, n] != Uf[:, n])[:8]
    assert same(got[:, :n], Uf[:, :n]) and not np.any(got[:, n + 1:])


@pytest.mark.gpu
def test_chol_append_at_its_size_limit(gx):
    """n = 25 600, the documented limit (200 KB of shared memory): a sparse integer U built on the device (four
    off-diagonals per column, a dense new column u), so that no 5 GB host matrix is needed.  25 601 is refused."""
    torch, dev, lib, ptr = gx.torch, gx.dev, gx.lib, gx.ptr
    n = 25_600
    ld = roundup(n + 1)
    rng = np.random.default_rng(25600)
    cols = np.repeat(np.arange(1, n), 4)
    rows = (rng.random(cols.size) * cols).astype(np.int64)
    rc = np.unique(np.stack([rows, cols], 1), axis=0)
    rows, cols = rc[:, 0], rc[:, 1]
    vals = rng.choice(np.array([-2.0, -1.0, 1.0, 2.0]), rows.size)
    diag = 2.0 ** rng.integers(0, 4, n + 1)
    u = rng.integers(-2, 3, n).astype(np.float64)
    # knew = U[:n, :n]^T u, exactly: diagonal term plus the sparse column sums
    knew = diag[:n] * u
    np.add.at(knew, cols, vals * u[rows])
    mag = np.abs(diag[:n] * u)
    np.add.at(mag, cols, np.abs(vals * u[rows]))
    assert mag.max() < 2.0 ** 52
    kpp = float(u @ u) + diag[n] ** 2
    want = torch.zeros((n + 1, ld), dtype=torch.float64, device=dev.torch_device)
    ar = torch.arange(n + 1, device=dev.torch_device)
    want[ar, ar] = dev.upload(diag)
    want[dev.upload(rows, dtype=torch.int64), dev.upload(cols, dtype=torch.int64)] = dev.upload(vals)
    want[:n, n] = dev.upload(u)
    Ud = want.clone()
    Ud[:, n] = -99.0
    Ud[n + 1:, n] = 0.0
    assert append_call(gx, Ud, n, ld, dev.upload(knew), kpp, info_init=5) == 0
    assert bool(torch.equal(Ud, want))
    del Ud, want
    small = dev.zeros(4)
    info = info_buf(gx)
    assert lib.gpx_chol_append(dev.h, ptr(small), n + 1, n + 2, ptr(small), 1.0, ptr(info), dev.stream) == -4  # GPX_ESIZE


@pytest.mark.gpu
def test_chol_append_reports_non_positive_pivot(gx):
    """d^2 = kpp - |x|^2 exactly 0 gives info = n + 1 and U[n, n] = 0; exactly -1 gives info = n + 1 and NaN; a later
    success writes info = 0 again."""
    n = 33
    Uf = int_factor(n + 1, 77)
    u = Uf[:n, n].copy()
    knew = gx.dev.upload(exact_product(Uf[:n, :n], u[:, None])[:, 0])
    ld = roundup(n + 1)
    Ud = put(gx, Uf, ld=ld)
    ss = float(u @ u)
    assert append_call(gx, Ud, n, ld, knew, ss) == n + 1
    assert get(Ud)[n, n] == 0.0 and same(get(Ud)[:n, n], u)
    assert append_call(gx, Ud, n, ld, knew, ss - 1.0) == n + 1
    assert np.isnan(get(Ud)[n, n])
    assert append_call(gx, Ud, n, ld, knew, ss + 4.0, info_init=n + 1) == 0
    assert get(Ud)[n, n] == 2.0


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 257, 258, 259, 260])
def test_colsumsq_is_exact(gx, n):
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    rng = np.random.default_rng(40 + n)
    for ncols in (1, 2, 255, 256, 1001):
        ldw = ncols + (ncols & 1)
        W = rng.integers(-5, 6, (max(n, 1), ldw)).astype(np.float64)
        base = rng.integers(-1000, 1000, ncols).astype(np.float64)
        Wd, based = dev.upload(W), dev.upload(base)
        ssq = (W[:n, :ncols] ** 2).sum(axis=0)
        for with_base in (False, True):
            out = dev.empty(ncols + 1).fill_(-3.25)
            gx.check(lib.gpx_colsumsq(dev.h, ptr(Wd), n, ncols, ldw, ptr(based) if with_base else None, ptr(out),
                                      dev.stream))
            o = get(out)
            assert same(o[:ncols], base - ssq if with_base else ssq), (ncols, with_base)
            assert o[ncols] == -3.25


DG_I = [1, 63, 64, 65, 128, 129, 200]
DG_J = [1, 2, 127, 128, 129, 257]
DG_K = [1, 15, 16, 17, 31, 32, 33, 4097]


def dgemm(gx, variant, Ad, lda, Bd, ldb, Cd, ldc, I, J, K, upper):
    fn = gx.lib.gpx_dgemm_tn_sub if variant == "generic" else gx.lib.gpx_dgemm_tn_sub_padded
    gx.check(fn(gx.dev.h, gx.ptr(Ad), lda, gx.ptr(Bd), ldb, gx.ptr(Cd), ldc, I, J, K, upper, gx.dev.stream), variant)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["generic", "padded"])
@pytest.mark.parametrize("I", DG_I)
def test_dgemm_tn_sub_is_exact(gx, variant, I):
    """C - A^T B on integer operands, bit for bit, across the 64 / 128-row tile edges, the odd-J scalar tail and the K
    chunk tails (16 rows in the generic core, 32 in the TMA kernel).  Rows of A and B past K hold non-zero integers,
    the columns past I / J too, and C's padding holds sentinels: none may leak.  upper_only = 1 updates exactly the
    entries j >= i and leaves the strictly-lower ones untouched."""
    rng = np.random.default_rng(I)
    lda, ldb, ldc = 256, 384, 384
    A = rng.integers(-3, 4, (max(DG_K), lda)).astype(np.float64)
    B = rng.integers(-3, 4, (max(DG_K), ldb)).astype(np.float64)
    Ad, Bd = gx.dev.upload(A), gx.dev.upload(B)
    for J in DG_J:
        C0 = sentinels(I, ldc)
        C0[:, :J] = rng.integers(-50, 51, (I, J))
        upper = np.triu(np.ones((I, J), dtype=bool))
        for K in DG_K:
            T = exact_product(A[:K, :I], B[:K, :J])
            for up in (0, 1):
                want = C0.copy()
                want[:, :J] -= np.where(upper, T, 0.0) if up else T
                Cd = gx.dev.upload(C0)
                dgemm(gx, variant, Ad, lda, Bd, ldb, Cd, ldc, I, J, K, up)
                got = get(Cd) + 0.0
                bad = np.argwhere(got.view(np.int64) != (want + 0.0).view(np.int64))
                assert bad.size == 0, f"J {J} K {K} upper_only {up}: {len(bad)} wrong, first {bad[:4].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["generic", "padded"])
def test_dgemm_tn_sub_in_the_potrf_layout(gx, variant):
    """The pointer layout gpx_potrf itself uses: A = B = the block row A12 = M[kb:kb+b, kb+b:n], C = the trailing block
    M[kb+b:, kb+b:] of the same matrix, upper_only = 1.  Only the upper triangle of the trailing block changes."""
    kb, b, rest = 128, 128, 300
    n = kb + b + rest
    ld = roundup(n)
    rng = np.random.default_rng(11)
    M = rng.integers(-4, 5, (n, ld)).astype(np.float64)
    A12 = M[kb:kb + b, kb + b:n]
    T = exact_product(A12, A12)
    want = M.copy()
    tr = want[kb + b:, kb + b:n]
    tr -= np.triu(T)
    Md = gx.dev.upload(M)
    off12, off22 = (kb * ld + kb + b) * 8, ((kb + b) * ld + kb + b) * 8
    fn = gx.lib.gpx_dgemm_tn_sub if variant == "generic" else gx.lib.gpx_dgemm_tn_sub_padded
    p = gx.ptr(Md)
    gx.check(fn(gx.dev.h, p + off12, ld, p + off12, ld, p + off22, ld, rest, rest, b, 1, gx.dev.stream))
    assert same(get(Md), want)


@pytest.mark.gpu
@pytest.mark.parametrize("blk", [128, 256])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_dgemm_tn_sub_lower_is_exact(gx, blk, world):
    """gpx_dgemm_tn_sub_lower: B is each rank's block-cyclic slice of a lower-triangular integer matrix (ragged last
    block, K not a multiple of the 32-row chunk); skipping the structurally-zero rows must not change a bit."""
    from gpexp_b200.engine import ShardedMIEngine
    V = blk * 2 * world + 77
    K, I = V - 45, 200
    rng = np.random.default_rng(blk + world)
    Lm = np.tril(rng.integers(-3, 4, (V, V)).astype(np.float64))
    A = rng.integers(-3, 4, (K, 256)).astype(np.float64)
    Ad = gx.dev.upload(A)
    for rank in range(world):
        g = ShardedMIEngine.cyclic_columns(V, blk, world, rank)
        nloc = g.size
        ld = roundup(nloc)
        Bd = put(gx, Lm[:K, g], ld=ld)
        C0 = rng.integers(-50, 51, (I, nloc)).astype(np.float64)
        Cd = put(gx, C0, ld=ld, fill=-11.0)
        gx.check(gx.lib.gpx_dgemm_tn_sub_lower(gx.dev.h, gx.ptr(Ad), 256, gx.ptr(Bd), ld, gx.ptr(Cd), ld, I, nloc, K,
                                               blk, world, rank, gx.dev.stream))
        got = get(Cd)
        assert same(got[:, :nloc], C0 - exact_product(A[:, :I], Lm[:K, g])), rank
        assert np.all(got[:, nloc:] == -11.0)


# ------------------------------------------------------------------------------------------------
# 2. where info lands
# ------------------------------------------------------------------------------------------------
def pivot_positions(n):
    return sorted({k for k in (0, 1, 30, 31, 32, 33, 63, 64, 127, 128, 129, 255, 256, n - 2, n - 1) if 0 <= k < n})


@pytest.mark.gpu
@pytest.mark.parametrize("n", [129, 300, 515])
def test_potrf_info_marks_the_first_bad_pivot(gx, n):
    """Pivot k exactly 0 (U[k, k] = 0 in the integer construction), exactly -1 (a_kk lowered by 1), or NaN (on the
    diagonal at k, or above it in column k): info = k + 1, whichever sub-panel, block or ragged block k falls in."""
    U, A = int_case(n)
    ld = roundup(n)
    for k in pivot_positions(n):
        Uz = U.copy()
        Uz[k, k] = 0.0
        Az = exact_product(Uz, Uz)
        assert potrf(gx, put(gx, Az, ld=ld), n, ld) == k + 1, ("zero", k)
        Az[k, k] -= 1.0
        assert potrf(gx, put(gx, Az, ld=ld), n, ld) == k + 1, ("negative", k)
        for i in sorted({k, k // 2, k - 1, 0} - {-1}):
            An = A.copy()
            An[i, k] = An[k, i] = np.nan
            assert potrf(gx, put(gx, An, ld=ld), n, ld) == k + 1, ("nan", i, k)


@pytest.mark.gpu
def test_potrf_resets_a_stale_info(gx):
    U, A = int_case(129)
    assert potrf(gx, put(gx, A, ld=256), 129, 256, info_init=7) == 0
    assert potrf(gx, put(gx, A, ld=256), 0, 256, info_init=7) == 0


# ------------------------------------------------------------------------------------------------
# 3. rounding: backward-error bounds on real Grams
# ------------------------------------------------------------------------------------------------
GRAM_N = [129, 1000, 2049, 4096]
NUGGETS = [1e-2, 1e-6, 1e-10, 1e-12]
# family, gpx parameters (d = 2), point distribution
FAMILIES = {
    "se": (0, [0.3, 0.4, 1.0], "box"),
    "matern": (1, [0.3, 1.0], "box"),
    "mehler": (2, [0.8, 0.8], "normal"),
}


def points(fam, n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1.5, 1.5, (n, 2)) if FAMILIES[fam][2] == "box" else rng.standard_normal((n, 2))


def set_family(gx, fam):
    family, params, _ = FAMILIES[fam]
    gx.dev.set_kernel(family, 2, params)


def gram(gx, X, Y, ld, nugget=None):
    """K(X, Y) from gpx_gram into a zeroed nx x ld buffer (+ nugget on the diagonal)."""
    out = gx.dev.zeros(X.n, ld)
    gx.check(gx.lib.gpx_gram(gx.dev.h, gx.ptr(X.X), X.n, X.ld, gx.ptr(Y.X), Y.n, Y.ld, gx.ptr(out), ld,
                             0 if nugget is None else 1, None, 0.0 if nugget is None else float(nugget), gx.dev.stream))
    return out


def gram_case(gx, fam, n, nugget):
    """(D points, A = K(D, D) + nugget I, U = gpx_potrf(A)) on the device, cached for the module."""
    key = (fam, n, nugget)
    set_family(gx, fam)  # the cross-covariance blocks the callers form next use the same family
    if key not in gx.grams:
        D = gx.dev.points(points(fam, n, n))
        Ad = gram(gx, D, D, roundup(n), nugget)
        Ud = Ad.clone()
        assert potrf(gx, Ud, n, roundup(n)) == 0, key
        gx.grams[key] = (D, Ad, Ud)
    return gx.grams[key]


def edge_indices(n, b):
    return sorted({e for k in range(b, n, b) for e in (k - 1, k)} | {0, n - 1})


def factor_sample(n, seed):
    """Entries (i, j), i <= j: pairs of 128-block edge indices up to four blocks apart and with the last column, each
    32-edge index with itself and its right neighbour, a stride through the diagonal, and 300 random upper entries."""
    rng = np.random.default_rng(seed)
    e128, e32 = edge_indices(n, 128), edge_indices(n, 32)
    pairs = {(a, b) for a in e128 for b in e128 if a <= b and (b - a < 4 * 128 or b == n - 1)}
    pairs |= {(e, e) for e in e32} | {(e, min(e + 1, n - 1)) for e in e32}
    pairs |= {(i, i) for i in range(0, n, max(1, n // 200))}
    r = rng.integers(0, n, (300, 2))
    pairs |= {(int(min(a, b)), int(max(a, b))) for a, b in r}
    return np.array(sorted(pairs, key=lambda p: (p[0], p[1])))


def chunked_residuals(t, X, Y, lengths, chunk=256):
    """exact_residuals over rows of X, Y truncated per chunk to the longest needed length (entries sorted by it)."""
    order = np.argsort(lengths, kind="stable")
    r, mag = np.empty(len(t)), np.empty(len(t))
    for s in range(0, len(t), chunk):
        o = order[s:s + chunk]
        L = int(lengths[o].max())
        r[o], mag[o] = exact_residuals(t[o], X[o, :L], Y[o, :L])
    return r, mag


def check_bound(res, mag, n, what, extra=0.0):
    bound = (n + 2) * U_RND * (mag + extra) + 2 * (n + 2) * TINY
    ratio = np.abs(res) / bound
    assert np.all(np.abs(res) <= bound), f"{what}: worst residual / bound = {ratio.max():.3g}"
    return float(ratio.max())


@pytest.mark.gpu
@pytest.mark.parametrize("fam", list(FAMILIES))
@pytest.mark.parametrize("n", GRAM_N)
def test_potrf_backward_error_on_grams(gx, fam, n):
    """|A - U^T U|_ij <= (n + 2) u (|U|^T |U|)_ij (Higham Thm 10.3), for any summation order, with the residual exact;
    and gpx_logdet_chol within (n + 2) u sum |2 log U_ii| + n ulp of fsum(2 log U_ii)."""
    dev, lib, ptr = gx.dev, gx.lib, gx.ptr
    S = factor_sample(n, n)
    i, j = S[:, 0], S[:, 1]
    for nugget in NUGGETS:
        _, Ad, Ud = gram_case(gx, fam, n, nugget)
        A, U = get(Ad)[:, :n], np.triu(get(Ud)[:, :n])
        res, mag = chunked_residuals(A[i, j], U[:, i].T, U[:, j].T, np.minimum(i, j) + 1)
        check_bound(res, mag, n, f"{fam} nugget {nugget}")
        out = dev.zeros(1)
        gx.check(lib.gpx_logdet_chol(dev.h, ptr(Ud), n, roundup(n), ptr(out), dev.stream))
        terms = 2.0 * np.log(np.diag(U))
        ref = math.fsum(terms.tolist())
        got = float(out.item())
        assert abs(got - ref) <= (n + 2) * U_RND * float(np.abs(terms).sum()) + n * np.spacing(abs(ref)), (nugget, got, ref)


def solve_sample(n, m, seed):
    """(row, column) entries: every 32-edge row in three columns (first, last, one random) and 400 random entries."""
    rng = np.random.default_rng(seed)
    cols = [0, m - 1, int(rng.integers(0, m))]
    ent = {(r, c) for r in edge_indices(n, 32) for c in cols}
    ent |= {(int(r), int(c)) for r, c in zip(rng.integers(0, n, 400), rng.integers(0, m, 400))}
    return np.array(sorted(ent))


@pytest.mark.gpu
@pytest.mark.parametrize("fam", list(FAMILIES))
@pytest.mark.parametrize("n", GRAM_N)
def test_solves_backward_error_on_grams(gx, fam, n):
    """gpx_trsm: |b - U^T x|_i <= (n + 2) u (|U^T| |x|)_i; gpx_trsm_back the same for U (Higham Thm 8.5), with U the
    computed factor of a real Gram and b a cross-covariance block K(D, Y)."""
    torch, dev, lib, ptr = gx.torch, gx.dev, gx.lib, gx.ptr
    m = 301
    ldb = m + 1
    for nugget in NUGGETS:
        D, _, Ud = gram_case(gx, fam, n, nugget)
        ldu = roundup(n)
        U = np.triu(get(Ud)[:, :n])
        Y = dev.points(points(fam, m, 10 * n + 1))
        Bd = gram(gx, D, Y, ldb)
        B = get(Bd)[:, :m]
        Xf = Bd.clone()
        gx.check(lib.gpx_trsm(dev.h, ptr(Ud), n, ldu, ptr(Xf), m, ldb, dev.stream))
        Utd = dev.zeros(n, ldu)
        gx.check(lib.gpx_transpose(dev.h, ptr(Ud), n, n, ldu, ptr(Utd), ldu, dev.stream))
        Xb = Bd.clone()
        gx.check(lib.gpx_trsm_back(dev.h, ptr(Utd), n, ldu, ptr(Xb), m, ldb, dev.stream))
        xf, xb = get(Xf)[:, :m], get(Xb)[:, :m]
        E = solve_sample(n, m, n + 3)
        r, c = E[:, 0], E[:, 1]
        res, mag = chunked_residuals(B[r, c], U[:, r].T, xf[:, c].T, r + 1)     # row r of U^T: U[k, r], k <= r
        check_bound(res, mag, n, f"trsm {fam} nugget {nugget}")
        # row r of U: U[r, k], k >= r -- reversed so that the live part leads
        res, mag = chunked_residuals(B[r, c], U[r, ::-1], xb[::-1, c].T, n - r)
        check_bound(res, mag, n, f"trsm_back {fam} nugget {nugget}")


@pytest.mark.gpu
@pytest.mark.parametrize("fam", list(FAMILIES))
@pytest.mark.parametrize("n", GRAM_N)
def test_trsm_gram_backward_error_and_its_two_paths(gx, fam, n):
    """gpx_trsm_gram W = U^-T K(D, Y) on both update paths: the TMA kernel (ldu, ldw whole tiles) and the predicated
    one (ldw = ny + 1).  Each meets the bound of Thm 8.5 against K(D, Y) from gpx_gram, and var_out is within
    (n + 2) u (k(y, y) + sum w^2) of k(y, y) - sum w^2 computed exactly from the returned W.  The two paths are
    bit-identical: both accumulate every entry over K in the same order of 4-row DMMA steps from zero and subtract the
    sum once, and the rows past K read as zeros in both."""
    torch, dev, lib, ptr = gx.torch, gx.dev, gx.lib, gx.ptr
    ny = 301
    for nugget in NUGGETS:
        D, _, Ud = gram_case(gx, fam, n, nugget)
        ldu = roundup(n)
        U = np.triu(get(Ud)[:, :n])
        Y = dev.points(points(fam, ny, 10 * n + 2))
        K = get(gram(gx, D, Y, ny + 1))[:, :ny]
        kyy = dev.zeros(ny)
        gx.check(lib.gpx_prior_diag(dev.h, ptr(Y.X), ny, Y.ld, ptr(kyy), dev.stream))
        kyy = get(kyy)
        Ws = []
        for ldw in (roundup(ny), ny + 1):
            Wd, var = dev.zeros(n, ldw), dev.zeros(ny)
            gx.check(lib.gpx_trsm_gram(dev.h, ptr(Ud), n, ldu, ptr(D.X), D.ld, ptr(Y.X), ny, Y.ld, ptr(Wd), ldw, ptr(var),
                                       dev.stream))
            W, var = get(Wd)[:, :ny], get(var)
            Ws.append(W)
            E = solve_sample(n, ny, n + 5)
            r, c = E[:, 0], E[:, 1]
            res, mag = chunked_residuals(K[r, c], U[:, r].T, W[:, c].T, r + 1)
            check_bound(res, mag, n, f"trsm_gram ldw {ldw} {fam} nugget {nugget}")
            exact_var, ssq = exact_residuals(kyy, W.T, W.T)
            vres = var - exact_var
            check_bound(vres, ssq, n, f"var_out ldw {ldw} {fam} nugget {nugget}", extra=kyy)
        assert same(Ws[0], Ws[1]), (fam, n, nugget)


# ------------------------------------------------------------------------------------------------
# 4. exact properties of the real data
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fam", list(FAMILIES))
@pytest.mark.parametrize("n", GRAM_N)
def test_scaling_by_powers_of_two_and_repeat_runs_are_bit_exact(gx, fam, n):
    """gpx_potrf(4^k A) = 2^k gpx_potrf(A), gpx_trsm / gpx_trsm_back (U, 2^k B) = 2^k (U, B), bit for bit: every
    operation scales exactly away from overflow and underflow.  A second run of each call repeats the first bit for
    bit."""
    torch, dev, lib, ptr = gx.torch, gx.dev, gx.lib, gx.ptr
    ld, m = roundup(n), 129
    ldb = m + 1
    for nugget in NUGGETS:
        D, Ad, Ud = gram_case(gx, fam, n, nugget)
        U2 = Ad.clone()
        assert potrf(gx, U2, n, ld) == 0
        assert torch.equal(U2, Ud), "repeat potrf"
        Utd = dev.zeros(n, ld)
        gx.check(lib.gpx_transpose(dev.h, ptr(Ud), n, n, ld, ptr(Utd), ld, dev.stream))
        B = gram(gx, D, dev.points(points(fam, m, 10 * n + 3)), ldb)

        def solves(Bin):
            xf, xb = Bin.clone(), Bin.clone()
            gx.check(lib.gpx_trsm(dev.h, ptr(Ud), n, ld, ptr(xf), m, ldb, dev.stream))
            gx.check(lib.gpx_trsm_back(dev.h, ptr(Utd), n, ld, ptr(xb), m, ldb, dev.stream))
            return xf, xb
        xf, xb = solves(B)
        xf2, xb2 = solves(B)
        assert torch.equal(xf, xf2) and torch.equal(xb, xb2), "repeat solves"
        for k in (-200, -20, 1, 20, 200):
            Us = Ad * 4.0 ** k
            assert potrf(gx, Us, n, ld) == 0
            assert torch.equal(torch.triu(Us[:, :n]), torch.triu(Ud[:, :n]) * 2.0 ** k), (nugget, k)
            sf, sb = solves(B * 2.0 ** k)
            assert torch.equal(sf, xf * 2.0 ** k) and torch.equal(sb, xb * 2.0 ** k), (nugget, k)
