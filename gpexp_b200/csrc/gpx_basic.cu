// HBM-bound kernels of the greedy design path: covariance evaluation (K1), incremental row append with
// running variance (K3+K4), arg-reduce with numpy tie-break (K7), pivot bookkeeping and the MI helpers (K6).
#include <math.h>

#include "gpx_common.cuh"

// ---------------------------------------------------------------------------------------------
// a1  pairwise k(X[j], Y[j]) with (1,d) broadcast                         kernels.py:49-65
// ---------------------------------------------------------------------------------------------
template <int FAM>
__global__ void __launch_bounds__(256) pairwise_kernel(const __grid_constant__ KParams kp, const double* __restrict__ X,
                                                        int64_t nx, int64_t ldx, const double* __restrict__ Y,
                                                        int64_t ny, int64_t ldy, double* __restrict__ out, int64_t n) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const int64_t jx = nx == 1 ? 0 : j;
    const int64_t jy = ny == 1 ? 0 : j;
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < GPX_MAX_DIM; ++i)
        if (i < kp.d) kacc_dim<FAM>(acc, kp, i, X[i * ldx + jx], Y[i * ldy + jy]);
    out[j] = kfinish<FAM>(acc, kp);
}

extern "C" int gpx_kernel_pairwise(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny,
                                   int64_t ldy, double* out, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(nx >= 0 && ny >= 0, GPX_EINVAL, "negative size");
    GPX_REQUIRE(nx == ny || nx == 1 || ny == 1, GPX_EINVAL,
                "point counts must match or one side must be a single point (kernels.py:58-63)");
    const int64_t n = nx > ny ? nx : ny;
    if (n == 0 || nx == 0 || ny == 0) return GPX_OK;
    GPX_REQUIRE(X && Y && out, GPX_EINVAL, "NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n + 255) / 256);
    GPX_DISPATCH_FAMILY(h->kp.family, (pairwise_kernel<FAM><<<grid, 256, 0, st>>>(h->kp, X, nx, ldx, Y, ny, ldy, out, n)));
    return gpx_check_launch("gpx_kernel_pairwise");
}

extern "C" int gpx_prior_diag(gpx_handle h, const double* X, int64_t n, int64_t ldx, double* out, void* stream) {
    return gpx_kernel_pairwise(h, X, n, ldx, X, n, ldx, out, stream);
}

// ---------------------------------------------------------------------------------------------
// K1  Gram block.  One thread owns one column j (its coordinates stay in registers), a block walks
// GRAM_ROWS rows whose coordinates sit in shared memory (broadcast reads); stores are coalesced in j.
// Algorithmic traffic: 8 B written per element (+ 8 d (nx+ny) read).
// ---------------------------------------------------------------------------------------------
#define GRAM_ROWS 16

// per-dimension weight folded into the coordinates of the SE instantiation: (x - y)^2 a/2 * 256/ln2 = ((x - y) w)^2
__device__ __forceinline__ double gram_se_weight(const KParams& kp, int q) { return sqrt(kp.a[q] * (0.5 * 0x1.71547652b82fep+8)); }

// GRAM_ROWS (or fewer) rows of two adjacent columns: covariance, optional nugget on the diagonal, streaming stores
template <int FAM, int D, bool DIAG, bool PAIR>
__device__ __forceinline__ void gram_rows(const KParams& kp, const double (&sx)[D][GRAM_ROWS], const double (&y0)[D],
                                          const double (&y1)[D], const double* __restrict__ s_tab, int rows, int64_t i0,
                                          int64_t j, double* __restrict__ dst, int64_t ld, const double* __restrict__ nugvec,
                                          double nug, bool second = true) {
    // rows in flight per thread: 4 for small d; fewer once 2*D coordinates + D-term sums fill the register file
    constexpr int RU = D <= 4 ? 4 : (D <= 8 ? 2 : 1);
#pragma unroll RU
    for (int r = 0; r < rows; ++r, dst += ld) {
        double a0 = 0.0, a1 = 0.0;
        double v0, v1;
        if (FAM == GPX_SE) {
            // weighted coordinates: one subtraction and one FMA per dimension, exponent already in table units
#pragma unroll
            for (int i = 0; i < D; ++i) {
                const double d0 = sx[i][r] - y0[i], d1 = sx[i][r] - y1[i];
                a0 = fma(d0, d0, a0);
                a1 = fma(d1, d1, a1);
            }
            v0 = gpx_exp_tab_scaled(a0, s_tab);
            v1 = gpx_exp_tab_scaled(a1, s_tab);
        } else {
#pragma unroll
            for (int i = 0; i < D; ++i) {
                kacc_dim<FAM>(a0, kp, i, sx[i][r], y0[i]);
                kacc_dim<FAM>(a1, kp, i, sx[i][r], y1[i]);
            }
            v0 = kfinish_tab<FAM>(a0, kp, s_tab);
            v1 = kfinish_tab<FAM>(a1, kp, s_tab);
        }
        if (DIAG) {
            const int64_t row = i0 + r;
            if (row == j) v0 += nugvec ? nugvec[row] : nug;
            if (row == j + 1) v1 += nugvec ? nugvec[row] : nug;
        }
        if (PAIR) {
            __stcs(reinterpret_cast<double2*>(dst), make_double2(v0, v1));
        } else {
            __stcs(dst, v0);
            if (second) __stcs(dst + 1, v1);
        }
    }
}

template <int FAM, int D, bool DIAG>
__global__ void __launch_bounds__(256, 1) gram_kernel(const __grid_constant__ KParams kp, const double* __restrict__ X,
                                                       int64_t nx, int64_t ldx, const double* __restrict__ Y, int64_t ny,
                                                       int64_t ldy, double* __restrict__ out, int64_t ld,
                                                       const double* __restrict__ nugvec, double nug, int vec2) {
    __shared__ double sx[D][GRAM_ROWS];
    __shared__ double s_tab[256];
    s_tab[threadIdx.x] = kp.signal * gpx_exp2_tab[threadIdx.x];
    // two adjacent columns per thread (16-byte streaming stores) when the output rows are 16-byte aligned
    const int64_t j = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 2;
    double y0[D], y1[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const double w = FAM == GPX_SE ? gram_se_weight(kp, i) : 1.0;
        y0[i] = (j < ny) ? Y[i * ldy + j] * w : 0.0;
        y1[i] = (j + 1 < ny) ? Y[i * ldy + j + 1] * w : 0.0;
    }
    for (int64_t i0 = (int64_t)blockIdx.y * GRAM_ROWS; i0 < nx; i0 += (int64_t)gridDim.y * GRAM_ROWS) {
        __syncthreads();
        if (threadIdx.x < GRAM_ROWS * D) {
            const int i = threadIdx.x / GRAM_ROWS, r = threadIdx.x % GRAM_ROWS;
            const double w = FAM == GPX_SE ? gram_se_weight(kp, i) : 1.0;
            sx[i][r] = (i0 + r < nx) ? X[i * ldx + i0 + r] * w : 0.0;
        }
        __syncthreads();
        if (j < ny) {
            const int rows = (nx - i0) < GRAM_ROWS ? (int)(nx - i0) : GRAM_ROWS;
            double* dst = out + i0 * ld + j;
            // the common case (aligned rows, both columns live) runs a branch-free loop with one 16-byte store per row
            if (vec2 && j + 1 < ny) {
                gram_rows<FAM, D, DIAG, true>(kp, sx, y0, y1, s_tab, rows, i0, j, dst, ld, nugvec, nug);
            } else {
                gram_rows<FAM, D, DIAG, false>(kp, sx, y0, y1, s_tab, rows, i0, j, dst, ld, nugvec, nug, j + 1 < ny);
            }
        }
    }
}

extern "C" int gpx_gram(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny, int64_t ldy,
                        double* out, int64_t ld, int add_diag, const double* nugget_vec, double nugget, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(nx >= 0 && ny >= 0 && ld >= ny, GPX_EINVAL, "bad sizes");
    if (nx == 0 || ny == 0) return GPX_OK;
    GPX_REQUIRE(X && Y && out, GPX_EINVAL, "NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t gy = (nx + GRAM_ROWS - 1) / GRAM_ROWS;
    if (gy > 32768) gy = 32768;
    dim3 grid((unsigned)((ny + 511) / 512), (unsigned)gy);
    const int vec2 = ((ld & 1) == 0 && gpx_aligned16(out)) ? 1 : 0;
    if (add_diag) {
        GPX_DISPATCH_FAMILY(h->kp.family, GPX_DISPATCH_DIM(h->kp.d, (gram_kernel<FAM, D, true><<<grid, 256, 0, st>>>(
                                                                        h->kp, X, nx, ldx, Y, ny, ldy, out, ld, nugget_vec, nugget, vec2))));
    } else {
        GPX_DISPATCH_FAMILY(h->kp.family, GPX_DISPATCH_DIM(h->kp.d, (gram_kernel<FAM, D, false><<<grid, 256, 0, st>>>(
                                                                        h->kp, X, nx, ldx, Y, ny, ldy, out, ld, nugget_vec, nugget, vec2))));
    }
    return gpx_check_launch("gpx_gram");
}

// ---------------------------------------------------------------------------------------------
// Prepared side for the tensor-core Gram prologue: k = f(e), e = sum over the d+2 rows of  A-row(i) * B-row(j).
//   SE      e = -1/2 sum a (x-y)^2        rows q<d: (a_q x_q) * y_q ;  alpha = -1/2 sum a x^2 ;  beta = -1/2 sum a y^2
//   MATERN  e = sum (x-y)^2               rows q<d: (-2 x_q) * y_q   ;  alpha = sum x^2        ;  beta = sum y^2
//           (every nu; MATERN12 reports maxabs = +inf, as it has no expanded form: see gpx_expanded_form)
//   MEHLER  e = -sum c (a x^2 - b x y + a y^2)   rows q<d: (c b x_q) * y_q ; alpha = -sum c a x^2 ; beta = -sum c a y^2
//   row d   : alpha_i on side A, 1 on side B       row d+1 : 1 on side A, beta_j on side B       rows > d+1 : 0
// For the stationary families the handle's centre is subtracted from every coordinate first (the kernel only sees
// x - y), which keeps |alpha|, |beta| -- the terms that cancel against sum u v -- as small as the data allow.
// maxabs (nullable): max_j |alpha_j| resp. |beta_j|, the number the host checks before trusting this form.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) prep_side_kernel(const __grid_constant__ KParams kp, const __grid_constant__ KCenter ctr,
                                                         int side, const double* __restrict__ X, int64_t n, int64_t ldx,
                                                         double* __restrict__ rows, int64_t ld,
                                                         unsigned long long* __restrict__ maxabs) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    double s = 0.0;
    if (j < ld) {
        const bool live = j < n;
#pragma unroll
        for (int i = 0; i < GPX_KROWS; ++i) {
            double r = 0.0;
            if (i < kp.d && live) {
                double x = X[i * ldx + j];
                if (kp.family == GPX_SE) {
                    x -= ctr.c[i];
                    s = fma(x * x, kp.a[i], s);
                    r = side == GPX_SIDE_A ? x * kp.a[i] : x;
                } else if (gpx_is_matern(kp.family)) {
                    x -= ctr.c[i];
                    s = fma(x, x, s);
                    r = side == GPX_SIDE_A ? -2.0 * x : x;
                } else if (kp.family == GPX_MEHLER) {
                    s = fma(x * x, kp.c[i] * kp.a[i], s);
                    r = side == GPX_SIDE_A ? kp.c[i] * kp.b[i] * x : x;
                }
            }
            if (i < kp.d) rows[i * ld + j] = r;
        }
        if (kp.family == GPX_SE) s *= -0.5;
        if (kp.family == GPX_MEHLER) s = -s;
        if (!live) s = 0.0;
        const double one = live ? 1.0 : 0.0;
        rows[(int64_t)kp.d * ld + j] = side == GPX_SIDE_A ? s : one;
        rows[(int64_t)(kp.d + 1) * ld + j] = side == GPX_SIDE_A ? one : s;
        for (int i = kp.d + 2; i < GPX_KROWS; ++i) rows[(int64_t)i * ld + j] = 0.0;
    }
    if (maxabs) {
        double m = gpx_expanded_form(kp.family) ? fabs(s) : INFINITY;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, off));
        // non-negative doubles order like their bit patterns
        if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(maxabs, (unsigned long long)__double_as_longlong(m));
    }
}

extern "C" int gpx_set_center(gpx_handle h, const double* center_host) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    for (int i = 0; i < GPX_MAX_DIM; ++i) h->center[i] = (center_host && h->has_kernel && i < h->kp.d) ? center_host[i] : 0.0;
    return GPX_OK;
}

extern "C" int gpx_prep_side(gpx_handle h, int side, const double* X, int64_t n, int64_t ldx, double* rows, int64_t ld,
                             double* maxabs, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(side == GPX_SIDE_A || side == GPX_SIDE_B, GPX_EINVAL, "bad side");
    GPX_REQUIRE(n >= 0 && ld >= n, GPX_EINVAL, "bad sizes");
    GPX_REQUIRE(h->kp.d + 2 <= GPX_KROWS, GPX_ESIZE, "the expanded form carries d + 2 rows: d <= GPX_KROWS - 2");
    if (ld == 0) return GPX_OK;
    GPX_REQUIRE(rows && (X || n == 0), GPX_EINVAL, "NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (maxabs) {
        cudaError_t e = cudaMemsetAsync(maxabs, 0, sizeof(double), st);
        if (e != cudaSuccess) {
            gpx_set_error("gpx_prep_side: cudaMemsetAsync: %s", cudaGetErrorString(e));
            return (int)e;
        }
    }
    KCenter ctr;
    for (int i = 0; i < GPX_MAX_DIM; ++i) ctr.c[i] = h->center[i];
    prep_side_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, st>>>(h->kp, ctr, side, X, n, ldx, rows, ld,
                                                                  reinterpret_cast<unsigned long long*>(maxabs));
    return gpx_check_launch("gpx_prep_side");
}

// ---------------------------------------------------------------------------------------------
// K7  arg-reduce and deterministic sum: per-block partials + last-block-done finish (one launch).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) argreduce_kernel(const double* __restrict__ v, const double* __restrict__ w,
                                                         const uint8_t* __restrict__ mask, int64_t n, int minimize,
                                                         double* red_val, int64_t* red_idx, unsigned int* counter,
                                                         double* best, int64_t* idx) {
    __shared__ double sv[8];
    __shared__ int64_t si[8];
    __shared__ bool last;
    const bool mn = minimize != 0;
    double bv = 0.0;
    int64_t bi = -1;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < n; j += (int64_t)gridDim.x * 256) {
        if (mask && mask[j]) continue;
        const double s = w ? v[j] * w[j] : v[j];
        if (gpx_better(s, j, bv, bi, mn)) {
            bv = s;
            bi = j;
        }
    }
    gpx_warp_argreduce(bv, bi, mn);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        sv[warp] = bv;
        si[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? sv[lane] : 0.0;
        bi = lane < 8 ? si[lane] : -1;
        gpx_warp_argreduce(bv, bi, mn);
        if (lane == 0) {
            red_val[blockIdx.x] = bv;
            red_idx[blockIdx.x] = bi;
            __threadfence();
            const unsigned int t = atomicAdd(counter, 1u);
            last = (t == gridDim.x - 1);
        }
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    bv = 0.0;
    bi = -1;
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += 256) {
        const double ov = __ldcg(red_val + b);
        const int64_t oi = __ldcg(red_idx + b);
        if (gpx_better(ov, oi, bv, bi, mn)) {
            bv = ov;
            bi = oi;
        }
    }
    gpx_warp_argreduce(bv, bi, mn);
    if (lane == 0) {
        sv[warp] = bv;
        si[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? sv[lane] : 0.0;
        bi = lane < 8 ? si[lane] : -1;
        gpx_warp_argreduce(bv, bi, mn);
        if (lane == 0) {
            best[0] = bv;
            idx[0] = bi;
            *counter = 0u;
        }
    }
}

int gpx_argreduce_impl(gpx_handle h, const double* v, const double* weights, const uint8_t* mask, int64_t n,
                       int minimize, double* best, int64_t* idx, cudaStream_t st) {
    int64_t blocks = (n + 1023) / 1024;
    if (blocks < 1) blocks = 1;
    if (blocks > GPX_RED_SLOTS) blocks = GPX_RED_SLOTS;
    argreduce_kernel<<<(unsigned)blocks, 256, 0, st>>>(v, weights, mask, n, minimize, h->red_val, h->red_idx,
                                                      h->red_counter, best, idx);
    return gpx_check_launch("gpx_argreduce");
}

extern "C" int gpx_argreduce(gpx_handle h, const double* v, const double* weights, const uint8_t* mask, int64_t n,
                             int minimize, double* best, int64_t* idx, void* stream) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    GPX_REQUIRE(n >= 0 && best && idx && (v || n == 0), GPX_EINVAL, "bad arguments");
    return gpx_argreduce_impl(h, v, weights, mask, n, minimize, best, idx, (cudaStream_t)stream);
}

__device__ __forceinline__ double gpx_block_sum(double s, double* sm) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sm[warp] = s;
    __syncthreads();
    double t = 0.0;
    if (warp == 0) {
        t = lane < 8 ? sm[lane] : 0.0;
#pragma unroll
        for (int off = 4; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
    }
    return t;  // valid in warp 0
}

// WT: out = sum_j w[j] v[j] in the same tree (one fma per term in place of the add)
template <bool WT>
__global__ void __launch_bounds__(256) sum_kernel(const double* __restrict__ v, const double* __restrict__ w, int64_t n,
                                                   double* red_val, unsigned int* counter, double* out) {
    __shared__ double sm[8];
    __shared__ bool last;
    double s = 0.0;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < n; j += (int64_t)gridDim.x * 256) {
        if (WT) s = fma(w[j], v[j], s);
        else s += v[j];
    }
    s = gpx_block_sum(s, sm);
    if (threadIdx.x == 0) {
        red_val[blockIdx.x] = s;
        __threadfence();
        last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    s = 0.0;
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += 256) s += __ldcg(red_val + b);
    s = gpx_block_sum(s, sm);
    if (threadIdx.x == 0) {
        out[0] = s;
        *counter = 0u;
    }
}

int gpx_sum_impl(gpx_handle h, const double* v, const double* w, int64_t n, double* out, cudaStream_t st) {
    int64_t blocks = (n + 4095) / 4096;
    if (blocks < 1) blocks = 1;
    if (blocks > 1024) blocks = 1024;
    // slots [1024, 2048) of the scratch and ticket 1, so that a sum can sit next to an arg-reduce
    if (w) sum_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(v, w, n, h->red_val + 1024, h->red_counter + 1, out);
    else sum_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(v, w, n, h->red_val + 1024, h->red_counter + 1, out);
    return gpx_check_launch("gpx_sum");
}

extern "C" int gpx_sum(gpx_handle h, const double* v, int64_t n, double* out, void* stream) {
    GPX_REQUIRE(h != nullptr && out && n >= 0 && (v || n == 0), GPX_EINVAL, "bad arguments");
    return gpx_sum_impl(h, v, nullptr, n, out, (cudaStream_t)stream);
}

extern "C" int gpx_sum_w(gpx_handle h, const double* v, const double* w, int64_t n, double* out, void* stream) {
    GPX_REQUIRE(h != nullptr && out && n >= 0 && (v || n == 0), GPX_EINVAL, "bad arguments");
    return gpx_sum_impl(h, v, w, n, out, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// K3+K4 incremental row append.  Two adjacent columns per thread (16-byte streaming loads), the pivot's
// W-column in shared memory, 16 independent loads in flight per thread (gpx_append_two_columns).  Reads 8*n*ncols bytes.
// ---------------------------------------------------------------------------------------------
template <int FAM, int SRC, int NT>
__global__ void __launch_bounds__(NT) append_row_kernel(const __grid_constant__ KParams kp, const double* __restrict__ rec,
                                                          const double* __restrict__ src_row, const double* __restrict__ Y,
                                                          int64_t ncols, int64_t ldy, double* __restrict__ W, int64_t ldw,
                                                          int n, double* __restrict__ var) {
    extern __shared__ double sl[];
    const int64_t j = ((int64_t)blockIdx.x * NT + threadIdx.x) * 2;
    gpx_append_two_columns<FAM, SRC == GPX_ROW_KERNEL>(kp, rec, src_row, Y, ncols, ldy, W, ldw, n, var, j, sl, NT);
}

extern "C" int gpx_append_row(gpx_handle h, int row_source, const double* rec, const double* src_row, const double* Y,
                              int64_t ncols, int64_t ldy, double* W, int64_t ldw, int64_t n, double* var, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(row_source == GPX_ROW_KERNEL || row_source == GPX_ROW_MATRIX, GPX_EINVAL, "bad row source");
    GPX_REQUIRE(ncols >= 0 && n >= 0, GPX_EINVAL, "negative size");
    if (ncols == 0) return GPX_OK;
    GPX_REQUIRE(rec && W && var, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE((ldw % 2) == 0 && ldw >= ncols + (ncols & 1), GPX_EALIGN, "ldw must be even and cover an even column count");
    GPX_REQUIRE(gpx_aligned16(W), GPX_EALIGN, "W must be 16-byte aligned");
    if (row_source == GPX_ROW_KERNEL) {
        GPX_REQUIRE(Y != nullptr, GPX_EINVAL, "Y is NULL");
        GPX_REQUIRE((ldy % 2) == 0 && ldy >= ncols + (ncols & 1) && gpx_aligned16(Y), GPX_EALIGN,
                    "Y must be 16-byte aligned with an even leading dimension");
    } else {
        GPX_REQUIRE(src_row != nullptr && gpx_aligned16(src_row), GPX_EALIGN, "src_row must be 16-byte aligned");
    }
    const size_t smem = (size_t)((n + 15) / 16 * 16) * sizeof(double);
    GPX_REQUIRE(smem <= 200 * 1024, GPX_ESIZE, "design size exceeds the shared-memory column buffer (25600)");
    cudaStream_t st = (cudaStream_t)stream;
    // 256 columns per 128-thread block.  (Measured in round 2: 64-thread blocks for narrow problems change nothing --
    // 48.1 vs 46 us at n = 255, C = 1e5: the 31 us of streaming sit between ~15 us of launch, ramp and tail.)
    const unsigned grid = (unsigned)((ncols + 255) / 256);
#define GPX_APPEND_LAUNCH(F, S)                                                                                      \
    do {                                                                                                             \
        if (smem > 48 * 1024) {                                                                                      \
            const int rc_ = gpx_ensure_smem(h, (const void*)append_row_kernel<F, S, 128>, 200 * 1024, "append_row"); \
            if (rc_) return rc_;                                                                                     \
        }                                                                                                            \
        append_row_kernel<F, S, 128><<<grid, 128, smem, st>>>(h->kp, rec, src_row, Y, ncols, ldy, W, ldw, (int)n, var); \
    } while (0)
    if (row_source == GPX_ROW_KERNEL) {
        GPX_DISPATCH_FAMILY(h->kp.family, GPX_APPEND_LAUNCH(FAM, GPX_ROW_KERNEL));
    } else {
        GPX_APPEND_LAUNCH(GPX_SE, GPX_ROW_MATRIX);
    }
#undef GPX_APPEND_LAUNCH
    return gpx_check_launch("gpx_append_row");
}

// ---------------------------------------------------------------------------------------------
// Pivot bookkeeping (single small blocks; latency only)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_pivot_kernel(const double* __restrict__ W, int64_t ldw, int n,
                                                            const double* __restrict__ var, const double* __restrict__ X,
                                                            int64_t ldx, int d, const double* __restrict__ score,
                                                            const int64_t* __restrict__ idx, int64_t offset,
                                                            const int64_t* __restrict__ index_map,
                                                            const double* __restrict__ nu, double noise,
                                                            double* __restrict__ rec) {
    const int64_t p = idx[0];
    if (p < 0) {
        if (threadIdx.x == 0 && blockIdx.x == 0) {
            rec[0] = score ? score[0] : 0.0;
            rec[1] = -1.0;
            rec[2] = 1.0;
        }
        return;
    }
    if (blockIdx.x == 0) {
        if (threadIdx.x == 0) {
            rec[0] = score ? score[0] : 0.0;
            rec[1] = (double)(index_map ? index_map[p] : p + offset);
            rec[2] = var[p] + (nu ? nu[p] : noise);
        }
        if (threadIdx.x < GPX_MAX_DIM) rec[3 + threadIdx.x] = threadIdx.x < d ? X[threadIdx.x * ldx + p] : 0.0;
    }
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) rec[GPX_PIVOT_HDR + i] = W[(int64_t)i * ldw + p];
}

static int gather_pivot_impl(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var, const double* X,
                             int64_t ldx, const double* score_dev, const int64_t* idx_dev, int64_t index_offset,
                             const int64_t* index_map, const double* nu, double noise, double* rec, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(n >= 0 && var && X && idx_dev && rec && (W || n == 0), GPX_EINVAL, "bad arguments");
    unsigned grid = (unsigned)((n + 255) / 256);
    if (grid < 1) grid = 1;
    if (grid > 64) grid = 64;
    gather_pivot_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, (int)n, var, X, ldx, h->kp.d, score_dev, idx_dev,
                                                              index_offset, index_map, nu, noise, rec);
    return gpx_check_launch("gpx_gather_pivot");
}

extern "C" int gpx_gather_pivot(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var, const double* X,
                                int64_t ldx, const double* score_dev, const int64_t* idx_dev, int64_t index_offset,
                                const int64_t* index_map, double noise, double* rec, void* stream) {
    return gather_pivot_impl(h, W, ldw, n, var, X, ldx, score_dev, idx_dev, index_offset, index_map, nullptr, noise, rec,
                             stream);
}

extern "C" int gpx_gather_pivot_nu(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var,
                                   const double* X, int64_t ldx, const double* score_dev, const int64_t* idx_dev,
                                   int64_t index_offset, const int64_t* index_map, const double* nu, double noise,
                                   double* rec, void* stream) {
    return gather_pivot_impl(h, W, ldw, n, var, X, ldx, score_dev, idx_dev, index_offset, index_map, nu, noise, rec, stream);
}

__global__ void __launch_bounds__(256) select_pivot_kernel(const double* __restrict__ recs, int nrec, int64_t stride, int n,
                                                            int minimize, double* __restrict__ out) {
    __shared__ int win;
    if (threadIdx.x == 0) {
        double bv = 0.0;
        int64_t bi = -1;
        int bw = 0;
        for (int r = 0; r < nrec; ++r) {
            const double v = recs[r * stride];
            const int64_t i = (int64_t)recs[r * stride + 1];
            if (gpx_better(v, i, bv, bi, minimize != 0)) {
                bv = v;
                bi = i;
                bw = r;
            }
        }
        win = bw;
    }
    __syncthreads();
    const double* src = recs + (int64_t)win * stride;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < GPX_PIVOT_HDR + n; i += gridDim.x * 256) out[i] = src[i];
}

extern "C" int gpx_select_pivot(gpx_handle h, const double* recs, int nrec, int64_t stride, int64_t n, int minimize,
                                double* rec_out, void* stream) {
    GPX_REQUIRE(h && recs && rec_out && nrec >= 1 && n >= 0 && stride >= GPX_PIVOT_HDR + n, GPX_EINVAL, "bad arguments");
    unsigned grid = (unsigned)((GPX_PIVOT_HDR + n + 255) / 256);
    if (grid > 64) grid = 64;
    select_pivot_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(recs, nrec, stride, (int)n, minimize, rec_out);
    return gpx_check_launch("gpx_select_pivot");
}

__global__ void __launch_bounds__(256) store_pivot_kernel(const double* __restrict__ rec, int n, double* U, int64_t ldu,
                                                           int64_t* picks, double* scores, double* pivots) {
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256)
        if (U) U[(int64_t)i * ldu + n] = rec[GPX_PIVOT_HDR + i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (U) U[(int64_t)n * ldu + n] = sqrt(rec[2]);
        if (picks) picks[n] = (int64_t)rec[1];
        if (scores) scores[n] = rec[0];
        if (pivots) pivots[n] = rec[2];
    }
}

extern "C" int gpx_store_pivot(gpx_handle h, const double* rec, int64_t n, double* U, int64_t ldu, int64_t* picks,
                               double* scores, double* pivots, void* stream) {
    GPX_REQUIRE(h && rec && n >= 0, GPX_EINVAL, "bad arguments");
    unsigned grid = (unsigned)((n + 255) / 256);
    if (grid < 1) grid = 1;
    if (grid > 64) grid = 64;
    store_pivot_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rec, (int)n, U, ldu, picks, scores, pivots);
    return gpx_check_launch("gpx_store_pivot");
}

__global__ void set_mask_kernel(uint8_t* mask, const int64_t* idx, uint8_t value) {
    if (idx[0] >= 0) mask[idx[0]] = value;
}

extern "C" int gpx_set_mask(gpx_handle h, uint8_t* mask, const int64_t* idx_dev, uint8_t value, void* stream) {
    GPX_REQUIRE(h && mask && idx_dev, GPX_EINVAL, "bad arguments");
    set_mask_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(mask, idx_dev, value);
    return gpx_check_launch("gpx_set_mask");
}

// ---------------------------------------------------------------------------------------------
// K4  column sums of squares (posterior variance from a materialised W)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) colsumsq_kernel(const double* __restrict__ W, int64_t n, int64_t ncols, int64_t ldw,
                                                        const double* __restrict__ base, double* __restrict__ out) {
    const int64_t j = ((int64_t)blockIdx.x * 128 + threadIdx.x) * 2;
    if (j >= ncols) return;
    double a0 = 0.0, a1 = 0.0;
    int64_t i = 0;
    for (; i + 4 <= n; i += 4) {
        double2 w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const double2*>(W + (i + u) * ldw + j);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            a0 = fma(w[u].x, w[u].x, a0);
            a1 = fma(w[u].y, w[u].y, a1);
        }
    }
    for (; i < n; ++i) {
        const double2 w = *reinterpret_cast<const double2*>(W + i * ldw + j);
        a0 = fma(w.x, w.x, a0);
        a1 = fma(w.y, w.y, a1);
    }
    out[j] = base ? base[j] - a0 : a0;
    if (j + 1 < ncols) out[j + 1] = base ? base[j + 1] - a1 : a1;
}

extern "C" int gpx_colsumsq(gpx_handle h, const double* W, int64_t n, int64_t ncols, int64_t ldw, const double* base,
                            double* out, void* stream) {
    GPX_REQUIRE(h && out && n >= 0 && ncols >= 0, GPX_EINVAL, "bad arguments");
    if (ncols == 0) return GPX_OK;
    GPX_REQUIRE(W || n == 0, GPX_EINVAL, "W is NULL");
    GPX_REQUIRE(n == 0 || ((ldw % 2) == 0 && ldw >= ncols + (ncols & 1) && gpx_aligned16(W)), GPX_EALIGN,
                "W must be 16-byte aligned with an even leading dimension");
    colsumsq_kernel<<<(unsigned)((ncols + 255) / 256), 128, 0, (cudaStream_t)stream>>>(W, n, ncols, ldw, base, out);
    return gpx_check_launch("gpx_colsumsq");
}

// ---------------------------------------------------------------------------------------------
// transpose (row-major points (n,d) <-> dimension-major (d,ld), and U <-> U^T)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_kernel(const double* __restrict__ in, int64_t rows, int64_t cols,
                                                         int64_t ld_in, double* __restrict__ out, int64_t ld_out) {
    __shared__ double tile[32][33];
    const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8)
        if (r0 + r < rows && c0 + tx < cols) tile[r][tx] = in[(r0 + r) * ld_in + c0 + tx];
    __syncthreads();
    for (int c = ty; c < 32; c += 8)
        if (c0 + c < cols && r0 + tx < rows) out[(c0 + c) * ld_out + r0 + tx] = tile[tx][c];
}

extern "C" int gpx_transpose(gpx_handle h, const double* in, int64_t rows, int64_t cols, int64_t ld_in, double* out,
                             int64_t ld_out, void* stream) {
    GPX_REQUIRE(h && rows >= 0 && cols >= 0, GPX_EINVAL, "bad arguments");
    if (rows == 0 || cols == 0) return GPX_OK;
    GPX_REQUIRE(in && out && ld_in >= cols && ld_out >= rows, GPX_EINVAL, "bad arguments");
    const int64_t gy = (rows + 31) / 32;
    if (gy <= 65535) {
        dim3 grid((unsigned)((cols + 31) / 32), (unsigned)gy);
        transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, rows, cols, ld_in, out, ld_out);
    } else {
        // tall input (points (n,d) with huge n): walk the rows in slabs
        const int64_t slab = 65535LL * 32;
        for (int64_t r0 = 0; r0 < rows; r0 += slab) {
            const int64_t rr = rows - r0 < slab ? rows - r0 : slab;
            dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rr + 31) / 32));
            transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in + r0 * ld_in, rr, cols, ld_in, out + r0, ld_out);
        }
    }
    return gpx_check_launch("gpx_transpose");
}

// ---------------------------------------------------------------------------------------------
// K6  mutual-information helpers
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) score_mi_kernel(const double* __restrict__ num, const double* __restrict__ pd,
                                                        const double* __restrict__ nu, double noise,
                                                        const uint8_t* __restrict__ mask, int64_t n,
                                                        double* __restrict__ score) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    if (mask && mask[j]) {
        score[j] = -INFINITY;
        return;
    }
    const double den = 1.0 / pd[j] - (nu ? nu[j] : noise);  // var(y | V minus A minus y)   experimentalDesign.py:277-281
    score[j] = num[j] / den;                                 // :284
}

static int score_mi_impl(gpx_handle h, const double* num_var, const double* prec_diag, const double* nu, double noise,
                         const uint8_t* mask, int64_t n, double* score_out, double* best, int64_t* idx, void* stream) {
    GPX_REQUIRE(h && num_var && prec_diag && score_out && best && idx && n >= 1, GPX_EINVAL, "bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    score_mi_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(num_var, prec_diag, nu, noise, mask, n, score_out);
    int rc = gpx_check_launch("gpx_score_mi");
    if (rc) return rc;
    return gpx_argreduce_impl(h, score_out, nullptr, mask, n, 0, best, idx, st);
}

extern "C" int gpx_score_mi(gpx_handle h, const double* num_var, const double* prec_diag, double noise,
                            const uint8_t* mask, int64_t n, double* score_out, double* best, int64_t* idx, void* stream) {
    return score_mi_impl(h, num_var, prec_diag, nullptr, noise, mask, n, score_out, best, idx, stream);
}

extern "C" int gpx_score_mi_nu(gpx_handle h, const double* num_var, const double* prec_diag, const double* nu,
                               double noise, const uint8_t* mask, int64_t n, double* score_out, double* best, int64_t* idx,
                               void* stream) {
    return score_mi_impl(h, num_var, prec_diag, nu, noise, mask, n, score_out, best, idx, stream);
}

// out[i] = sum_{k >= max(i,p)} Y[k,i] * Y[k,p]   (Y lower triangular, row-major).  Reads ~4 n^2 bytes.
// 2-D decomposition: a block owns 256 columns x MI_KCH rows and writes one partial per column; the partials
// are added in row-chunk order by a second kernel (deterministic).  Blocks above the diagonal write zeros.
#define MI_KCH 256

// global column of local column i: contiguous slice (blk = 0: i + col_offset) or block-cyclic (local block i / blk of rank
// `col_offset` among `world` ranks is global block (i / blk) * world + col_offset)
__device__ __forceinline__ int64_t mi_global_col(int64_t i, int64_t col_offset, int64_t blk, int64_t world) {
    return blk > 0 ? ((i / blk) * world + col_offset) * blk + (i % blk) : i + col_offset;
}

__global__ void __launch_bounds__(128) mi_prec_partial_kernel(const double* __restrict__ Y, int64_t nrows, int64_t ncols,
                                                               int64_t ldy, int64_t col_offset, int64_t blk, int64_t world,
                                                               const int64_t* __restrict__ pdev,
                                                               const double* __restrict__ ycol, double* __restrict__ part) {
    __shared__ double syp[MI_KCH];
    const int64_t p = pdev[0];  // GLOBAL index of the pivot column
    const int64_t i = ((int64_t)blockIdx.x * 128 + threadIdx.x) * 2;  // local column
    const int64_t k0 = (int64_t)blockIdx.y * MI_KCH;
    int64_t k1 = k0 + MI_KCH;
    if (k1 > nrows) k1 = nrows;
    double* dst = part + (int64_t)blockIdx.y * ldy;
    // smallest global column of the block (256 local columns never straddle a cyclic block: blk is a multiple of 256 or 0)
    const int64_t i0g = mi_global_col((int64_t)blockIdx.x * 256, col_offset, blk, world);
    const int64_t lo_blk = i0g > p ? i0g : p;
    if (p < 0 || k1 <= lo_blk) {  // nothing in this row chunk reaches these columns
        if (i < ncols) {
            dst[i] = 0.0;
            if (i + 1 < ncols) dst[i + 1] = 0.0;
        }
        return;
    }
    // column p of Y: from the dense vector when given (sharded pools), else from the local matrix
    for (int t = threadIdx.x; t < MI_KCH; t += 128)
        syp[t] = (k0 + t < k1) ? (ycol ? ycol[k0 + t] : Y[(k0 + t) * ldy + (p - col_offset)]) : 0.0;  // ycol == NULL: dense, blk == 0
    __syncthreads();
    if (i >= ncols) return;
    const int64_t ig = mi_global_col(i, col_offset, blk, world);
    int64_t k = ig > p ? ig : p;  // column i+1 also starts here: Y[i, i+1] = 0 is stored explicitly
    if (k < k0) k = k0;
    double a0 = 0.0, a1 = 0.0;
    for (; k + 4 <= k1; k += 4) {
        double2 y[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) y[u] = __ldcs(reinterpret_cast<const double2*>(Y + (k + u) * ldy + i));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double yp = syp[k + u - k0];
            a0 = fma(y[u].x, yp, a0);
            a1 = fma(y[u].y, yp, a1);
        }
    }
    for (; k < k1; ++k) {
        const double2 y = __ldcs(reinterpret_cast<const double2*>(Y + k * ldy + i));
        const double yp = syp[k - k0];
        a0 = fma(y.x, yp, a0);
        a1 = fma(y.y, yp, a1);
    }
    dst[i] = a0;
    if (i + 1 < ncols) dst[i + 1] = a1;
}

__global__ void __launch_bounds__(256) mi_prec_reduce_kernel(const double* __restrict__ part, int nchunks, int64_t n,
                                                              int64_t ldy, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += part[(int64_t)c * ldy + i];
    out[i] = s;
}

extern "C" int64_t gpx_mi_prec_column_workspace(int64_t nrows, int64_t ldy) {
    if (nrows <= 0) return 0;
    return ((nrows + MI_KCH - 1) / MI_KCH) * ldy;
}

extern "C" int gpx_mi_prec_column(gpx_handle h, const double* Y, int64_t nrows, int64_t ncols, int64_t ldy,
                                  int64_t col_offset, int64_t cyclic_blk, int64_t cyclic_world, const int64_t* p_dev,
                                  const double* ycol, double* workspace, double* out, void* stream) {
    GPX_REQUIRE(h && Y && p_dev && out && workspace && nrows >= 1 && ncols >= 1 && col_offset >= 0, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(cyclic_blk == 0 || (cyclic_blk % 256 == 0 && cyclic_world >= 1 && col_offset < cyclic_world && ycol != nullptr),
                GPX_EINVAL, "block-cyclic slices: blk a multiple of 256, col_offset = rank < world, pivot column as a vector");
    GPX_REQUIRE((ldy % 2) == 0 && ldy >= ncols + (ncols & 1) && gpx_aligned16(Y), GPX_EALIGN,
                "Y must be 16-byte aligned with an even leading dimension");
    GPX_REQUIRE(ycol != nullptr || (col_offset == 0 && ncols == nrows), GPX_EINVAL,
                "a column slice of Y needs the pivot column as a dense vector");
    const int64_t nchunks = (nrows + MI_KCH - 1) / MI_KCH;
    GPX_REQUIRE(nchunks <= 65535, GPX_ESIZE, "pool too large for one launch");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)((ncols + 255) / 256), (unsigned)nchunks);
    mi_prec_partial_kernel<<<grid, 128, 0, st>>>(Y, nrows, ncols, ldy, col_offset, cyclic_blk, cyclic_world, p_dev, ycol,
                                                 workspace);
    int rc = gpx_check_launch("gpx_mi_prec_column partial");
    if (rc) return rc;
    mi_prec_reduce_kernel<<<(unsigned)((ncols + 255) / 256), 256, 0, st>>>(workspace, (int)nchunks, ncols, ldy, out);
    return gpx_check_launch("gpx_mi_prec_column reduce");
}

// rec[2] = var[p] (if var), rec[HDR + i] = W[i, p] for i < n; no-op when *idx < 0 (the caller zeroes rec first:
// the record is then summed across ranks, only the owner of p contributes)
__global__ void __launch_bounds__(256) gather_column_kernel(const double* __restrict__ W, int64_t ldw, int64_t n,
                                                             const double* __restrict__ var, const int64_t* __restrict__ idx,
                                                             double* __restrict__ rec) {
    const int64_t p = idx[0];
    if (p < 0) return;
    if (blockIdx.x == 0 && threadIdx.x == 0 && var) rec[2] = var[p];
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        rec[GPX_PIVOT_HDR + i] = W[i * ldw + p];
}

extern "C" int gpx_gather_column(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var,
                                 const int64_t* idx_dev, double* rec, void* stream) {
    GPX_REQUIRE(h && idx_dev && rec && n >= 0 && (W || n == 0), GPX_EINVAL, "bad arguments");
    int64_t grid = (n + 255) / 256;
    if (grid < 1) grid = 1;
    if (grid > 1024) grid = 1024;
    gather_column_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, n, var, idx_dev, rec);
    return gpx_check_launch("gpx_gather_column");
}

// local index of a global pivot: out[0] = rec[1] - offset if it falls in [0, count), else -1
__global__ void local_index_kernel(const double* __restrict__ rec, int64_t offset, int64_t count, int64_t* out) {
    const int64_t g = (int64_t)rec[1] - offset;
    out[0] = (rec[1] >= 0.0 && g >= 0 && g < count) ? g : -1;
    out[1] = (int64_t)rec[1];
}

extern "C" int gpx_local_index(gpx_handle h, const double* rec, int64_t offset, int64_t count, int64_t* out2, void* stream) {
    GPX_REQUIRE(h && rec && out2, GPX_EINVAL, "bad arguments");
    local_index_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(rec, offset, count, out2);
    return gpx_check_launch("gpx_local_index");
}

// block-cyclic ownership: global index g lives on rank (g / blk) % world at local index ((g / blk) / world) * blk + g % blk
__global__ void local_index_cyclic_kernel(const double* __restrict__ rec, int64_t blk, int64_t world, int64_t rank, int64_t count,
                                          int64_t* out) {
    const int64_t g = (int64_t)rec[1];
    int64_t loc = -1;
    if (rec[1] >= 0.0 && (g / blk) % world == rank) {
        loc = ((g / blk) / world) * blk + g % blk;
        if (loc >= count) loc = -1;
    }
    out[0] = loc;
    out[1] = g;
}

extern "C" int gpx_local_index_cyclic(gpx_handle h, const double* rec, int64_t blk, int64_t world, int64_t rank, int64_t count,
                                      int64_t* out2, void* stream) {
    GPX_REQUIRE(h && rec && out2 && blk >= 1 && world >= 1 && rank >= 0 && rank < world, GPX_EINVAL, "bad arguments");
    local_index_cyclic_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(rec, blk, world, rank, count, out2);
    return gpx_check_launch("gpx_local_index_cyclic");
}

// A[rows[j] * ld + j] += vals ? vals[j] : value for j < n : the diagonal of a matrix whose columns are a scattered subset
// of a square one
__global__ void __launch_bounds__(256) add_at_rows_kernel(double* __restrict__ A, int64_t ld, const int64_t* __restrict__ rows,
                                                           int64_t n, const double* __restrict__ vals, double value) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j < n) A[rows[j] * ld + j] += vals ? vals[j] : value;
}

static int add_at_rows_impl(gpx_handle h, double* A, int64_t ld, const int64_t* rows, int64_t n, const double* vals,
                            double value, void* stream) {
    GPX_REQUIRE(h && n >= 0, GPX_EINVAL, "bad arguments");
    if (n == 0) return GPX_OK;
    GPX_REQUIRE(A && rows && ld >= n, GPX_EINVAL, "bad arguments");
    add_at_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A, ld, rows, n, vals, value);
    return gpx_check_launch("gpx_add_at_rows");
}

extern "C" int gpx_add_at_rows(gpx_handle h, double* A, int64_t ld, const int64_t* rows, int64_t n, double value, void* stream) {
    return add_at_rows_impl(h, A, ld, rows, n, nullptr, value, stream);
}

extern "C" int gpx_add_at_rows_vec(gpx_handle h, double* A, int64_t ld, const int64_t* rows, int64_t n, const double* vals,
                                   double value, void* stream) {
    return add_at_rows_impl(h, A, ld, rows, n, vals, value, stream);
}


// ---------------------------------------------------------------------------------------------
// Resident posterior covariance (the O(M*C) bytes/step alternative to the per-step contraction, SURVEY.md section 7):
//     cov[m,c] = k(m,c) - sum_{i<n} W_M[i,m] W_C[i,c]   is kept in HBM (8*M*C bytes) and every greedy step applies
//     cov -= a b^T   (a = the new row of W_M, b = the new row of W_C)  while accumulating  r[c] = sum_m cov[m,c]^2
// in the same pass: 16 bytes of HBM traffic per (m,c) pair and step, independent of the design size n.
// Block = 512 columns (16-byte accesses) x one row segment; per-segment partial sums are added in a fixed order.
// WT: weighted integration points, r[c] = sum_m fma(wM[m] cov[m,c], cov[m,c], r) (w = 2^-k scales r exactly).
// ---------------------------------------------------------------------------------------------
#define COV_MAX_SEG 160

template <bool WT>
__global__ void __launch_bounds__(256) cov_update_kernel(double* __restrict__ cov, int64_t ldc, int64_t M, int64_t C,
                                                          const double* __restrict__ a, const double* __restrict__ b,
                                                          const double* __restrict__ wM, int64_t rows_per_seg,
                                                          double* __restrict__ part, int64_t ldp) {
    const int64_t c = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 2;
    if (c >= C) return;
    const int64_t m0 = (int64_t)blockIdx.y * rows_per_seg;
    int64_t m1 = m0 + rows_per_seg;
    if (m1 > M) m1 = M;
    const bool upd = (a != nullptr);
    double b0 = 0.0, b1 = 0.0;
    if (upd) {
        const double2 bb = *reinterpret_cast<const double2*>(b + c);
        b0 = bb.x;
        b1 = bb.y;
    }
    double r0 = 0.0, r1 = 0.0;
    double* p = cov + m0 * ldc + c;
    int64_t m = m0;
    for (; m + 8 <= m1; m += 8) {
        double2 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldcs(reinterpret_cast<const double2*>(p + (int64_t)u * ldc));
        if (upd) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const double am = __ldg(a + m + u);
                v[u].x = fma(-am, b0, v[u].x);
                v[u].y = fma(-am, b1, v[u].y);
                __stcs(reinterpret_cast<double2*>(p + (int64_t)u * ldc), v[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (WT) {
                const double wm = __ldg(wM + m + u);
                r0 = fma(wm * v[u].x, v[u].x, r0);
                r1 = fma(wm * v[u].y, v[u].y, r1);
            } else {
                r0 = fma(v[u].x, v[u].x, r0);
                r1 = fma(v[u].y, v[u].y, r1);
            }
        }
        p += 8 * ldc;
    }
    for (; m < m1; ++m) {
        double2 v = __ldcs(reinterpret_cast<const double2*>(p));
        if (upd) {
            const double am = __ldg(a + m);
            v.x = fma(-am, b0, v.x);
            v.y = fma(-am, b1, v.y);
            __stcs(reinterpret_cast<double2*>(p), v);
        }
        if (WT) {
            const double wm = __ldg(wM + m);
            r0 = fma(wm * v.x, v.x, r0);
            r1 = fma(wm * v.y, v.y, r1);
        } else {
            r0 = fma(v.x, v.x, r0);
            r1 = fma(v.y, v.y, r1);
        }
        p += ldc;
    }
    double* dst = part + (int64_t)blockIdx.y * ldp + c;
    dst[0] = r0;
    if (c + 1 < C) dst[1] = r1;
}

extern "C" int gpx_cov_segments(int64_t M, int64_t C) {
    // row segments: ~2048 rows each for wide candidate sets; more (down to 64 rows) when few 512-column blocks would
    // otherwise leave most of the 148 SMs idle (cfg-1: 1 000 candidates = 2 column blocks)
    int64_t s = (M + 2047) / 2048;
    const int64_t colblocks = (C + 511) / 512;
    if (colblocks > 0 && s * colblocks < 2 * 148) {
        s = (2 * 148 + colblocks - 1) / colblocks;
        const int64_t cap = (M + 63) / 64;
        if (s > cap) s = cap;
    }
    if (s < 1) s = 1;
    if (s > COV_MAX_SEG) s = COV_MAX_SEG;
    return (int)s;
}

extern "C" int gpx_cov_update_w(gpx_handle h, double* cov, int64_t ldc, int64_t M, int64_t C, const double* a, const double* b,
                                const double* wM, double* partial, int64_t ldp, void* stream) {
    GPX_REQUIRE(h && cov && partial && M >= 1 && C >= 1, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE((a == nullptr) == (b == nullptr), GPX_EINVAL, "a and b must both be given or both be NULL");
    GPX_REQUIRE((ldc % 2) == 0 && ldc >= C + (C & 1) && gpx_aligned16(cov), GPX_EALIGN,
                "cov must be 16-byte aligned with an even leading dimension");
    GPX_REQUIRE(b == nullptr || gpx_aligned16(b), GPX_EALIGN, "b must be 16-byte aligned");
    GPX_REQUIRE(ldp >= C, GPX_EINVAL, "partial rows too short");
    const int seg = gpx_cov_segments(M, C);
    const int64_t rows = (M + seg - 1) / seg;
    dim3 grid((unsigned)((C + 511) / 512), (unsigned)seg);
    if (wM) cov_update_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(cov, ldc, M, C, a, b, wM, rows, partial, ldp);
    else cov_update_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(cov, ldc, M, C, a, b, wM, rows, partial, ldp);
    return gpx_check_launch("gpx_cov_update");
}

extern "C" int gpx_cov_update(gpx_handle h, double* cov, int64_t ldc, int64_t M, int64_t C, const double* a, const double* b,
                              double* partial, int64_t ldp, void* stream) {
    return gpx_cov_update_w(h, cov, ldc, M, C, a, b, nullptr, partial, ldp, stream);
}
