// SURVEY.md section 8(f) widening: what the continuous optimisers call on top of the hot path --
// the marginal log-likelihood (gp.py:394-446) and the gradient of the posterior variance / IVAR cost with
// respect to the design coordinates (experimentalDesign.py:148-179 -> gp.py:282-341 -> kernels.py:146-181).
// Squared-exponential kernels only: the reference defines `derivative` for SE (and 1-D Mehler), raises for
// Mehler-ND and has none for Matern.
#include <math.h>

#include "gpx_common.cuh"

// D(u, v)[k] = "dK(u, v)/du_k" exactly as kernels.py:176-180 computes it:
//     -signalSize * (u_k - v_k) / cl_k^2 * evaluate(u, v)      (evaluate already carries signalSize)
template <int D>
__global__ void __launch_bounds__(256) se_dgram_kernel(const __grid_constant__ KParams kp, const double* __restrict__ X,
                                                        int64_t nx, int64_t ldx, const double* __restrict__ Y, int64_t ny,
                                                        int64_t ldy, double* __restrict__ out, int64_t ld) {
    // out[i, j*D + k] = D(y_j, x_i)[k] ; one thread per (i, j)
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t i = blockIdx.y;
    if (j >= ny || i >= nx) return;
    double acc = 0.0, df[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        df[q] = Y[q * ldy + j] - X[q * ldx + i];
        acc = fma(df[q] * df[q], kp.a[q], acc);
    }
    const double kv = kp.signal * exp(-0.5 * acc);
#pragma unroll
    for (int q = 0; q < D; ++q) out[i * ld + j * D + q] = -kp.signal * df[q] * kp.a[q] * kv;
}

extern "C" int gpx_se_dgram(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny, int64_t ldy,
                            double* out, int64_t ld, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(h->kp.family == GPX_SE, GPX_EINVAL, "kernel derivatives exist for the squared-exponential family only");
    GPX_REQUIRE(nx >= 0 && ny >= 0 && ld >= ny * h->kp.d, GPX_EINVAL, "bad sizes");
    if (nx == 0 || ny == 0) return GPX_OK;
    GPX_REQUIRE(X && Y && out && nx <= 65535, GPX_EINVAL, "bad arguments");
    dim3 grid((unsigned)((ny + 255) / 256), (unsigned)nx);
    GPX_DISPATCH_DIM(h->kp.d, (se_dgram_kernel<D><<<grid, 256, 0, (cudaStream_t)stream>>>(h->kp, X, nx, ldx, Y, ny, ldy, out, ld)));
    return gpx_check_launch("gpx_se_dgram");
}

// out[(j*D + k), m] = 2 * At[j, m] * ( D(x_m, p_j)[k] - Qneg[(j*D + k), m] ) - At[j, m]^2 * diag[j*D + k]
//     gp.py:322-340 restated; diag (nullable) = d noise(p_j) / d p_j[k], the diagonal of the reference's symmetric
//     dSigdXreal in the heteroscedastic branch (gp.py:314-318, :334-336) -- zero for a constant noise.
template <int D>
__global__ void __launch_bounds__(256) se_var_grad_kernel(const __grid_constant__ KParams kp, const double* __restrict__ P,
                                                           int64_t n, int64_t ldp, const double* __restrict__ X, int64_t M,
                                                           int64_t ldx, const double* __restrict__ At,
                                                           const double* __restrict__ Qneg, const double* __restrict__ diag,
                                                           double* __restrict__ out) {
    const int64_t m = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t j = blockIdx.y;
    if (m >= M || j >= n) return;
    double acc = 0.0, df[D];
#pragma unroll
    for (int q = 0; q < D; ++q) {
        df[q] = X[q * ldx + m] - P[q * ldp + j];
        acc = fma(df[q] * df[q], kp.a[q], acc);
    }
    const double kv = kp.signal * exp(-0.5 * acc);
    const double at = At[j * ldx + m];
    const double a2 = 2.0 * at;
#pragma unroll
    for (int q = 0; q < D; ++q) {
        const int64_t r = j * D + q;
        const double dk = -kp.signal * df[q] * kp.a[q] * kv;
        double v = a2 * (dk - Qneg[r * ldx + m]);
        if (diag) v = fma(-at * at, diag[r], v);
        out[r * ldx + m] = v;
    }
}

extern "C" int gpx_se_var_grad(gpx_handle h, const double* P, int64_t n, int64_t ldp, const double* X, int64_t M, int64_t ldx,
                               const double* At, const double* Qneg, const double* diag, double* out, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(h->kp.family == GPX_SE, GPX_EINVAL, "kernel derivatives exist for the squared-exponential family only");
    GPX_REQUIRE(n >= 0 && M >= 0, GPX_EINVAL, "bad sizes");
    if (n == 0 || M == 0) return GPX_OK;
    GPX_REQUIRE(P && X && At && Qneg && out && n <= 65535, GPX_EINVAL, "bad arguments");
    dim3 grid((unsigned)((M + 255) / 256), (unsigned)n);
    GPX_DISPATCH_DIM(h->kp.d, (se_var_grad_kernel<D><<<grid, 256, 0, (cudaStream_t)stream>>>(h->kp, P, n, ldp, X, M, ldx, At, Qneg, diag, out)));
    return gpx_check_launch("gpx_se_var_grad");
}

// out[r] = scale * sum_c A[r, c]  (one block per row, fixed summation order); WT: sum_c w[c] A[r, c] in the same order
template <bool WT>
__global__ void __launch_bounds__(256) rowsum_kernel(const double* __restrict__ A, int64_t cols, int64_t ld, double scale,
                                                      const double* __restrict__ w, double* __restrict__ out) {
    __shared__ double sm[8];
    const double* row = A + (int64_t)blockIdx.x * ld;
    double s = 0.0;
    for (int64_t c = threadIdx.x; c < cols; c += 256) {
        if (WT) s = fma(w[c], row[c], s);
        else s += row[c];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sm[w];
        out[blockIdx.x] = scale * t;
    }
}

extern "C" int gpx_rowsum(gpx_handle h, const double* A, int64_t rows, int64_t cols, int64_t ld, double scale, double* out,
                          void* stream) {
    GPX_REQUIRE(h && rows >= 0 && cols >= 0, GPX_EINVAL, "bad arguments");
    if (rows == 0) return GPX_OK;
    GPX_REQUIRE(A && out && rows <= 2147483647LL, GPX_EINVAL, "bad arguments");
    rowsum_kernel<false><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(A, cols, ld, scale, nullptr, out);
    return gpx_check_launch("gpx_rowsum");
}

extern "C" int gpx_rowsum_w(gpx_handle h, const double* A, int64_t rows, int64_t cols, int64_t ld, const double* w, double* out,
                            void* stream) {
    GPX_REQUIRE(h && rows >= 0 && cols >= 0, GPX_EINVAL, "bad arguments");
    if (rows == 0) return GPX_OK;
    GPX_REQUIRE(A && out && w && rows <= 2147483647LL, GPX_EINVAL, "bad arguments");
    rowsum_kernel<true><<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(A, cols, ld, 1.0, w, out);
    return gpx_check_launch("gpx_rowsum_w");
}

// out[0] = log det(U^T U) = 2 sum_i log U[i,i]          (np.linalg.slogdet at gp.py:432 for a PD matrix)
__global__ void __launch_bounds__(256) logdet_kernel(const double* __restrict__ U, int64_t n, int64_t ld, double* out) {
    __shared__ double sm[8];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 256) s += log(U[i * ld + i]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sm[w];
        out[0] = 2.0 * t;
    }
}

extern "C" int gpx_logdet_chol(gpx_handle h, const double* U, int64_t n, int64_t ld, double* out, void* stream) {
    GPX_REQUIRE(h && out && n >= 0 && (U || n == 0), GPX_EINVAL, "bad arguments");
    logdet_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(U, n, ld, out);
    return gpx_check_launch("gpx_logdet_chol");
}
