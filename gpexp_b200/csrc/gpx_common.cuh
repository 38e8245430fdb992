// Shared declarations of the gpexp_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gpexp_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "gpexp_b200 is written for sm_100a (B200) only"
#endif

// ---------------------------------------------------------------------------------------------
// Kernel hyper-parameters.  Passed BY VALUE to every launch as a __grid_constant__ argument, so the
// ARD length-scales live in the constant bank without a module-global that handles would share.
// ---------------------------------------------------------------------------------------------
struct KParams {
    int family;
    int d;
    double signal;            // SE / MATERN32: signalSize ; MEHLER: prod_i (1 - t_i^2)^(-1/2)
    double c0;                // MATERN32: sqrt(3) / rho
    double a[GPX_MAX_DIM];    // SE: cl_i^-2            ; MEHLER: t_i^2
    double b[GPX_MAX_DIM];    // MEHLER: 2 t_i
    double c[GPX_MAX_DIM];    // MEHLER: 1 / (2 (1 - t_i^2))
};

#define GPX_SMEM_FUNCS 96

struct KCenter {
    double c[GPX_MAX_DIM];
};

struct gpx_context {
    int device;
    int sm_count;
    bool has_kernel;
    KParams kp;
    // reduction scratch, all device memory
    double* red_val;          // GPX_RED_SLOTS doubles
    int64_t* red_idx;         // GPX_RED_SLOTS indices
    unsigned int* red_counter;// last-block-done tickets (zero between calls)
    double* scal;             // a few device scalars (sum of varM ...)
    int64_t* iscal;
    // centre subtracted from every coordinate by gpx_prep_side (stationary families only): keeps the expanded-form
    // prologue k = f(alpha + beta + u.v) well conditioned for un-normalised inputs
    double center[GPX_MAX_DIM];
    // kernels already opted in to > 48 KB of dynamic shared memory ON THIS DEVICE (the attribute is per device)
    const void* smem_ready[GPX_SMEM_FUNCS];
    int n_smem_ready;
    // optional NCCL communicator (gpx_comm_init); the library resolves NCCL at run time, it does not link it
    void* nccl_comm;
    int comm_rank, comm_size;
    int ivar_ring;            // ring geometry of ivar_ws_kernel (gpx_set_ivar_ring)
    int ivar_core;            // GPX_CORE_DMMA | GPX_CORE_I8 (gpx_set_ivar_core)
    void* i8_scratch;         // caller memory for the INT8 core's operand slices (gpx_set_ivar_scratch)
    int64_t i8_scratch_bytes;
};

#ifndef GPX_DEFAULT_IVAR_RING
#define GPX_DEFAULT_IVAR_RING 1
#endif

#define GPX_RED_SLOTS 2048

void gpx_set_error(const char* fmt, ...);
int gpx_check_launch(const char* what);
// opt `func` in to `bytes` of dynamic shared memory once per handle (= per device)
int gpx_ensure_smem(gpx_handle h, const void* func, size_t bytes, const char* name);

#define GPX_REQUIRE(cond, code, msg)                 \
    do {                                             \
        if (!(cond)) {                               \
            gpx_set_error("%s: %s", __func__, msg);  \
            return (code);                           \
        }                                            \
    } while (0)

#define GPX_NEED_KERNEL(h) GPX_REQUIRE((h) && (h)->has_kernel, GPX_ENOKERNEL, "gpx_set_kernel has not been called")

static inline bool gpx_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---------------------------------------------------------------------------------------------
// Difference-form covariance evaluation, one dimension at a time (coordinates come from wherever
// the caller keeps them: registers, shared memory or strided global memory).
//   SE       kernels.py:121-122   signal * exp(-1/2 sum (x-y)^2 cl^-2)
//   MATERN32 kernels.py:87-89     signal * (1 + sqrt3 r / rho) exp(-sqrt3 r / rho)
//   MEHLER   kernels.py:282-285   prod_i (1-t^2)^(-1/2) exp(-(x^2 t^2 - 2 t x y + y^2 t^2) / (2 (1-t^2)))
// ---------------------------------------------------------------------------------------------
template <int FAM>
__device__ __forceinline__ void kacc_dim(double& acc, const KParams& kp, int i, double x, double y) {
    if (FAM == GPX_SE) {
        const double df = x - y;
        acc = fma(df * df, kp.a[i], acc);
    } else if (FAM == GPX_MATERN32) {
        const double df = x - y;
        acc = fma(df, df, acc);
    } else {
        const double num = x * x * kp.a[i] - kp.b[i] * x * y + y * y * kp.a[i];
        acc = fma(num, kp.c[i], acc);
    }
}

template <int FAM>
__device__ __forceinline__ double kfinish(double acc, const KParams& kp) {
    if (FAM == GPX_SE) return kp.signal * exp(-0.5 * acc);
    if (FAM == GPX_MATERN32) {
        const double t = kp.c0 * sqrt(acc);
        return kp.signal * (1.0 + t) * exp(-t);
    }
    return kp.signal * exp(-acc);
}

// ---------------------------------------------------------------------------------------------
// One new factor row for two adjacent columns j, j+1 (K3+K4):  w = (src - sum_i l[i] W[i, j]) / sqrt(pivot).
// Called by every thread of the block (it holds the block's barrier); sl = shared buffer of roundup(n, 16) doubles that
// receives the pivot's column l (zero padded).  Ordering is what the timing rests on: the first 16 rows of W are
// requested BEFORE the pivot column is staged and the source term k(x_p, y_j) evaluated, so their latency is hidden;
// every later batch is 16 independent 16-byte streaming loads; the ragged end of n is one more predicated batch, not a
// chain of short ones.  SRC_KERNEL: src from the kernel function of rec's coordinates and Y; else from src_row.
// ---------------------------------------------------------------------------------------------
template <int FAM, bool SRC_KERNEL>
__device__ __forceinline__ void gpx_append_two_columns(const KParams& kp, const double* __restrict__ rec,
                                                       const double* __restrict__ src_row, const double* __restrict__ Y,
                                                       int64_t ncols, int64_t ldy, double* __restrict__ W, int64_t ldw, int n,
                                                       double* __restrict__ var, int64_t j, double* sl, int nthreads) {
    const bool active = j < ncols;
    const bool two = j + 1 < ncols;
    const double* wp = W + j;
    double2 w[16];
    double v0 = 0.0, v1 = 0.0;
    if (active) {
#pragma unroll
        for (int u = 0; u < 16; ++u)
            w[u] = u < n ? __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)u * ldw)) : make_double2(0.0, 0.0);
        v0 = var[j];
        if (two) v1 = var[j + 1];
    }
    const int n16 = (n + 15) & ~15;
    for (int i = threadIdx.x; i < n16; i += nthreads) sl[i] = i < n ? rec[GPX_PIVOT_HDR + i] : 0.0;
    double s0 = 0.0, s1 = 0.0;
    if (active) {
        if (SRC_KERNEL) {
            double k0 = 0.0, k1 = 0.0;
#pragma unroll
            for (int q = 0; q < GPX_MAX_DIM; ++q)
                if (q < kp.d) {
                    const double xp = rec[3 + q];
                    const double2 y = *reinterpret_cast<const double2*>(Y + q * ldy + j);
                    kacc_dim<FAM>(k0, kp, q, xp, y.x);
                    kacc_dim<FAM>(k1, kp, q, xp, y.y);
                }
            s0 = kfinish<FAM>(k0, kp);
            s1 = kfinish<FAM>(k1, kp);
        } else {
            const double2 sv = *reinterpret_cast<const double2*>(src_row + j);
            s0 = sv.x;
            s1 = sv.y;
        }
    }
    // a non-positive pivot (numerically dependent point, noise 0) appends a zero row: "no reduction", what the
    // reference's pinv makes of a null direction (gp.py:181) -- instead of NaN from sqrt of a negative number
    const double lnn = rec[2] > 0.0 ? sqrt(rec[2]) : INFINITY;
    __syncthreads();
    if (!active) return;
    double a0 = 0.0, a1 = 0.0;
    if (n > 0) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(sl[u], w[u].x, a0);
            a1 = fma(sl[u], w[u].y, a1);
        }
    }
    int i = 16;
    for (; i + 16 <= n; i += 16) {
#pragma unroll
        for (int u = 0; u < 16; ++u) w[u] = __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)(i + u) * ldw));
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(sl[i + u], w[u].x, a0);
            a1 = fma(sl[i + u], w[u].y, a1);
        }
    }
    if (i < n) {
#pragma unroll
        for (int u = 0; u < 16; ++u)
            w[u] = i + u < n ? __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)(i + u) * ldw)) : make_double2(0.0, 0.0);
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(sl[i + u], w[u].x, a0);
            a1 = fma(sl[i + u], w[u].y, a1);
        }
    }
    const double w0 = (s0 - a0) / lnn;
    const double w1 = (s1 - a1) / lnn;
    double* dst = W + (int64_t)n * ldw + j;
    dst[0] = w0;
    dst[1] = two ? w1 : 0.0;
    var[j] = v0 - w0 * w0;
    if (two) var[j + 1] = v1 - w1 * w1;
}

// 2^(j/256): table-driven exp used by the covariance prologue of the hot kernel and by the Gram kernel.  exp(x) = 2^k * T[j] * e^r with
// n = rint(x * 256/ln2) = 256 k + j and |r| <= ln2/512, e^r - 1 by a degree-4 polynomial: 9 FP64-pipe operations, one
// compare and one shared-memory lookup per value (libdevice exp: 19 FP64 + 26 other instructions).
// The callers fold the signal variance (and a sign) into the table, tab[j] = s * 2^(j/256), so the result is s * exp(x)
// for any normal s; its exponent is assembled in the high word as (biased exponent of tab[j] e^r) + k.
//   accuracy  <= 2 ulp of s * exp(x) for an exact argument (measured over every table slot and |x| <= 700: the entry,
//             the polynomial and the final product each round once); the rounding of x itself adds |x| eps relative.
//   flush     a result below 2^-1022 (biased exponent <= 0) is returned as 0 -- no subnormals; so is every x below
//             -2^19 ln2/256 ~ -1453, where k << 20 would leave the int range (and, below -5.8e6, n its 32 bits).
//   OVF       a result above DBL_MAX (biased exponent > 2046), and every x above +1453, saturates to +-inf with the
//             sign of the table.  Only the Mehler exponent can be large and positive (x ~ y, kernels.py:282-285); the
//             SE and Matern exponents are <= 0 up to cancellation error, so their instantiations leave it out.
static __device__ const double gpx_exp2_tab[256] = {
#include "gpx_exp_table.inc"
};

// 2^k * res for a table value res = tab[j] e^r, with the flush / saturation rules above; nf = n exactly (as a double)
template <bool OVF>
__device__ __forceinline__ double gpx_exp_tab_scale(double res, int n, double nf) {
    const int hi = __double2hiint(res);
    const int k = n >> 8;
    const int e = ((hi >> 20) & 0x7ff) + k;                     // biased exponent of the result
    // |nf| > 2^19 first: there k (and beyond 2^31 n itself) has wrapped, so e means nothing
    if (nf < -0x1p19) return 0.0;
    if (OVF && (nf > 0x1p19 || e > 2046)) return __hiloint2double((hi & 0x80000000) | 0x7ff00000, 0);
    if (e <= 0) return 0.0;
    return __hiloint2double(hi + (k << 20), __double2loint(res));
}

template <bool OVF = false>
__device__ __forceinline__ double gpx_exp_tab(double x, const double* __restrict__ tab) {
    const double MAGIC = 6755399441055744.0;                    // 1.5 * 2^52
    const double t = fma(x, 0x1.71547652b82fep+8, MAGIC);       // x * 256/ln2, rounded to an integer in the low word
    const int n = __double2loint(t);
    const double nf = t - MAGIC;
    double r = fma(nf, -0x1.62e42fef80000p-9, x);               // ln2/256 split hi (exact products) + lo
    r = fma(nf, -0x1.1cf79abc9e3b4p-44, r);
    double p = fma(1.0 / 24.0, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    const double q = p * r;                                     // e^r - 1
    const double tj = tab[n & 255];
    return gpx_exp_tab_scale<OVF>(fma(tj, q, tj), n, nf);
}

// exp(-S * ln2/256) for an exponent that was accumulated ALREADY SCALED by 256/ln2 (S >= 0): the SE Gram kernel folds
// sqrt(a_q/2 * 256/ln2) into its coordinates, so that S = sum ((x_q - y_q) w_q)^2 costs two FP64 operations per dimension
// and the argument scaling of gpx_exp_tab disappears.  Same table, same polynomial, same flush rule (S > 2^19 gives 0).
__device__ __forceinline__ double gpx_exp_tab_scaled(double S, const double* __restrict__ tab) {
    const double MAGIC = 6755399441055744.0;                    // 1.5 * 2^52
    const double t = MAGIC - S;                                 // -rint(S) in the low word
    const int n = __double2loint(t);
    const double nf = t - MAGIC;                                // = -rint(S), exact
    const double r = (S + nf) * -0x1.62e42fefa39efp-9;          // (rint(S) - S) * ln2/256 : |S + nf| <= 1/2, exact sum
    double p = fma(1.0 / 24.0, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    const double q = p * r;                                     // e^r - 1
    const double tj = tab[n & 255];
    return gpx_exp_tab_scale<false>(fma(tj, q, tj), n, nf);
}

// difference-form finish with the table exp; `tab` already carries the signal variance (tab[j] = signal * 2^(j/256))
template <int FAM>
__device__ __forceinline__ double kfinish_tab(double acc, const KParams& kp, const double* __restrict__ tab) {
    if (FAM == GPX_SE) return gpx_exp_tab(-0.5 * acc, tab);
    if (FAM == GPX_MATERN32) {
        const double t = kp.c0 * sqrt(acc);
        return (1.0 + t) * gpx_exp_tab(-t, tab);
    }
    return gpx_exp_tab<true>(-acc, tab);
}

// Expanded form used by the tensor-core prologue:  k = kexpand(alpha(x) + beta(y) + sum_i u_i(x) v_i(y)).
template <int FAM>
__device__ __forceinline__ double kexpand(double e, const KParams& kp) {
    if (FAM == GPX_MATERN32) {
        const double t = kp.c0 * sqrt(fmax(e, 0.0));
        return kp.signal * (1.0 + t) * exp(-t);
    }
    return kp.signal * exp(e);
}

#define GPX_DIM_CASE(n, ...)     \
    case n: {                    \
        constexpr int D = n;     \
        __VA_ARGS__;             \
    } break;
#define GPX_DISPATCH_DIM(d, ...)                                                                            \
    switch (d) {                                                                                            \
        GPX_DIM_CASE(1, __VA_ARGS__) GPX_DIM_CASE(2, __VA_ARGS__) GPX_DIM_CASE(3, __VA_ARGS__)             \
        GPX_DIM_CASE(4, __VA_ARGS__) GPX_DIM_CASE(5, __VA_ARGS__) GPX_DIM_CASE(6, __VA_ARGS__)             \
        GPX_DIM_CASE(7, __VA_ARGS__) GPX_DIM_CASE(8, __VA_ARGS__) GPX_DIM_CASE(9, __VA_ARGS__)             \
        GPX_DIM_CASE(10, __VA_ARGS__) GPX_DIM_CASE(11, __VA_ARGS__) GPX_DIM_CASE(12, __VA_ARGS__)          \
        GPX_DIM_CASE(13, __VA_ARGS__) GPX_DIM_CASE(14, __VA_ARGS__) GPX_DIM_CASE(15, __VA_ARGS__)          \
        GPX_DIM_CASE(16, __VA_ARGS__)                                                                       \
        default: break;                                                                                     \
    }

#define GPX_DISPATCH_FAMILY(fam, ...)                         \
    do {                                                      \
        if ((fam) == GPX_SE) {                                \
            constexpr int FAM = GPX_SE;                       \
            __VA_ARGS__;                                      \
        } else if ((fam) == GPX_MATERN32) {                   \
            constexpr int FAM = GPX_MATERN32;                 \
            __VA_ARGS__;                                      \
        } else {                                              \
            constexpr int FAM = GPX_MEHLER;                   \
            __VA_ARGS__;                                      \
        }                                                     \
    } while (0)

// ---------------------------------------------------------------------------------------------
// (value, index) ordering of np.argmax / np.argmin: better value wins, ties go to the lower index.
// ---------------------------------------------------------------------------------------------
// A NaN beats every number (np.argmax / np.argmin return the first NaN), so NaN scores surface instead of hiding.
__device__ __forceinline__ bool gpx_better(double v, int64_t i, double bv, int64_t bi, bool minimize) {
    if (i < 0) return false;
    if (bi < 0) return true;
    const bool vn = (v != v), bn = (bv != bv);
    if (vn || bn) return vn && (!bn || i < bi);
    if (minimize ? (v < bv) : (v > bv)) return true;
    return (v == bv) && (i < bi);
}

__device__ __forceinline__ void gpx_warp_argreduce(double& v, int64_t& i, bool minimize) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, off);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, i, off);
        if (gpx_better(ov, oi, v, i, minimize)) {
            v = ov;
            i = oi;
        }
    }
}

// internal launchers shared between translation units
int gpx_launch_core_ivar(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* Ma_rows, int64_t M,
                         const double* Wc, int64_t ldc, const double* Cb_rows, int64_t C, int64_t n, double* partial,
                         int64_t ldp, int* nsplit_out, cudaStream_t st);
int gpx_launch_core_store(gpx_handle h, int prologue, const double* A, int64_t lda, const double* Ap, int64_t I,
                          const double* B, int64_t ldb, const double* Bp, int64_t J, int64_t K, double* out, int64_t ldo,
                          cudaStream_t st);
int gpx_ivar_splits(gpx_handle h, int64_t M, int64_t C);
int gpx_argreduce_impl(gpx_handle h, const double* v, const double* weights, const uint8_t* mask, int64_t n,
                       int minimize, double* best, int64_t* idx, cudaStream_t st);
int gpx_sum_impl(gpx_handle h, const double* v, int64_t n, double* out, cudaStream_t st);
