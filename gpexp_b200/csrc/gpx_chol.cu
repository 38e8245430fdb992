// K2 / K3: blocked FP64 Cholesky (A = U^T U, upper, row-major), triangular solves and the rank-1 append.
//
// potrf, right-looking in 128-wide block columns:
//   (1) diagonal block: one CTA, block in shared memory, 32x32 sub-panels factored by ONE WARP with
//       register-resident columns and shuffle broadcasts (the latency-critical part), the in-block panel
//       solve and rank-32 update by the whole CTA;
//   (2) block row  U12 = U11^-T A12   : one thread per column, forward substitution, U11 in shared memory;
//   (3) trailing   A22 -= U12^T U12   : DMMA core (gpx_dgemm_tn_sub, upper tiles only).
// trsm (W = U^-T B), left-looking in 128-row blocks: DMMA update (K = rows already solved) + the same
// forward-substitution kernel.  gpx_trsm_gram writes each 128-row block of the right-hand side K(D,Y) straight into W
// (difference-form Gram kernel), so the n x ny Gram matrix never exists beside W.
#include <math.h>

#include "gpx_common.cuh"

namespace {

constexpr int NB = 128;          // block size
constexpr int SLD = NB + 1;      // padded shared-memory stride

// ---- 32x32 upper Cholesky by one warp: lane j owns column j of the symmetric block ---------------
// On exit col[i] (i <= j) = U[i][j].  Returns 0 or 1 + local index of the first non-positive pivot.
__device__ __forceinline__ int warp_potf2_32(double (&col)[32], int lane) {
    int bad = 0;
    // both loops are fully unrolled with compile-time (k, i) so that col[] stays in registers
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        const double akk = __shfl_sync(0xffffffffu, col[k], k);
        if (!(akk > 0.0) && bad == 0) bad = k + 1;
        const double dkk = sqrt(akk);
        if (lane == k) col[k] = dkk;
        if (lane > k) col[k] = col[k] / dkk;  // U[k][lane]
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            if (i > k) {
                const double uki = __shfl_sync(0xffffffffu, col[k], i);  // U[k][i]
                if (lane >= i) col[i] = fma(-uki, col[k], col[i]);
            }
        }
    }
    return bad;
}

// ---- diagonal block factorisation -----------------------------------------------------------------
__global__ void __launch_bounds__(256, 1) potrf_diag_kernel(double* __restrict__ A, int64_t ld, int b, int64_t kb, int* info) {
    extern __shared__ double S[];  // NB x SLD, upper part meaningful
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // load (identity padding beyond b so that ragged blocks factor cleanly)
    for (int e = tid; e < NB * NB; e += 256) {
        const int r = e / NB, c = e % NB;
        double v = (r == c) ? 1.0 : 0.0;
        if (r < b && c < b && c >= r) v = A[(kb + r) * ld + kb + c];
        S[r * SLD + c] = v;
    }
    __syncthreads();
    for (int p = 0; p < NB; p += 32) {
        if (p >= b) break;
        if (warp == 0) {
            double col[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) col[i] = S[(p + i) * SLD + p + lane];
            const int bad = warp_potf2_32(col, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (i <= lane) S[(p + i) * SLD + p + lane] = col[i];
            if (lane == 0 && bad && p + bad <= b) atomicCAS(info, 0, (int)(kb + p + bad));
        }
        __syncthreads();
        const int rest = NB - (p + 32);
        if (rest > 0) {
            // in-block panel solve: rows p..p+32, columns p+32..NB : one thread per column
            if (tid < rest) {
                const int c = p + 32 + tid;
                double x[32];
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    double v = S[(p + r) * SLD + c];
#pragma unroll
                    for (int s = 0; s < r; ++s) v = fma(-S[(p + s) * SLD + p + r], x[s], v);
                    x[r] = v / S[(p + r) * SLD + p + r];
                }
#pragma unroll
                for (int r = 0; r < 32; ++r) S[(p + r) * SLD + c] = x[r];
            }
            __syncthreads();
            // rank-32 update of the trailing upper part of the block
            for (int e = tid; e < rest * rest; e += 256) {
                const int i = p + 32 + e / rest, j = p + 32 + e % rest;
                if (j < i) continue;
                double v = S[i * SLD + j];
#pragma unroll 8
                for (int s = 0; s < 32; ++s) v = fma(-S[(p + s) * SLD + i], S[(p + s) * SLD + j], v);
                S[i * SLD + j] = v;
            }
            __syncthreads();
        }
    }
    for (int e = tid; e < NB * NB; e += 256) {
        const int r = e / NB, c = e % NB;
        if (r < b && c < b && c >= r) A[(kb + r) * ld + kb + c] = S[r * SLD + c];
    }
}

// ---- forward substitution  X = T^-T B  for a b x b upper-triangular T (b <= 128), in place --------
// One thread per column; 32 solution entries live in registers at a time, earlier ones are re-read.
// TRANS_T == false : T[s][r] = Tm[s*ldt + r]   (U stored upper, row-major)             -> X = U^-T B
// TRANS_T == true  : T[s][r] = Tm[r*ldt + s], rows walked bottom-up                    -> X = L^-T B = U^-1 B (L = U^T)
// The coefficients sit in shared memory as a PACKED triangle (row s keeps columns (s & ~1) .. bw-1, bw = b rounded up to
// 32, zero padded): 65 KB instead of the 129 KB square, so three 128-thread CTAs share an SM (12 warps instead of 4), and
// every row segment starts 16-byte aligned, so the broadcast reads are 16 bytes.  One wave of CTAs: each stages the
// triangle once (8 loads in flight) and walks over its column chunks.  Same FMA order per entry as a plain forward
// substitution.  ncu (r02, 256 x 1 shape before the persistent loop): FP64 pipe 24 % active, stalls spread over
// fixed-latency waits 25 %, global loads 20 %, shared loads 16 %, the staging barrier 9 % -- latency, not a pipe.

__host__ __device__ __forceinline__ int tri_off(int s, int bw) {
    const int h = s >> 1;
    return s * bw - 2 * ((s & 1) ? h * h : h * (h - 1));
}

template <bool BACK, int TS_NT, int MINB, int UNR>
__global__ void __launch_bounds__(TS_NT, MINB) tri_solve_kernel(const double* __restrict__ Tm, int64_t ldt, int b,
                                                                 double* __restrict__ B, int64_t ldb, int64_t ncols) {
    extern __shared__ __align__(16) double St[];  // element (s, r), r >= (s & ~1): St[tri_off(s) + r - (s & ~1)]
    const int bw = (b + 31) & ~31;
    // coefficients: staged once per CTA (the CTA then walks over its column chunks), 8 independent loads in flight
#pragma unroll 8
    for (int e = threadIdx.x; e < b * bw; e += TS_NT) {
        const int s = e / bw, r = e - s * bw;
        const int c0 = s & ~1;
        // forward:  eq r: sum_{s<=r} U[s][r] x_s = rhs_r.   backward (rows reversed): eq r': sum_{s'<=r'} L[..]..
        // reversed indices: s' = b-1-s, r' = b-1-r ; U[r'][s'] with s' >= r'  <=>  s <= r ; L = U^T given: Tm[s'*ldt + r']
        const bool live = s <= r && r < b;
        const int64_t src = BACK ? (int64_t)(b - 1 - s) * ldt + (b - 1 - r) : (int64_t)s * ldt + r;
        const double v = live ? Tm[src] : 0.0;
        if (r >= c0) St[tri_off(s, bw) + r - c0] = v;
    }
    __syncthreads();
    const int64_t rstride = BACK ? -ldb : ldb;                       // walking the rows in solution order
    for (int64_t j = (int64_t)blockIdx.x * TS_NT + threadIdx.x; j < ncols; j += (int64_t)gridDim.x * TS_NT) {
        double* col = B + (BACK ? (int64_t)(b - 1) * ldb : 0) + j;  // row 0 of the solution order
        for (int rb = 0; rb < b; rb += 32) {
            double x[32];
            double* blk = col + rb * rstride;
#pragma unroll
            for (int r = 0; r < 32; ++r) x[r] = (rb + r < b) ? blk[r * rstride] : 0.0;
            const double* xsp = col;
#pragma unroll(UNR)
            for (int s = 0; s < rb; ++s, xsp += rstride) {
                const double xs = *xsp;
                const double2* ts = reinterpret_cast<const double2*>(St + tri_off(s, bw) + rb - (s & ~1));
#pragma unroll
                for (int r2 = 0; r2 < 16; ++r2) {
                    const double2 c = ts[r2];
                    x[2 * r2] = fma(-c.x, xs, x[2 * r2]);
                    x[2 * r2 + 1] = fma(-c.y, xs, x[2 * r2 + 1]);
                }
            }
            // the 32 x 32 diagonal triangle, right-looking: entry r receives its terms in the order s = 0 .. r-1
#pragma unroll
            for (int s = 0; s < 32; ++s) {
                if (rb + s < b) {
                    const double* row = St + tri_off(rb + s, bw) - (s & ~1);  // coefficient (rb+s, rb+r) at row[r]
                    x[s] = x[s] / row[s];
#pragma unroll
                    for (int r = s + 1; r < 32; ++r) x[r] = fma(-row[r], x[s], x[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < 32; ++r)
                if (rb + r < b) blk[r * rstride] = x[r];
        }
    }
}

template <bool BACK, int TS_NT, int MINB, int UNR>
int launch_tri_solve_v(gpx_handle h, const double* Tm, int64_t ldt, int b, double* B, int64_t ldb, int64_t ncols, cudaStream_t st) {
    const size_t smem_max = (size_t)tri_off(NB, NB) * sizeof(double);
    int rc = gpx_ensure_smem(h, (const void*)tri_solve_kernel<BACK, TS_NT, MINB, UNR>, smem_max, "tri_solve");
    if (rc) return rc;
    if (ncols <= 0 || b <= 0) return GPX_OK;
    const size_t smem = (size_t)tri_off(b, (b + 31) & ~31) * sizeof(double);
    // one wave of CTAs; each stages the triangle once and walks over its column chunks
    int64_t grid = (ncols + TS_NT - 1) / TS_NT;
    const int64_t wave = (int64_t)MINB * (h->sm_count > 0 ? h->sm_count : 148);
    if (grid > wave) grid = wave;
    tri_solve_kernel<BACK, TS_NT, MINB, UNR><<<(unsigned)grid, TS_NT, smem, st>>>(Tm, ldt, b, B, ldb, ncols);
    return gpx_check_launch("tri_solve");
}

// 128 threads x 3 CTAs per SM, two steps of the elimination loop unrolled: the best of the block shapes measured on B200
// (fused Gram/TRSM at n = 255 / 1024 over 1e5 columns: 0.68 / 5.30 ms; 256 x 1: 0.68 / 5.32; 256 x 2: 0.75 / 5.55;
// the 129 KB square layout with one 128-thread CTA per SM: 1.07 / 6.80; two columns per thread: 0.69 - 0.73 / 5.36 - 5.51).
template <bool BACK>
int launch_tri_solve(gpx_handle h, const double* Tm, int64_t ldt, int b, double* B, int64_t ldb, int64_t ncols, cudaStream_t st) {
    return launch_tri_solve_v<BACK, 128, 3, 2>(h, Tm, ldt, b, B, ldb, ncols, st);
}

__global__ void set_int_kernel(int* p, int v) { *p = v; }

}  // namespace

extern "C" int gpx_potrf(gpx_handle h, double* A, int64_t n, int64_t ld, int* info, void* stream) {
    GPX_REQUIRE(h && info && n >= 0, GPX_EINVAL, "bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    set_int_kernel<<<1, 1, 0, st>>>(info, 0);
    {
        int rc = gpx_check_launch("gpx_potrf");
        if (rc || n == 0) return rc;
    }
    GPX_REQUIRE(A && ld >= n, GPX_EINVAL, "bad matrix");
    GPX_REQUIRE((ld % 2) == 0 && gpx_aligned16(A), GPX_EALIGN, "A must be 16-byte aligned with an even leading dimension");
    const size_t smem = (size_t)NB * SLD * sizeof(double);
    {
        int rc = gpx_ensure_smem(h, (const void*)potrf_diag_kernel, smem, "gpx_potrf");
        if (rc) return rc;
    }
    for (int64_t kb = 0; kb < n; kb += NB) {
        const int b = (int)(n - kb < NB ? n - kb : NB);
        potrf_diag_kernel<<<1, 256, smem, st>>>(A, ld, b, kb, info);
        int rc = gpx_check_launch("gpx_potrf diag");
        if (rc) return rc;
        const int64_t rest = n - kb - b;
        if (rest > 0) {
            double* A12 = A + kb * ld + kb + b;
            rc = launch_tri_solve<false>(h, A + kb * ld + kb, ld, b, A12, ld, rest, st);
            if (rc) return rc;
            rc = gpx_dgemm_tn_sub(h, A12, ld, A12, ld, A + (kb + b) * ld + kb + b, ld, rest, rest, b, 1, stream);
            if (rc) return rc;
        }
    }
    return GPX_OK;
}

extern "C" int gpx_trsm_gram(gpx_handle h, const double* U, int64_t n, int64_t ldu, const double* D, int64_t ldd,
                             const double* Y, int64_t ny, int64_t ldy, double* W, int64_t ldw, double* var_out, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(n >= 0 && ny >= 0, GPX_EINVAL, "negative size");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (ny == 0) return GPX_OK;
    if (n > 0) {
        GPX_REQUIRE(U && D && Y && W, GPX_EINVAL, "NULL pointer");
        // whole 128-wide tiles readable on both operands -> the TMA update kernel; else the predicated one
        const bool padded = (ldu % NB) == 0 && ldu >= (n + NB - 1) / NB * NB && (ldw % NB) == 0 && ldw >= (ny + NB - 1) / NB * NB &&
                            gpx_aligned16(U) && gpx_aligned16(W);
        for (int64_t kb = 0; kb < n; kb += NB) {
            const int b = (int)(n - kb < NB ? n - kb : NB);
            // block row:  W[kb:kb+b, :] = K(D[kb:kb+b], Y)            difference-form Gram, written once (8 b ny bytes)
            rc = gpx_gram(h, D + kb, b, ldd, Y, ny, ldy, W + kb * ldw, ldw, 0, nullptr, 0.0, stream);
            if (rc) return rc;
            //             W[kb:kb+b, :] -= U[0:kb, kb:kb+b]^T W[0:kb, :]  FP64 DMMA update
            if (kb > 0) {
                rc = padded ? gpx_dgemm_tn_sub_padded(h, U + kb, ldu, W, ldw, W + kb * ldw, ldw, b, ny, kb, 0, stream)
                            : gpx_dgemm_tn_sub(h, U + kb, ldu, W, ldw, W + kb * ldw, ldw, b, ny, kb, 0, stream);
                if (rc) return rc;
            }
            //             W[kb:kb+b, :] = U_kk^-T W[kb:kb+b, :]           forward substitution
            rc = launch_tri_solve<false>(h, U + kb * ldu + kb, ldu, b, W + kb * ldw, ldw, ny, st);
            if (rc) return rc;
        }
    }
    if (var_out) {
        GPX_REQUIRE(Y != nullptr, GPX_EINVAL, "Y is required for the variance output");
        rc = gpx_prior_diag(h, Y, ny, ldy, var_out, stream);
        if (rc) return rc;
        if (n > 0) rc = gpx_colsumsq(h, W, n, ny, ldw, var_out, var_out, stream);
        if (rc) return rc;
    }
    return GPX_OK;
}

static int trsm_forward(gpx_handle h, const double* U, int64_t n, int64_t ldu, double* B, int64_t ncols, int64_t ldb,
                        int lower_tri_rhs, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    for (int64_t kb = 0; kb < n; kb += NB) {
        const int b = (int)(n - kb < NB ? n - kb : NB);
        int64_t active = ncols;
        if (lower_tri_rhs && kb + b < active) active = kb + b;  // block row kb of U^-T is zero right of its diagonal block
        int rc;
        if (kb > 0) {
            rc = gpx_dgemm_tn_sub(h, U + kb, ldu, B, ldb, B + kb * ldb, ldb, b, active, kb, 0, stream);
            if (rc) return rc;
        }
        rc = launch_tri_solve<false>(h, U + kb * ldu + kb, ldu, b, B + kb * ldb, ldb, active, st);
        if (rc) return rc;
    }
    return GPX_OK;
}

extern "C" int gpx_trsm(gpx_handle h, const double* U, int64_t n, int64_t ldu, double* B, int64_t ncols, int64_t ldb,
                        void* stream) {
    GPX_REQUIRE(h && n >= 0 && ncols >= 0, GPX_EINVAL, "bad arguments");
    if (n == 0 || ncols == 0) return GPX_OK;
    GPX_REQUIRE(U && B, GPX_EINVAL, "NULL pointer");
    return trsm_forward(h, U, n, ldu, B, ncols, ldb, 0, stream);
}

// Y = U^-T as an explicit lower-triangular matrix (MI set-up: precision diagonal and columns come from it).
__global__ void __launch_bounds__(256) set_identity_kernel(double* Y, int64_t n, int64_t ld) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n * ld) return;
    const int64_t r = e / ld, c = e % ld;
    Y[e] = (r == c) ? 1.0 : 0.0;
}

extern "C" int gpx_trtri_t(gpx_handle h, const double* U, int64_t n, int64_t ldu, double* Y, int64_t ldy, void* stream) {
    GPX_REQUIRE(h && n >= 0, GPX_EINVAL, "bad arguments");
    if (n == 0) return GPX_OK;
    GPX_REQUIRE(U && Y && ldy >= n, GPX_EINVAL, "bad arguments");
    const int64_t total = n * ldy;
    set_identity_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(Y, n, ldy);
    int rc = gpx_check_launch("gpx_trtri_t identity");
    if (rc) return rc;
    return trsm_forward(h, U, n, ldu, Y, n, ldy, 1, stream);
}

extern "C" int gpx_trsm_back(gpx_handle h, const double* Ut, int64_t n, int64_t ldu, double* B, int64_t ncols, int64_t ldb,
                             void* stream) {
    GPX_REQUIRE(h && n >= 0 && ncols >= 0, GPX_EINVAL, "bad arguments");
    if (n == 0 || ncols == 0) return GPX_OK;
    GPX_REQUIRE(Ut && B, GPX_EINVAL, "NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    // bottom-up over block rows; Ut = U^T (lower, row-major) so that the update operand is K-major:
    //   B[kb:kb+b, :] -= sum_{k >= kb+b} U[kb+i, k] B[k, :] = sum_k Ut[k*ldu + kb + i] B[k, :]
    const int64_t nblk = (n + NB - 1) / NB;
    for (int64_t blk = nblk - 1; blk >= 0; --blk) {
        const int64_t kb = blk * NB;
        const int b = (int)(n - kb < NB ? n - kb : NB);
        const int64_t below = n - kb - b;
        int rc;
        if (below > 0) {
            rc = gpx_dgemm_tn_sub(h, Ut + (kb + b) * ldu + kb, ldu, B + (kb + b) * ldb, ldb, B + kb * ldb, ldb, b, ncols,
                                  below, 0, stream);
            if (rc) return rc;
        }
        rc = launch_tri_solve<true>(h, Ut + kb * ldu + kb, ldu, b, B + kb * ldb, ldb, ncols, st);
        if (rc) return rc;
    }
    return GPX_OK;
}

// ---- rank-1 append: one CTA, x in shared memory, 32-row panels ---------------------------------------
__global__ void __launch_bounds__(1024, 1) chol_append_kernel(double* __restrict__ U, int n, int64_t ld,
                                                               const double* __restrict__ knew, double kpp, int* info) {
    extern __shared__ double x[];  // n entries
    __shared__ double red[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < n; i += 1024) x[i] = knew[i];
    __syncthreads();
    for (int rb = 0; rb < n; rb += 32) {
        const int b = n - rb < 32 ? n - rb : 32;
        if (warp == 0) {
            // solve the 32x32 triangle: lane r owns x[rb+r]
            double xr = lane < b ? x[rb + lane] : 0.0;
            for (int s = 0; s < b; ++s) {
                const double uss = U[(int64_t)(rb + s) * ld + rb + s];
                const double xs = __shfl_sync(0xffffffffu, xr, s) / uss;
                if (lane == s) xr = xs;
                if (lane > s && lane < b) xr = fma(-U[(int64_t)(rb + s) * ld + rb + lane], xs, xr);
            }
            if (lane < b) x[rb + lane] = xr;
        }
        __syncthreads();
        for (int i = rb + 32 + tid; i < n; i += 1024) {
            double v = x[i];
#pragma unroll 8
            for (int s = 0; s < 32; ++s) v = fma(-U[(int64_t)(rb + s) * ld + i], x[rb + s], v);
            x[i] = v;
        }
        __syncthreads();
    }
    double ss = 0.0;
    for (int i = tid; i < n; i += 1024) {
        ss = fma(x[i], x[i], ss);
        U[(int64_t)i * ld + n] = x[i];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    if (warp == 0) {
        ss = red[lane];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
        if (lane == 0) {
            const double d2 = kpp - ss;
            info[0] = d2 > 0.0 ? 0 : n + 1;
            U[(int64_t)n * ld + n] = sqrt(d2);
        }
    }
}

extern "C" int gpx_chol_append(gpx_handle h, double* U, int64_t n, int64_t ld, const double* knew, double kpp, int* info,
                               void* stream) {
    GPX_REQUIRE(h && U && info && n >= 0 && ld > n, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(knew || n == 0, GPX_EINVAL, "knew is NULL");
    const size_t smem = (size_t)n * sizeof(double);
    GPX_REQUIRE(smem <= 200 * 1024, GPX_ESIZE, "design size exceeds the shared-memory buffer (25600)");
    // the kernel's static reduction buffer (red[32]) counts against the 48 KB a launch gets without the opt-in
    if (smem + 32 * sizeof(double) > 48 * 1024) {
        int rc = gpx_ensure_smem(h, (const void*)chol_append_kernel, 200 * 1024, "gpx_chol_append");
        if (rc) return rc;
    }
    chol_append_kernel<<<1, 1024, smem, (cudaStream_t)stream>>>(U, (int)n, ld, knew, kpp, info);
    return gpx_check_launch("gpx_chol_append");
}
