// Deleting a point from the middle of a greedy design (IVAR, MI, maximum variance), and the keep-or-swap rule of the
// exchange pass.
//
// Engine state: K_DD + diag(noise) = U^T U (U upper triangular, column i = W[0..i-1, p_i] and sqrt(pivot_i), as
// gpx_store_pivot writes it) and W_X = U^-T K(D, X).  Deleting design position j:
//   H = U without column j is upper Hessenberg in rows j..n-1.  Givens rotations G_i on rows (i, i+1), i = j..n-2, each
//   zeroing H[i+1, i] (c = a / rho, s = b / rho, rho = hypot(a, b) >= 0; the identity when a = b = 0), turn rows j..n-2
//   into the factor U' of the design without point j; row n-1 becomes zero.  The same rotations applied to rows j..n-1
//   of W give W' in rows j..n-2 and a residual row r in row n-1 (the part of x's covariance with the design that only
//   the deleted point explained): var' = var + r^2, and for the resident covariance cov' = cov + r_M r_C^T.
// Since K(D \ j, X) = H^T W = (G H)^T (G W) and G is orthogonal, this is exact algebra; rows 0..j-1 of W do not change.
#include <math.h>

#include "gpx_common.cuh"

namespace {

// ---------------------------------------------------------------------------------------------
// The factor downdate: one block, columns of H spread cyclically over the threads (column k = j + tid + q NT).
// Step i applies rotation i to every column k > i and writes U'[i, k]; the owner of column i + 1 then determines
// rotation i + 1 from its carry and the old diagonal U[i+2, i+2] (staged in shared memory up front, so no global load is
// on the step's critical path), and the loads of row i + 2 for step i + 1 are issued before the barrier.
// One barrier per rotation: O((n - j)^2 / NT) arithmetic per thread, latency bound (the measured time is in README.md).
// ---------------------------------------------------------------------------------------------
constexpr int DF_NT = 1024;
constexpr int DF_CPT = 8;   // columns per thread: at most DF_NT * DF_CPT rotations

struct DeleteFactorArgs {
    double* U;
    int64_t ldu;
    double* rot;
    int64_t* picks;
    double* scores;
    double* pivots;
};

// Block b downdates factor b: independent factors of one design (MI keeps two) go in one launch of two blocks.
__global__ void __launch_bounds__(DF_NT, 1) delete_factor_kernel(DeleteFactorArgs f0, DeleteFactorArgs f1, int n, int j) {
    const bool b0 = blockIdx.x == 0;
    double* __restrict__ U = b0 ? f0.U : f1.U;
    const int64_t ldu = b0 ? f0.ldu : f1.ldu;
    double* __restrict__ rot = b0 ? f0.rot : f1.rot;
    int64_t* __restrict__ picks = b0 ? f0.picks : f1.picks;
    double* __restrict__ scores = b0 ? f0.scores : f1.scores;
    double* __restrict__ pivots = b0 ? f0.pivots : f1.pivots;
    extern __shared__ double sdiag[];          // sdiag[k - j] = U[k+1, k+1], k = j .. n-2
    __shared__ double srot[2][3];              // (c, s, rho) of the current and the next rotation
    const int tid = threadIdx.x;
    const int last = n - 2;                    // last column of H that is rotated
    const int m = n - 1 - j;                   // number of rotations = columns of H from j on
    // rows 0..j-1: column k <- column k+1 (k = j .. n-2), one warp per row, 32 columns at a time
    for (int r = tid >> 5; r < j; r += DF_NT / 32) {
        double* row = U + (int64_t)r * ldu;
        for (int k0 = j; k0 <= last; k0 += 32) {
            const int k = k0 + (tid & 31);
            const double v = k <= last ? row[k + 1] : 0.0;
            __syncwarp();
            if (k <= last) row[k] = v;
        }
    }
    // history: positions j+1..n-1 move down by one (warp 0, 32 entries at a time)
    if (tid < 32 && (picks || scores)) {
        for (int k0 = j; k0 <= last; k0 += 32) {
            const int k = k0 + tid;
            const int64_t pv = (picks && k <= last) ? picks[k + 1] : 0;
            const double sv = (scores && k <= last) ? scores[k + 1] : 0.0;
            __syncwarp();
            if (k <= last) {
                if (picks) picks[k] = pv;
                if (scores) scores[k] = sv;
            }
        }
    }
    // carries t = H[j, k] and the first operands x = H[j+1, k] of my columns; the old diagonal
    double t[DF_CPT], x[DF_CPT];
#pragma unroll
    for (int q = 0; q < DF_CPT; ++q) {
        const int k = j + tid + q * DF_NT;
        t[q] = x[q] = 0.0;
        if (k <= last) {
            t[q] = U[(int64_t)j * ldu + k + 1];
            if (k > j) x[q] = U[(int64_t)(j + 1) * ldu + k + 1];
            sdiag[k - j] = U[(int64_t)(k + 1) * ldu + k + 1];
        }
    }
    __syncthreads();
    if (m > 0 && tid == 0) {                   // rotation j from column j (owned by thread 0, q = 0)
        const double a = t[0], b = sdiag[0], rho = hypot(a, b);
        const bool id = !(rho > 0.0);
        srot[0][0] = id ? 1.0 : a / rho;
        srot[0][1] = id ? 0.0 : b / rho;
        srot[0][2] = rho;
    }
    __syncthreads();
    for (int i = j; i <= last; ++i) {
        const int slot = (i - j) & 1;
        const double c = srot[slot][0], s = srot[slot][1], rho = srot[slot][2];
        if (tid == 0) {
            rot[2 * (i - j)] = c;
            rot[2 * (i - j) + 1] = s;
        }
#pragma unroll
        for (int q = 0; q < DF_CPT; ++q) {
            const int k = j + tid + q * DF_NT;
            if (k == i) {
                U[(int64_t)i * ldu + i] = rho;
                if (pivots) pivots[i] = rho * rho;
            } else if (k > i && k <= last) {
                const double o = fma(c, t[q], s * x[q]);
                t[q] = fma(c, x[q], -s * t[q]);
                U[(int64_t)i * ldu + k] = o;
            }
        }
        // operands of step i + 1 (columns k > i + 1 read H[i+2, k] = U[i+2, k+1], never a diagonal entry)
#pragma unroll
        for (int q = 0; q < DF_CPT; ++q) {
            const int k = j + tid + q * DF_NT;
            if (k > i + 1 && k <= last) x[q] = U[(int64_t)(i + 2) * ldu + k + 1];
        }
        // the owner of column i + 1 determines rotation i + 1
        const int nk = i + 1;
        if (nk <= last && ((nk - j) % DF_NT) == tid) {
            const int qn = (nk - j) / DF_NT;
            double a = 0.0;
#pragma unroll
            for (int q = 0; q < DF_CPT; ++q)
                if (q == qn) a = t[q];
            const double b = sdiag[nk - j], r = hypot(a, b);
            const bool id = !(r > 0.0);
            srot[slot ^ 1][0] = id ? 1.0 : a / r;
            srot[slot ^ 1][1] = id ? 0.0 : b / r;
            srot[slot ^ 1][2] = r;
        }
        __syncthreads();
    }
    // the (n-1) x (n-1) factor: old column n-1 and row n-1 are cleared
    for (int r = tid; r < n; r += DF_NT) U[(int64_t)r * ldu + n - 1] = 0.0;
    if (tid == 0) {
        if (picks) picks[n - 1] = -1;
        if (scores) scores[n - 1] = 0.0;
        if (pivots) pivots[n - 1] = 0.0;
    }
}

// ---------------------------------------------------------------------------------------------
// The same rotations on rows j..n-1 of a factor W (ncols columns): two adjacent columns per thread (16-byte streaming
// accesses), the rotations staged in shared memory a chunk at a time, 16 rows of loads in flight per thread as in
// gpx_append_two_columns.  Each column is a chain: t = W[j]; for each rotation: W[i] = c t + s W[i+1],
// t = c W[i+1] - s t; finally W[n-1] = t (the residual row) and var += t^2.  Reads and writes 16 (n - j) bytes per column.
// ---------------------------------------------------------------------------------------------
constexpr int DR_NT = 128;
constexpr int DR_CHUNK = 1024;   // rotations per shared-memory chunk (a multiple of 16)

__global__ void __launch_bounds__(DR_NT) delete_rows_kernel(const double* __restrict__ rot, int j, int n,
                                                             double* __restrict__ W, int64_t ldw, int64_t ncols,
                                                             double* __restrict__ var) {
    __shared__ double2 srot[DR_CHUNK];
    const int64_t col = ((int64_t)blockIdx.x * DR_NT + threadIdx.x) * 2;
    const bool active = col < ncols;
    const bool two = col + 1 < ncols;
    const int m = n - 1 - j;
    double* wp = W + col;
    double2 t = make_double2(0.0, 0.0);
    double2 x[16];
    if (active) {
        t = __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)j * ldw));
#pragma unroll
        for (int u = 0; u < 16; ++u)
            x[u] = u < m ? __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)(j + 1 + u) * ldw)) : make_double2(0.0, 0.0);
    }
    for (int r0 = 0; r0 < m; r0 += DR_CHUNK) {
        const int len = m - r0 < DR_CHUNK ? m - r0 : DR_CHUNK;
        __syncthreads();
        for (int i = threadIdx.x; i < len; i += DR_NT) srot[i] = reinterpret_cast<const double2*>(rot)[r0 + i];
        __syncthreads();
        if (!active) continue;
        for (int b = 0; b < len; b += 16) {
            double2 o[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                if (b + u < len) {
                    const double2 cs = srot[b + u];
                    o[u].x = fma(cs.x, t.x, cs.y * x[u].x);
                    o[u].y = fma(cs.x, t.y, cs.y * x[u].y);
                    t.x = fma(cs.x, x[u].x, -cs.y * t.x);
                    t.y = fma(cs.x, x[u].y, -cs.y * t.y);
                }
            }
            const int64_t row0 = (int64_t)j + r0 + b;   // rotated rows row0 .. row0+15
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                if (b + u < len) {
                    double* dst = wp + (row0 + u) * ldw;
                    if (two) __stcs(reinterpret_cast<double2*>(dst), o[u]);
                    else dst[0] = o[u].x;
                }
            }
            // the next 16 rows (they may lie in the next chunk: chunks are whole batches of 16)
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int r = r0 + b + 16 + u;
                if (r < m) x[u] = __ldcs(reinterpret_cast<const double2*>(wp + (int64_t)(j + 1 + r) * ldw));
            }
        }
    }
    if (!active) return;
    double* dst = wp + (int64_t)(n - 1) * ldw;
    if (two) {
        *reinterpret_cast<double2*>(dst) = t;
        var[col] = fma(t.x, t.x, var[col]);
        var[col + 1] = fma(t.y, t.y, var[col + 1]);
    } else {
        dst[0] = t.x;
        var[col] = fma(t.x, t.x, var[col]);
    }
}

// local column of global index g on this rank, or -1: the contiguous block [offset, offset + C) when blk == 0, else the
// block-cyclic map of gpx_local_index_cyclic (global block g / blk lives on rank (g / blk) % world as local block
// (g / blk) / world)
__device__ __forceinline__ int64_t exchange_local(int64_t g, int64_t offset, int64_t blk, int64_t world, int64_t rank,
                                                  int64_t C) {
    int64_t p = g - offset;
    if (blk > 0) p = (g >= 0 && (g / blk) % world == rank) ? ((g / blk) / world) * blk + g % blk : -1;
    return (p >= 0 && p < C) ? p : -1;
}

// keep-or-swap: the removed point (global index *inc) stays unless a challenger beats its own score s, discounted to
// (1 - rtol) s when scores are minimised and inflated to (1 + rtol) s when they are maximised; it wins ties
template <bool MAXIMISE>
__global__ void exchange_keep_kernel(const int64_t* __restrict__ inc, int64_t offset, int64_t blk, int64_t world, int64_t rank,
                                     int64_t C, const double* __restrict__ scores, const double* __restrict__ weights,
                                     double rtol, double* __restrict__ best, int64_t* __restrict__ idx,
                                     double* __restrict__ inc_score) {
    const int64_t p = exchange_local(inc[0], offset, blk, world, rank, C);
    if (p < 0) {
        inc_score[0] = 0.0;
        return;
    }
    const double s = weights ? scores[p] * weights[p] : scores[p];   // the arg-reduce's own product
    inc_score[0] = s;
    const double d = MAXIMISE ? (1.0 + rtol) * s : (1.0 - rtol) * s;
    if (idx[0] < 0 || (MAXIMISE ? d >= best[0] : d <= best[0])) {
        best[0] = d;
        idx[0] = p;
    }
}

__global__ void exchange_unmask_kernel(const int64_t* __restrict__ inc, int64_t offset, int64_t blk, int64_t world,
                                       int64_t rank, int64_t C, uint8_t* __restrict__ mask) {
    const int64_t p = exchange_local(inc[0], offset, blk, world, rank, C);
    if (p >= 0) mask[p] = 0;
}

__global__ void exchange_record_kernel(const int64_t* __restrict__ inc, const double* __restrict__ inc_score, int64_t n,
                                       const int64_t* __restrict__ picks, double* __restrict__ pick_scores,
                                       int64_t* __restrict__ swaps, double* __restrict__ trace) {
    if (picks[n] == inc[0]) {
        if (pick_scores) pick_scores[n] = inc_score[0];
    } else if (swaps) {
        swaps[0] += 1;
    }
    if (trace) trace[0] = pick_scores ? pick_scores[n] : 0.0;
}

}  // namespace

extern "C" int gpx_design_delete_factor(gpx_handle h, double* U, int64_t n, int64_t ldu, int64_t j, double* rot,
                                        int64_t* picks, double* scores, double* pivots, void* stream) {
    GPX_REQUIRE(h && U, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(n >= 1 && j >= 0 && j < n, GPX_EINVAL, "position j must satisfy 0 <= j < n");
    GPX_REQUIRE(ldu >= n, GPX_EINVAL, "ldu < n");
    GPX_REQUIRE(n - 1 - j <= (int64_t)DF_NT * DF_CPT, GPX_ESIZE, "more than 8192 rotations (n - 1 - j)");
    GPX_REQUIRE(rot != nullptr || j == n - 1, GPX_EINVAL, "rot is NULL");
    const size_t smem = (size_t)(n - 1 - j > 0 ? n - 1 - j : 1) * sizeof(double);
    if (smem > 48 * 1024) {
        const int rc = gpx_ensure_smem(h, (const void*)delete_factor_kernel, (size_t)DF_NT * DF_CPT * sizeof(double),
                                       "delete_factor");
        if (rc) return rc;
    }
    const DeleteFactorArgs f{U, ldu, rot, picks, scores, pivots};
    delete_factor_kernel<<<1, DF_NT, smem, (cudaStream_t)stream>>>(f, f, (int)n, (int)j);
    return gpx_check_launch("gpx_design_delete_factor");
}

extern "C" int gpx_design_delete_factors(gpx_handle h, int64_t n, int64_t j, double* U0, int64_t ldu0, double* rot0,
                                         int64_t* picks, double* scores, double* pivots, double* U1, int64_t ldu1,
                                         double* rot1, void* stream) {
    GPX_REQUIRE(h && U0 && U1, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(n >= 1 && j >= 0 && j < n, GPX_EINVAL, "position j must satisfy 0 <= j < n");
    GPX_REQUIRE(ldu0 >= n && ldu1 >= n, GPX_EINVAL, "ldu < n");
    GPX_REQUIRE(n - 1 - j <= (int64_t)DF_NT * DF_CPT, GPX_ESIZE, "more than 8192 rotations (n - 1 - j)");
    GPX_REQUIRE((rot0 != nullptr && rot1 != nullptr && rot0 != rot1) || j == n - 1, GPX_EINVAL,
                "rot0 and rot1 must be two separate buffers");
    GPX_REQUIRE(U0 != U1, GPX_EINVAL, "U0 and U1 must be two separate factors");
    const size_t smem = (size_t)(n - 1 - j > 0 ? n - 1 - j : 1) * sizeof(double);
    if (smem > 48 * 1024) {
        const int rc = gpx_ensure_smem(h, (const void*)delete_factor_kernel, (size_t)DF_NT * DF_CPT * sizeof(double),
                                       "delete_factor");
        if (rc) return rc;
    }
    const DeleteFactorArgs f0{U0, ldu0, rot0, picks, scores, pivots};
    const DeleteFactorArgs f1{U1, ldu1, rot1, nullptr, nullptr, nullptr};
    delete_factor_kernel<<<2, DF_NT, smem, (cudaStream_t)stream>>>(f0, f1, (int)n, (int)j);
    return gpx_check_launch("gpx_design_delete_factors");
}

extern "C" int gpx_design_delete_rows(gpx_handle h, const double* rot, int64_t j, int64_t n, double* W, int64_t ldw,
                                      int64_t ncols, double* var, void* stream) {
    GPX_REQUIRE(h && n >= 1 && j >= 0 && j < n && ncols >= 0, GPX_EINVAL, "bad arguments (0 <= j < n, ncols >= 0)");
    if (ncols == 0) return GPX_OK;
    GPX_REQUIRE(W && var && (rot || j == n - 1), GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE((ldw % 2) == 0 && ldw >= ncols + (ncols & 1) && gpx_aligned16(W) && gpx_aligned16(rot), GPX_EALIGN,
                "W and rot must be 16-byte aligned, ldw even and covering an even column count");
    GPX_REQUIRE(n <= INT32_MAX, GPX_ESIZE, "n too large");
    const unsigned grid = (unsigned)((ncols + 2 * DR_NT - 1) / (2 * DR_NT));
    delete_rows_kernel<<<grid, DR_NT, 0, (cudaStream_t)stream>>>(rot, (int)j, (int)n, W, ldw, ncols, var);
    return gpx_check_launch("gpx_design_delete_rows");
}

extern "C" int gpx_exchange_keep(gpx_handle h, const int64_t* inc, int64_t index_offset, int64_t C, const double* scores,
                                 double rtol, double* best, int64_t* idx, double* inc_score, void* stream) {
    GPX_REQUIRE(h && inc && scores && best && idx && inc_score && C >= 0, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(rtol >= 0.0, GPX_EINVAL, "rtol must be >= 0");
    exchange_keep_kernel<false><<<1, 1, 0, (cudaStream_t)stream>>>(inc, index_offset, 0, 1, 0, C, scores, nullptr, rtol, best,
                                                                    idx, inc_score);
    return gpx_check_launch("gpx_exchange_keep");
}

extern "C" int gpx_exchange_keep_max(gpx_handle h, const int64_t* inc, int64_t index_offset, int64_t blk, int64_t world,
                                     int64_t rank, int64_t C, const double* scores, const double* weights, double rtol,
                                     double* best, int64_t* idx, double* inc_score, void* stream) {
    GPX_REQUIRE(h && inc && scores && best && idx && inc_score && C >= 0, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(blk >= 0 && world >= 1 && rank >= 0 && rank < world, GPX_EINVAL, "blk >= 0, 0 <= rank < world");
    GPX_REQUIRE(rtol >= 0.0, GPX_EINVAL, "rtol must be >= 0");
    exchange_keep_kernel<true><<<1, 1, 0, (cudaStream_t)stream>>>(inc, index_offset, blk, world, rank, C, scores, weights,
                                                                   rtol, best, idx, inc_score);
    return gpx_check_launch("gpx_exchange_keep_max");
}

extern "C" int gpx_exchange_unmask(gpx_handle h, const int64_t* inc, int64_t index_offset, int64_t blk, int64_t world,
                                   int64_t rank, int64_t C, uint8_t* mask, void* stream) {
    GPX_REQUIRE(h && inc && mask && C >= 0, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(blk >= 0 && world >= 1 && rank >= 0 && rank < world, GPX_EINVAL, "blk >= 0, 0 <= rank < world");
    exchange_unmask_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(inc, index_offset, blk, world, rank, C, mask);
    return gpx_check_launch("gpx_exchange_unmask");
}

extern "C" int gpx_exchange_record(gpx_handle h, const int64_t* inc, const double* inc_score, int64_t n, const int64_t* picks,
                                   double* pick_scores, int64_t* swaps, double* trace, void* stream) {
    GPX_REQUIRE(h && inc && inc_score && picks && n >= 0, GPX_EINVAL, "bad arguments");
    exchange_record_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(inc, inc_score, n, picks, pick_scores, swaps, trace);
    return gpx_check_launch("gpx_exchange_record");
}
