/*
 * gpexp_b200 -- C ABI of the B200-native greedy experimental-design hot path.
 *
 * The reference (goroda/GPEXP) is pure Python/numpy and has NO native or FFI layer
 * (SURVEY.md section 8b), so there is no existing binding to mirror: every entry point
 * below cites the reference Python function whose arithmetic it replaces, and
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *     the library never frees caller memory and allocates nothing after gpx_create;
 *   - all arithmetic is IEEE float64;
 *   - point sets are stored dimension-major ("SoA"): coordinate i of point j is X[i*ldx + j];
 *   - matrices are row-major with an explicit leading dimension; leading dimensions and
 *     column offsets handed to the tensor-core routines must be even (16-byte rows);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream and
 *     never synchronise the device unless stated;
 *   - return value: 0 = OK, <0 = bad argument (GPX_E*), >0 = cudaError_t of a failed launch;
 *     gpx_last_error() returns a thread-local host string;
 *   - no exceptions, no exit(), re-entrant per handle, one handle per device;
 *   - a handle's calls share its reduction scratch (arg-reduce / sum tickets and partials): issue them on ONE stream at
 *     a time; use a second handle (gpx_create on the same device) for a second concurrent stream or host thread;
 *   - shared-memory opt-ins are tracked per handle, i.e. per device.
 */
#ifndef GPEXP_B200_H
#define GPEXP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPX_VERSION 200

#define GPX_MAX_DIM 16 /* largest supported input dimension                              */
#define GPX_KROWS 16   /* rows of a prepared side: d scaled coordinates + (alpha, 1) + (1, beta), zero padded;
                          the expanded-form prologue therefore serves d <= 14, larger d use the difference form */

/* kernel families (gpExp/kernels.py) */
#define GPX_SE 0       /* KernelSquaredExponential, iso or ARD      kernels.py:100-123     */
#define GPX_MATERN32 1 /* KernelIsoMatern, nu = 3/2                 kernels.py:72-91       */
#define GPX_MEHLER 2   /* KernelMehlerND / KernelMehler1D           kernels.py:183-293     */

/* error codes */
#define GPX_OK 0
#define GPX_EINVAL (-1)    /* bad argument                                                   */
#define GPX_EALIGN (-2)    /* pointer / leading dimension not 16-byte aligned                */
#define GPX_ENOKERNEL (-3) /* gpx_set_kernel not called                                      */
#define GPX_ESIZE (-4)     /* size exceeds a documented limit                                */
#define GPX_ENOCOMM (-5)   /* collective requested but gpx_comm_init was not called / NCCL not found */

/* covariance prologue of the tensor-core routines */
#define GPX_PRO_EXPANDED 1 /* k = f(sum of products of two prepared sides): one extra DMMA chunk; *_rows arguments are
                              gpx_prep_side outputs.  Cancellation error ~ eps * max|alpha|: see gpx_prep_side.        */
#define GPX_PRO_DIFF 2     /* k = f(sum a (x-y)^2) from raw coordinates (the arithmetic of kernels.py:121-122 itself);
                              *_rows arguments are the dimension-major coordinate arrays.  No cancellation.            */

/* sides of a prepared point set for the tensor-core Gram prologue */
#define GPX_SIDE_A 0 /* the "row" operand (integration points / design rows)                  */
#define GPX_SIDE_B 1 /* the "column" operand (candidates / query points)                      */

/* row sources of gpx_append_row */
#define GPX_ROW_KERNEL 0 /* new row starts from k(x_p, y_j)                                   */
#define GPX_ROW_MATRIX 1 /* new row starts from a given device row (MI precision downdate)    */

typedef struct gpx_context* gpx_handle;

int gpx_version(void);
const char* gpx_last_error(void);
/* kernels launched by this library since it was loaded (process-wide; bench.py reports the difference over its timed
 * region as `gpu_launches`) */
int64_t gpx_launch_count(void);

/* One handle per device.  Allocates a small reduction scratch; nothing else. */
int gpx_create(int device, gpx_handle* out);
int gpx_destroy(gpx_handle h);

/* Kernel family + hyper-parameters.  They travel to every launch as a __grid_constant__ struct,
 * i.e. they live in the constant bank (ARD length-scales in constant memory).
 *   GPX_SE       params_host = cl[0..d) , signalSize           (nparams = d+1)  kernels.py:103-111
 *   GPX_MATERN32 params_host = rho, signalSize                 (nparams = 2)    kernels.py:74-78
 *   GPX_MEHLER   params_host = t[0..d)                          (nparams = d)    kernels.py:185-189 */
int gpx_set_kernel(gpx_handle h, int family, int d, const double* params_host, int nparams);

/* a1  Kernel.evaluate (kernels.py:49-65): out[j] = k(X[j], Y[j]); nx == ny, or one of them 1
 *     (the (1,d) broadcast that the reference does with np.tile).  out has max(nx,ny) entries. */
int gpx_kernel_pairwise(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny,
                        int64_t ldy, double* out, void* stream);

/* k(x,x) per point: the prior variance the cost functions start from (gp.py:251,
 * experimentalDesign.py:816-818, :260). */
int gpx_prior_diag(gpx_handle h, const double* X, int64_t n, int64_t ldx, double* out, void* stream);

/* K1 / a5  calculateCovarianceMatrix (gp_kernel_utilities.py:34-68) generalised to a cross block:
 *     out[i*ld + j] = k(X[i], Y[j]) ; if add_diag: out[i*ld+i] += nugget_vec ? nugget_vec[i] : nugget.
 *     Difference form (x-y)^2, one pass, coalesced stores. */
int gpx_gram(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny, int64_t ldy,
             double* out, int64_t ld, int add_diag, const double* nugget_vec, double nugget, void* stream);

/* K2  Blocked Cholesky of the symmetric row-major matrix A (upper triangle read):  A = U^T U,
 *     U upper-triangular written in place (strictly-lower part left untouched).  Replaces
 *     np.linalg.pinv at gp.py:181 / experimentalDesign.py:268,280,826 for positive-definite Grams.
 *     info[0] = 0 or (1 + index of the first non-positive pivot). */
int gpx_potrf(gpx_handle h, double* A, int64_t n, int64_t ld, int* info, void* stream);

/* K2  Rank-1 append: given U (n x n) and the new column knew[0..n) = k(D, x_new), kpp = k(x,x)+nugget,
 *     writes U[0..n, n] = U^-T knew and U[n,n] = sqrt(kpp - |.|^2).  info as gpx_potrf. */
int gpx_chol_append(gpx_handle h, double* U, int64_t n, int64_t ld, const double* knew, double kpp, int* info,
                    void* stream);

/* Centre subtracted from every coordinate by gpx_prep_side for the stationary families (SE, Matern: k depends on x - y
 * only, kernels.py:121-122, :87-89); ignored for Mehler.  center_host: d doubles, or NULL for the origin.  Both sides
 * of a contraction must be prepared under the same centre. */
int gpx_set_center(gpx_handle h, const double* center_host);

/* Prepared side of a point set for the GPX_PRO_EXPANDED prologue: k(x,y) = f(sum_r rowsA[r][i] * rowsB[r][j]) with
 *     rows  : GPX_KROWS x ld = d scaled coordinates, then (alpha_i | 1) and (1 | beta_j) for side A | B, then zeros;
 *     maxabs (nullable, device): max |alpha| resp. |beta| -- the expanded form loses eps * (max|alpha| + max|beta|) to
 *     cancellation, so the caller switches to GPX_PRO_DIFF when that exceeds its tolerance (1e-11 in gpexp_b200). */
int gpx_prep_side(gpx_handle h, int side, const double* X, int64_t n, int64_t ldx, double* rows, int64_t ld,
                  double* maxabs, void* stream);

/* K1+K3  W = U^-T K(D, Y):  left-looking blocked TRSM whose 128-row blocks of the right-hand side are written straight
 *     into W by the difference-form Gram kernel, updated by the FP64 DMMA routine (the TMA kernel when ldu, ldw are
 *     multiples of 128 covering whole tiles -- zero-initialised padding --, else the predicated one) and finished by a
 *     forward substitution.  Replaces np.dot(precision, kernelvals) at gp.py:253-255 / experimentalDesign.py:836-837.
 *     D: design coordinates (d x ldd), Y: query coordinates (d x ldy).
 *     var_out (nullable): var[j] = k(y_j,y_j) - sum_i W[i,j]^2     (K4, a7 GP.evaluateVariance). */
int gpx_trsm_gram(gpx_handle h, const double* U, int64_t n, int64_t ldu, const double* D, int64_t ldd, const double* Y,
                  int64_t ny, int64_t ldy, double* W, int64_t ldw, double* var_out, void* stream);

/* In-place B <- U^-T B for a materialised right-hand side (n x ncols). */
int gpx_trsm(gpx_handle h, const double* U, int64_t n, int64_t ldu, double* B, int64_t ncols, int64_t ldb,
             void* stream);

/* In-place B <- U^-1 B (back substitution), used for GP.train coefficients (gp.py:101) and the precision
 * matrix.  Ut is the TRANSPOSE of U (lower-triangular, row-major; make it with gpx_transpose) so that the
 * block update operand is K-major for the tensor-core routine. */
int gpx_trsm_back(gpx_handle h, const double* Ut, int64_t n, int64_t ldu, double* B, int64_t ncols, int64_t ldb,
                  void* stream);

/* Y = U^-T as an explicit lower-triangular row-major matrix (zero above the diagonal).  MI set-up:
 * diag((K+noise I)^-1) = column sums of squares of Y, columns of the precision come from gpx_mi_prec_column. */
int gpx_trtri_t(gpx_handle h, const double* U, int64_t n, int64_t ldu, double* Y, int64_t ldy, void* stream);

/* C[i,j] -= sum_k A[k*lda+i] * B[k*ldb+j]   (i<I, j<J, k<K), FP64 DMMA.  upper_only != 0 updates only the entries
 * j >= i and leaves the strictly-lower ones untouched (symmetric rank-k update of the Cholesky trailing matrix). */
int gpx_dgemm_tn_sub(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                     int64_t ldc, int64_t I, int64_t J, int64_t K, int upper_only, void* stream);

/* The same update on the TMA + mbarrier kernel, for callers that GUARANTEE fully padded operands: every 128-wide tile
 * covering A's I columns and B's J columns is readable and finite (lda >= roundup(I,128), ldb >= roundup(J,128) counted
 * from the pointers handed in).  Used by the column-sharded MI set-up. */
int gpx_dgemm_tn_sub_padded(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                            int64_t ldc, int64_t I, int64_t J, int64_t K, int upper_only, void* stream);

/* The padded update for an operand B that is one rank's column slice of a LOWER-triangular matrix (B[k, c] = 0 for
 * k < global(c)) in a block-cyclic column distribution: local column j belongs to global block (j / blk) * world + rank.
 * The structurally-zero leading rows of every 128-column tile are skipped (the Y = U^-T half of the MI set-up executes
 * V^3/3 flop instead of 2 V^3/3).  blk: a multiple of 128. */
int gpx_dgemm_tn_sub_lower(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                           int64_t I, int64_t J, int64_t K, int blk, int world, int rank, void* stream);

/* Pivot record: what one greedy step needs to know about the chosen point.  Layout (doubles):
 *   [0] score  [1] global index (exact integer < 2^53)  [2] var_D(p) + noise (the squared divisor)
 *   [3 .. 3+GPX_MAX_DIM) coordinates of x_p   [GPX_PIVOT_HDR .. GPX_PIVOT_HDR + n) column W[0..n, p]   */
#define GPX_PIVOT_HDR (3 + GPX_MAX_DIM)

/* Fill a pivot record from the local candidate `*idx_dev` (device int64, local index):
 *     rec[1] = index_map ? index_map[*idx_dev] : *idx_dev + index_offset (the GLOBAL index), rec[0] = *score_dev. */
int gpx_gather_pivot(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var, const double* X,
                     int64_t ldx, const double* score_dev, const int64_t* idx_dev, int64_t index_offset,
                     const int64_t* index_map, double noise, double* rec, void* stream);

/* Pick the winning record among `nrec` records spaced `stride` doubles apart (NCCL all-gather output):
 * lowest score if minimize else highest, ties -> lowest global index (np.argmax / np.argmin order). */
int gpx_select_pivot(gpx_handle h, const double* recs, int nrec, int64_t stride, int64_t n, int minimize,
                     double* rec_out, void* stream);

/* K3+K4 incremental: append row n of W for every column j < ncols and update the running variance
 *     w = (src_j - sum_{i<n} rec.col[i] * W[i,j]) / sqrt(rec[2]);  W[n,j] = w;  var[j] -= w*w
 *     src_j = k(x_p, Y[j]) (GPX_ROW_KERNEL; experimentalDesign.py:829-837, gp.py:246-256 restated
 *     incrementally) or src_row[j] (GPX_ROW_MATRIX).  HBM-bound: reads 8*n*ncols bytes. */
int gpx_append_row(gpx_handle h, int row_source, const double* rec, const double* src_row, const double* Y,
                   int64_t ncols, int64_t ldy, double* W, int64_t ldw, int64_t n, double* var, void* stream);

/* K7  arg-reduce with np.argmax/np.argmin tie-break (lowest index).  score_j = v[j] * (weights?weights[j]:1);
 *     entries with mask[j] != 0 are skipped.  best[0] = score, idx[0] = local index (-1 if all masked). */
int gpx_argreduce(gpx_handle h, const double* v, const double* weights, const uint8_t* mask, int64_t n,
                  int minimize, double* best, int64_t* idx, void* stream);

/* Deterministic sum of n doubles (fixed tree order). */
int gpx_sum(gpx_handle h, const double* v, int64_t n, double* out, void* stream);

/* Operand pipeline of the IVAR contraction kernel (A/B measurements; results are bit-identical): 0 = 32-row chunks x 3
 * stages fed by one bulk copy per operand row; 1 = the same ring fed by one 2-D tensor-map TMA load per operand chunk;
 * 2 = 24-row chunks x 4 stages, two chunks ahead, tensor-map loads. */
int gpx_set_ivar_ring(gpx_handle h, int ring);

/* Arithmetic of the IVAR contraction on padded operands (leading dimensions covering whole 128-wide tiles):
 *     GPX_CORE_I8    (default) W_M^T W_C emulated exactly enough on the INT8 tensor cores: 7 fixed-point 8-bit slices
 *                    per factor entry, 28 slice products, error <= 7.04 n 2^-52 max|W_M[:,m]| max|W_C[:,c]| per pair
 *                    plus one FP64 rounding (DESIGN.md section 5).  Needs the scratch of gpx_set_ivar_scratch and
 *                    1 <= n <= GPX_I8_MAX_N; otherwise the call uses the FP64 core.
 *     GPX_CORE_DMMA  the FP64 DMMA kernel (ring per gpx_set_ivar_ring).
 * Unpadded operands always use the FP64 generic core.  The GPX_IVAR_CORE environment variable (dmma | i8) sets the
 * default of new handles. */
#define GPX_CORE_DMMA 1
#define GPX_CORE_I8 2
#define GPX_I8_MAX_N 16384 /* largest design size the INT8 core runs */
int gpx_set_ivar_core(gpx_handle h, int core);

/* Bytes of scratch the INT8 core needs for M integration points, C candidates and designs up to n_max points. */
int64_t gpx_ivar_scratch_bytes(gpx_handle h, int64_t M, int64_t C, int64_t n_max);

/* Caller memory (any alignment; NULL, 0 to detach) the INT8 core re-slices the factors into on every scoring call.
 * The handle only keeps the pointer; calls on the handle's stream use it in order. */
int gpx_set_ivar_scratch(gpx_handle h, void* scratch, int64_t bytes);

/* Workspace (doubles) gpx_score_ivar needs for C candidates. */
int64_t gpx_score_ivar_workspace(gpx_handle h, int64_t M, int64_t C);

/* K5+K7  IVAR cost of design+{c} for every candidate c (restates the per-candidate
 *     costFunctionGP_IVAR.evaluate loop, experimentalDesign.py:105-117 -> gp.py:178-181,246-256):
 *         r[c]     = sum_m ( k(m,c) - sum_{i<n} Wm[i,m] Wc[i,c] )^2            FP64 DMMA contraction
 *         cost[c]  = | sum(varM)/M - (r[c] / (varC[c] + noise)) / M |           (reduction = 0 if the
 *                    denominator is numerically zero: the pinv null-direction rule, SURVEY.md section 7)
 *     then arg-min with lowest-index tie-break into best/idx (a NaN score wins, as in np.argmin).  mask (nullable):
 *     candidates with mask[c] != 0 are skipped by the arg-min (their scores are still written); if all are masked,
 *     best[0] = 0.0 and idx[0] = -1.
 *     Ma_rows : integration points, Cb_rows : candidates -- per `prologue` the prepared sides (GPX_SIDE_A / GPX_SIDE_B)
 *     or the raw coordinates; leading dimensions ldm / ldc. */
int gpx_score_ivar(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* varM, const double* Ma_rows,
                   int64_t M, const double* Wc, int64_t ldc, const double* varC, const double* Cb_rows, int64_t C, int64_t n,
                   double noise, double zero_tol, const uint8_t* mask, double* workspace, double* score_out, double* best,
                   int64_t* idx, void* stream);

/* ---- Resident posterior covariance: the HBM-bound alternative for greedy IVAR loops (SURVEY.md section 7) -----------
 * cov (M x ldcov, row m = integration point, 8*M*C bytes resident) holds cov_D(m,c); each greedy step is ONE pass
 *     cov -= a b^T ,  partial[seg][c] = sum_{m in seg} cov[m,c]^2          (16 B of HBM traffic per pair, any n)
 * a = new row of W_M (M), b = new row of W_C (C); a = b = NULL only reduces.  partial: gpx_cov_segments(M, C) x ldp. */
int gpx_cov_segments(int64_t M, int64_t C);
int gpx_cov_update(gpx_handle h, double* cov, int64_t ldcov, int64_t M, int64_t C, const double* a, const double* b,
                   double* partial, int64_t ldp, void* stream);
/* cov = K(mc, cand) - Wm^T Wc for a given design (DMMA contraction, Gram in the prologue); n = 0 gives K itself. */
int gpx_cov_from_factors(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* Ma_rows, int64_t M,
                         const double* Wc, int64_t ldc, const double* Cb_rows, int64_t C, int64_t n, double* cov, int64_t ldcov,
                         void* stream);
/* IVAR costs + arg-min from the per-segment sums (same finalisation as gpx_score_ivar). */
int gpx_score_ivar_partials(gpx_handle h, const double* partial, int nseg, int64_t ldp, const double* varM, int64_t M,
                            const double* varC, int64_t C, double noise, double zero_tol, const uint8_t* mask,
                            double* score_out, double* best, int64_t* idx, void* stream);

/* K6  MI score = num_var[j] / (1/prec_diag[j] - noise), arg-max over unmasked j
 *     (experimentalDesign.py:259-285 restated: denominator = 1/[(K_SS+noise I)^-1]_yy - noise). */
int gpx_score_mi(gpx_handle h, const double* num_var, const double* prec_diag, double noise, const uint8_t* mask,
                 int64_t n, double* score_out, double* best, int64_t* idx, void* stream);

/* K6  column p of P = Y^T Y for the lower-triangular Y = U^-T:  out[i] = sum_{k >= max(i,p)} Y[k,i] Y[k,p].
 *     Y is nrows x ncols (row-major): the whole matrix (col_offset = 0, ncols = nrows, ycol = NULL) or the column slice
 *     [col_offset, col_offset+ncols) owned by this rank, in which case column p arrives as the dense vector ycol[nrows]
 *     (all-reduced from its owner).  *p_dev is the GLOBAL index.  workspace: gpx_mi_prec_column_workspace doubles.
 *     cyclic_blk > 0: the slice is block-cyclic instead of contiguous -- local column i is global column
 *     ((i / blk) * cyclic_world + col_offset) * blk + i % blk, col_offset being the rank; blk a multiple of 256. */
int64_t gpx_mi_prec_column_workspace(int64_t nrows, int64_t ldy);
int gpx_mi_prec_column(gpx_handle h, const double* Y, int64_t nrows, int64_t ncols, int64_t ldy, int64_t col_offset,
                       int64_t cyclic_blk, int64_t cyclic_world, const int64_t* p_dev, const double* ycol, double* workspace,
                       double* out, void* stream);

/* Sharded pools: copy column *idx_dev of W (n rows) into rec[GPX_PIVOT_HDR..] and var[*idx_dev] into rec[2];
 * nothing is written when *idx_dev < 0, so zeroed records can be summed across ranks (owner contributes). */
int gpx_gather_column(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var, const int64_t* idx_dev,
                      double* rec, void* stream);

/* out2[0] = local index of the pivot in rec (global index rec[1]) for the block [offset, offset+count), or -1;
 * out2[1] = the global index. */
int gpx_local_index(gpx_handle h, const double* rec, int64_t offset, int64_t count, int64_t* out2, void* stream);
/* the same for a block-cyclic distribution (global g on rank (g / blk) % world at ((g / blk) / world) * blk + g % blk) */
int gpx_local_index_cyclic(gpx_handle h, const double* rec, int64_t blk, int64_t world, int64_t rank, int64_t count,
                           int64_t* out2, void* stream);
/* A[rows[j] * ld + j] += value, j < n (nugget / identity on the diagonal of a scattered column subset) */
int gpx_add_at_rows(gpx_handle h, double* A, int64_t ld, const int64_t* rows, int64_t n, double value, void* stream);

/* Column sums of squares: out[j] = sum_{i<n} W[i,j]^2 (optionally out[j] = base[j] - that). */
int gpx_colsumsq(gpx_handle h, const double* W, int64_t n, int64_t ncols, int64_t ldw, const double* base,
                 double* out, void* stream);

/* Small utilities the host layer needs so that no arithmetic runs on the CPU. */
int gpx_transpose(gpx_handle h, const double* in, int64_t rows, int64_t cols, int64_t ld_in, double* out,
                  int64_t ld_out, void* stream);
int gpx_set_mask(gpx_handle h, uint8_t* mask, const int64_t* idx_dev, uint8_t value, void* stream);
/* history of a greedy run: picks[n] = rec global index, scores[n] = rec score, pivots[n] = rec[2] (var_D(p) + noise, the
 * number whose smallness flags an ill-conditioned design), column n of the design factor U (each nullable) */
int gpx_store_pivot(gpx_handle h, const double* rec, int64_t n, double* U, int64_t ldu, int64_t* picks,
                    double* scores, double* pivots, void* stream);

/* ---- N1  collectives (SURVEY.md 8b).  NCCL is resolved at run time (dlopen of libnccl.so.2, preferring the copy the
 * process already loaded); a caller that never shards never needs it.  One communicator per handle. --------------------- */
#define GPX_COMM_ID_BYTES 128
/* rank 0: fill id_host (GPX_COMM_ID_BYTES bytes) and hand it to every rank by any host channel */
int gpx_comm_unique_id(void* id_host, int nbytes);
int gpx_comm_init(gpx_handle h, const void* id_host, int rank, int nranks);
int gpx_comm_destroy(gpx_handle h);
int gpx_comm_size(gpx_handle h); /* 0 without a communicator */
/* recv[r*count .. (r+1)*count) = rank r's send[0..count) : the pivot-record exchange of a sharded greedy step */
int gpx_comm_allgather(gpx_handle h, const double* send, double* recv, int64_t count, void* stream);
int gpx_comm_bcast(gpx_handle h, double* buf, int64_t count, int root, void* stream);
int gpx_comm_allreduce_sum(gpx_handle h, double* buf, int64_t count, void* stream);

/* ---- Whole greedy loops in one call: steps n_begin .. n_end-1 issued back to back on `stream`, no host round trip.
 * The structs only carry device pointers and sizes the caller already owns (layouts as in the per-step entry points).
 * With a communicator of more than one rank and rec_all != NULL every step exchanges the ranks' pivot records
 * (ncclAllGather of 19+n doubles) and all ranks append the same winner. ---------------------------------------------- */
typedef struct gpx_ivar_state {
    const double* Xm;      /* integration points, d x ldm (replicated on every rank) */
    int64_t M, ldm;
    double* Wm;            /* ncap x ldm */
    double* varM;          /* ldm */
    const double* Ma_rows; /* prologue rows of the integration points (prepared side A or raw coordinates) */
    const double* Xc;      /* local candidates, d x ldc */
    int64_t C, ldc;
    double* Wc;            /* ncap x ldc */
    double* varC;          /* ldc */
    const double* Cb_rows; /* prologue rows of the candidates (prepared side B or raw coordinates) */
    int64_t ncap;          /* rows allocated in Wm / Wc */
    int64_t index_offset;  /* global index of local candidate 0 */
    int prologue;          /* GPX_PRO_EXPANDED | GPX_PRO_DIFF */
    int nseg;              /* resident mode: gpx_cov_segments(M, C) */
    double noise, zero_tol;
    double* workspace;     /* gpx_score_ivar_workspace doubles */
    double* scores;        /* ldc */
    double* best;          /* 1 */
    int64_t* idx;          /* 1 */
    double* rec;           /* GPX_PIVOT_HDR + ncap */
    double* rec_all;       /* comm_size x (GPX_PIVOT_HDR + ncap), or NULL */
    double* rec_win;       /* GPX_PIVOT_HDR + ncap, or NULL */
    double* U;             /* nullable: ncap x ldu design factor (K_DD + noise I = U^T U), grown column by column */
    int64_t ldu;
    int64_t* picks;        /* ncap */
    double* pick_scores;   /* nullable, ncap */
    double* pick_pivots;   /* nullable, ncap */
    double* cov;           /* nullable: resident posterior covariance M x ldcov -> rank-1 update instead of the contraction */
    int64_t ldcov, ldp;
} gpx_ivar_state;

/* discrete greedy IVAR (SURVEY.md 3.2: arg-min over c of costFunctionGP_IVAR.evaluate(design + [c]),
 * experimentalDesign.py:79-117), steps n_begin .. n_end-1 */
int gpx_ivar_greedy_run(gpx_handle h, const gpx_ivar_state* s, int64_t n_begin, int64_t n_end, void* stream);

/* The same loop as ONE cooperative kernel launch (three grid-wide phases per step), for a resident single-GPU state
 * (s->cov != NULL): removes the per-launch issue cost that bounds small problems such as BASELINE configs[0]
 * (1 000 candidates x 10 000 integration points: 20 steps in 0.72 ms instead of 1.2 ms, measured on B200).  Entry and
 * exit state are those of gpx_ivar_greedy_run, so the two can be mixed within one design.  n_end <= 1024; cov and W_C
 * 16-byte aligned with even leading dimensions. */
int gpx_ivar_greedy_small(gpx_handle h, const gpx_ivar_state* s, int64_t n_begin, int64_t n_end, void* stream);

typedef struct gpx_var_state {
    const double* X;       /* local pool, d x ld */
    int64_t C, ld;
    double* W;             /* ncap x ld */
    double* var;           /* ld */
    const double* weights; /* nullable, C */
    int64_t ncap, index_offset;
    double noise;          /* nugget of the pivoted factorisation: 0.0 for the reference driver (experimentalDesign.py:825) */
    double* best;
    int64_t* idx;
    double* rec;
    double* rec_all;
    double* rec_win;
    int64_t* picks;
    double* pick_scores;
    double* pick_pivots;
} gpx_var_state;

/* performGreedyVarExperimentalDesign (experimentalDesign.py:787-845), steps n_begin .. n_end-1 */
int gpx_var_greedy_run(gpx_handle h, const gpx_var_state* s, int64_t n_begin, int64_t n_end, void* stream);

/* sizeof(gpx_ivar_state) (which = 0) / sizeof(gpx_var_state) (which = 1) as compiled into the library */
int64_t gpx_state_bytes(int which);

/* ---- SURVEY.md 8(f): callers of the hot path (continuous optimisers, model fitting) --------------------------- */

/* Kernel derivative Gram, squared-exponential only (kernels.py:146-181, KernelSquaredExponential.derivative):
 *     out[i*ld + j*d + k] = -signalSize * (Y[j]_k - X[i]_k) / cl_k^2 * k(Y[j], X[i])   (the reference's formula,
 *     which carries signalSize twice).  ld >= ny*d. */
int gpx_se_dgram(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny, int64_t ldy,
                 double* out, int64_t ld, void* stream);

/* Posterior-variance gradient with respect to the design coordinates (GP.evaluateVarianceDerivative, gp.py:282-341):
 *     out[(j*d+k)*ldx + m] = 2 At[j,m] ( D(x_m, p_j)[k] - Qneg[(j*d+k), m] ) - At[j,m]^2 diag[j*d+k],
 *     At = P K(D, X) (n x ldx), Qneg = -(dK/dp)^T At from gpx_se_dgram + gpx_dgemm_tn_sub.  P: design points, X: query
 *     points.  diag (nullable): d noise(p_j)/d p_j[k] of a heteroscedastic noise function (gp.py:314-318), the caller
 *     having added the same numbers to the derivative Gram before forming Qneg. */
int gpx_se_var_grad(gpx_handle h, const double* P, int64_t n, int64_t ldp, const double* X, int64_t M, int64_t ldx,
                    const double* At, const double* Qneg, const double* diag, double* out, void* stream);

/* f3  Hyper-parameter gradient of the marginal log-likelihood, squared-exponential kernels (gp.py:447-468 with
 *     kernels.py:125-144):  out[q] = 1/2 tr((alpha alpha^T - P) dK/dtheta_q), theta = cl_0..cl_{d-1}, signalSize, noise
 *     (d + 2 entries; the noise entry is the bare trace -- the caller applies the reference's 2*noise factor).
 *     P: precision (n x ldp), alpha = P y.  workspace: gpx_se_loglike_grad_workspace(n, d) doubles. */
int64_t gpx_se_loglike_grad_workspace(int64_t n, int d);
int gpx_se_loglike_grad(gpx_handle h, const double* X, int64_t n, int64_t ldx, const double* P, int64_t ldp,
                        const double* alpha, double* workspace, double* out, void* stream);

/* f4  Matrix-free Gram x vector: out[i] = sum_j k(X[i], Y[j]) b[j]   (covTimesV, gp_kernel_utilities.py:107-142: the
 *     linear operator inside the Nystrom eigen-solver).  workspace: gpx_gram_matvec_workspace(n) doubles. */
int64_t gpx_gram_matvec_workspace(int64_t n);
int gpx_gram_matvec(gpx_handle h, const double* X, int64_t n, int64_t ldx, const double* Y, int64_t m, int64_t ldy,
                    const double* b, double* workspace, double* out, void* stream);

/* Dense helpers of the FITC (sparse-GP) precision, gp_kernel_utilities.py:70-104 / gp.py:182-208:
 *     gpx_scale_rows_cols  out[i,j] = scale * A[i,j] * (r ? r[i] : 1) * (c ? c[j] : 1)
 *     gpx_diag_update      A[i,i]   = scale * A[i,i] + (d ? d[i] : shift)
 *     gpx_axpby            y        = alpha x + beta y
 *     gpx_coldot           out[j]   = (base ? base[j] : 0) - sum_i A[i,j] B[i,j]      (k^T P k with P k materialised) */
int gpx_scale_rows_cols(gpx_handle h, const double* A, int64_t rows, int64_t cols, int64_t lda, const double* r,
                        const double* c, double scale, double* out, int64_t ldo, void* stream);
int gpx_diag_update(gpx_handle h, double* A, int64_t n, int64_t ld, double scale, const double* d, double shift, void* stream);
int gpx_axpby(gpx_handle h, int64_t n, double alpha, const double* x, double beta, double* y, void* stream);
int gpx_coldot(gpx_handle h, const double* A, const double* B, int64_t n, int64_t ncols, int64_t ld, const double* base,
               double* out, void* stream);

/* out[r] = scale * sum_c A[r,c], fixed order (row mean of the gradient matrix = costFunctionGP_IVAR.derivative,
 * experimentalDesign.py:166-169). */
int gpx_rowsum(gpx_handle h, const double* A, int64_t rows, int64_t cols, int64_t ld, double scale, double* out, void* stream);

/* out[0] = log det(U^T U) = 2 sum log U_ii  (np.linalg.slogdet at gp.py:432 for the marginal log-likelihood). */
int gpx_logdet_chol(gpx_handle h, const double* U, int64_t n, int64_t ld, double* out, void* stream);

/* Yard-stick kernels used only by bench.py to establish the FP64 ceilings on the box. */
int gpx_bench_dmma(gpx_handle h, int64_t iters, double* sink, void* stream);
int gpx_bench_dfma(gpx_handle h, int64_t iters, double* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPEXP_B200_H */
