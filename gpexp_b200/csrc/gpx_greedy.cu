// Whole greedy loops behind ONE C-ABI call, and the collectives they need.
//
// The per-step sequence of the greedy drivers (experimentalDesign.py:787-845 and the discrete IVAR driver of SURVEY.md 3.2)
// is a handful of small launches around one big one; issued from Python through ctypes the small ones cost ~10 us each and
// dominate the small configurations (cfg-1: 20 steps x 1 000 candidates).  gpx_ivar_greedy_run / gpx_var_greedy_run issue
// the same launches back to back from C, with the bookkeeping fused:
//
//   IVAR step   sum(varM) -> contraction (or resident partials) -> finalise + arg-min -> gather pivot (+ store)
//               [-> ncclAllGather -> select (+ store)] -> append row to W_C and W_M (one launch) [-> cov -= a b^T]
//   var step    arg-max -> gather pivot (+ store) [-> ncclAllGather -> select (+ store)] -> append row
//
// Nothing is read back: picks / scores / pivots accumulate in device arrays the caller reads once at the end.
//
// NCCL is resolved at run time (dlopen of the libnccl.so.2 the process already has, e.g. the one PyTorch loaded), so the
// library has no link-time dependency on it; a caller that never calls gpx_comm_init never touches it.
#include <cooperative_groups.h>
#include <dlfcn.h>
#include <math.h>
#include <string.h>

#include "gpx_common.cuh"

// ---------------------------------------------------------------------------------------------
// N1  collectives (SURVEY.md 8b): ncclAllGather of pivot records, broadcast / all-reduce for the MI set-up
// ---------------------------------------------------------------------------------------------
namespace {

struct NcclId {
    char internal[128];  // ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128), passed by value like the original
};
typedef void* NcclComm;
enum { NCCL_FLOAT64 = 8, NCCL_SUM = 0 };

struct NcclApi {
    void* lib;
    int (*GetUniqueId)(NcclId*);
    int (*CommInitRank)(NcclComm*, int, NcclId, int);
    int (*CommDestroy)(NcclComm);
    int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t);
    int (*Broadcast)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t);
    int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t);
    const char* (*GetErrorString)(int);
};
NcclApi g_nccl = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

int nccl_load() {
    if (g_nccl.lib) return GPX_OK;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the copy the process already uses, if any
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) {
        gpx_set_error("gpx_comm: libnccl.so.2 not found (%s)", dlerror());
        return GPX_ENOCOMM;
    }
    NcclApi a;
    a.lib = lib;
    a.GetUniqueId = (int (*)(NcclId*))dlsym(lib, "ncclGetUniqueId");
    a.CommInitRank = (int (*)(NcclComm*, int, NcclId, int))dlsym(lib, "ncclCommInitRank");
    a.CommDestroy = (int (*)(NcclComm))dlsym(lib, "ncclCommDestroy");
    a.AllGather = (int (*)(const void*, void*, size_t, int, NcclComm, cudaStream_t))dlsym(lib, "ncclAllGather");
    a.Broadcast = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclBroadcast");
    a.AllReduce = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclAllReduce");
    a.GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllGather || !a.Broadcast || !a.AllReduce) {
        gpx_set_error("gpx_comm: libnccl.so.2 lacks a required symbol");
        return GPX_ENOCOMM;
    }
    g_nccl = a;
    return GPX_OK;
}

int nccl_check(int r, const char* what) {
    if (r == 0) return GPX_OK;
    gpx_set_error("%s: NCCL error %d (%s)", what, r, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    return 10000 + r;
}

}  // namespace

extern "C" int gpx_comm_unique_id(void* id_host, int nbytes) {
    GPX_REQUIRE(id_host && nbytes >= GPX_COMM_ID_BYTES, GPX_EINVAL, "id buffer must hold GPX_COMM_ID_BYTES bytes");
    int rc = nccl_load();
    if (rc) return rc;
    NcclId id;
    rc = nccl_check(g_nccl.GetUniqueId(&id), "ncclGetUniqueId");
    if (rc) return rc;
    memcpy(id_host, id.internal, GPX_COMM_ID_BYTES);
    return GPX_OK;
}

extern "C" int gpx_comm_init(gpx_handle h, const void* id_host, int rank, int nranks) {
    GPX_REQUIRE(h && id_host && nranks >= 1 && rank >= 0 && rank < nranks, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE(h->nccl_comm == nullptr, GPX_EINVAL, "this handle already has a communicator");
    int rc = nccl_load();
    if (rc) return rc;
    NcclId id;
    memcpy(id.internal, id_host, GPX_COMM_ID_BYTES);
    cudaSetDevice(h->device);
    NcclComm comm = nullptr;
    rc = nccl_check(g_nccl.CommInitRank(&comm, nranks, id, rank), "ncclCommInitRank");
    if (rc) return rc;
    h->nccl_comm = comm;
    h->comm_rank = rank;
    h->comm_size = nranks;
    return GPX_OK;
}

extern "C" int gpx_comm_destroy(gpx_handle h) {
    if (!h || !h->nccl_comm) return GPX_OK;
    int rc = nccl_check(g_nccl.CommDestroy((NcclComm)h->nccl_comm), "ncclCommDestroy");
    h->nccl_comm = nullptr;
    h->comm_size = 0;
    return rc;
}

extern "C" int gpx_comm_size(gpx_handle h) { return (h && h->nccl_comm) ? h->comm_size : 0; }

extern "C" int gpx_comm_allgather(gpx_handle h, const double* send, double* recv, int64_t count, void* stream) {
    GPX_REQUIRE(h && h->nccl_comm, GPX_ENOCOMM, "gpx_comm_init has not been called");
    GPX_REQUIRE(send && recv && count >= 0, GPX_EINVAL, "bad arguments");
    return nccl_check(g_nccl.AllGather(send, recv, (size_t)count, NCCL_FLOAT64, (NcclComm)h->nccl_comm, (cudaStream_t)stream),
                      "ncclAllGather");
}

extern "C" int gpx_comm_bcast(gpx_handle h, double* buf, int64_t count, int root, void* stream) {
    GPX_REQUIRE(h && h->nccl_comm, GPX_ENOCOMM, "gpx_comm_init has not been called");
    GPX_REQUIRE(buf && count >= 0 && root >= 0 && root < h->comm_size, GPX_EINVAL, "bad arguments");
    return nccl_check(g_nccl.Broadcast(buf, buf, (size_t)count, NCCL_FLOAT64, root, (NcclComm)h->nccl_comm, (cudaStream_t)stream),
                      "ncclBroadcast");
}

extern "C" int gpx_comm_allreduce_sum(gpx_handle h, double* buf, int64_t count, void* stream) {
    GPX_REQUIRE(h && h->nccl_comm, GPX_ENOCOMM, "gpx_comm_init has not been called");
    GPX_REQUIRE(buf && count >= 0, GPX_EINVAL, "bad arguments");
    return nccl_check(g_nccl.AllReduce(buf, buf, (size_t)count, NCCL_FLOAT64, NCCL_SUM, (NcclComm)h->nccl_comm,
                                       (cudaStream_t)stream),
                      "ncclAllReduce");
}

// ---------------------------------------------------------------------------------------------
// fused pivot bookkeeping
// ---------------------------------------------------------------------------------------------
namespace {

struct PivotSinks {
    double* U;          // nullable: design factor, column n receives the pivot's W column, U[n,n] = sqrt(pivot)
    int64_t ldu;
    int64_t* picks;     // nullable
    double* scores;     // nullable
    double* pivots;     // nullable
};

__device__ __forceinline__ void sink_header(const PivotSinks& k, int n, double score, double gidx, double pivot) {
    if (k.U) k.U[(int64_t)n * k.ldu + n] = sqrt(pivot);
    if (k.picks) k.picks[n] = (int64_t)gidx;
    if (k.scores) k.scores[n] = score;
    if (k.pivots) k.pivots[n] = pivot;
}

// rec <- pivot record of local candidate *idx ; with `store` the history / factor column are written as well
// (single-rank runs: the local record IS the winner)
__global__ void __launch_bounds__(256) gather_store_kernel(const double* __restrict__ W, int64_t ldw, int n,
                                                            const double* __restrict__ var, const double* __restrict__ X,
                                                            int64_t ldx, int d, const double* __restrict__ score,
                                                            const int64_t* __restrict__ idx, int64_t offset, double noise,
                                                            double* __restrict__ rec, int store, PivotSinks k) {
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
            const double sc = score ? score[0] : 0.0, piv = var[p] + noise;
            rec[0] = sc;
            rec[1] = (double)(p + offset);
            rec[2] = piv;
            if (store) sink_header(k, n, sc, (double)(p + offset), piv);
        }
        if (threadIdx.x < GPX_MAX_DIM) rec[3 + threadIdx.x] = threadIdx.x < d ? X[threadIdx.x * ldx + p] : 0.0;
    }
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const double w = W[(int64_t)i * ldw + p];
        rec[GPX_PIVOT_HDR + i] = w;
        if (store && k.U) k.U[(int64_t)i * k.ldu + n] = w;
    }
}

// winner among the ranks' records (better score, ties to the lowest global index) -> out, history, factor column
__global__ void __launch_bounds__(256) select_store_kernel(const double* __restrict__ recs, int nrec, int64_t stride, int n,
                                                            int minimize, double* __restrict__ out, PivotSinks k) {
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
    for (int i = blockIdx.x * 256 + threadIdx.x; i < GPX_PIVOT_HDR + n; i += gridDim.x * 256) {
        const double v = src[i];
        out[i] = v;
        if (k.U && i >= GPX_PIVOT_HDR) k.U[(int64_t)(i - GPX_PIVOT_HDR) * k.ldu + n] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) sink_header(k, n, src[0], src[1], src[2]);
}

// K3+K4 for TWO factors in one launch (greedy IVAR appends the same pivot's row to W_C and to W_M): blocks
// [0, blocks0) serve matrix 0, the rest matrix 1.  Same arithmetic as append_row_kernel<FAM, GPX_ROW_KERNEL>.
struct AppendSide {
    const double* Y;
    int64_t ncols, ldy;
    double* W;
    int64_t ldw;
    double* var;
};

template <int FAM, int NT>
__global__ void __launch_bounds__(NT) append_row2_kernel(const __grid_constant__ KParams kp, const double* __restrict__ rec,
                                                          AppendSide s0, AppendSide s1, unsigned blocks0, int n) {
    extern __shared__ double sl[];
    const bool first = blockIdx.x < blocks0;
    const AppendSide& s = first ? s0 : s1;
    const int64_t j = ((int64_t)(first ? blockIdx.x : blockIdx.x - blocks0) * NT + threadIdx.x) * 2;
    gpx_append_two_columns<FAM, true>(kp, rec, nullptr, s.Y, s.ncols, s.ldy, s.W, s.ldw, n, s.var, j, sl, NT);
}

int launch_gather_store(gpx_handle h, const double* W, int64_t ldw, int64_t n, const double* var, const double* X, int64_t ldx,
                        const double* score, const int64_t* idx, int64_t offset, double noise, double* rec, int store,
                        const PivotSinks& k, cudaStream_t st) {
    unsigned grid = (unsigned)((n + 255) / 256);
    if (grid < 1) grid = 1;
    if (grid > 64) grid = 64;
    gather_store_kernel<<<grid, 256, 0, st>>>(W, ldw, (int)n, var, X, ldx, h->kp.d, score, idx, offset, noise, rec, store, k);
    return gpx_check_launch("greedy gather");
}

int launch_select_store(const double* recs, int nrec, int64_t stride, int64_t n, int minimize, double* out, const PivotSinks& k,
                        cudaStream_t st) {
    unsigned grid = (unsigned)((GPX_PIVOT_HDR + n + 255) / 256);
    if (grid > 64) grid = 64;
    select_store_kernel<<<grid, 256, 0, st>>>(recs, nrec, stride, (int)n, minimize, out, k);
    return gpx_check_launch("greedy select");
}

bool side_ok(const AppendSide& s) {
    return s.Y && s.W && s.var && s.ncols >= 1 && (s.ldw % 2) == 0 && s.ldw >= s.ncols + (s.ncols & 1) && (s.ldy % 2) == 0 &&
           s.ldy >= s.ncols + (s.ncols & 1) && gpx_aligned16(s.W) && gpx_aligned16(s.Y);
}

template <int FAM>
int launch_append2_fam(gpx_handle h, const double* rec, const AppendSide& s0, const AppendSide& s1, int64_t n, cudaStream_t st) {
    const size_t smem = (size_t)((n + 15) / 16 * 16) * sizeof(double);
    if (smem > 48 * 1024) {
        int rc = gpx_ensure_smem(h, (const void*)append_row2_kernel<FAM, 128>, 200 * 1024, "append_row2");
        if (rc) return rc;
    }
    const unsigned b0 = (unsigned)((s0.ncols + 255) / 256), b1 = (unsigned)((s1.ncols + 255) / 256);
    append_row2_kernel<FAM, 128><<<b0 + b1, 128, smem, st>>>(h->kp, rec, s0, s1, b0, (int)n);
    return gpx_check_launch("greedy append");
}

int launch_append2(gpx_handle h, const double* rec, const AppendSide& s0, const AppendSide& s1, int64_t n, cudaStream_t st) {
    int rc = GPX_OK;
    GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_append2_fam<FAM>(h, rec, s0, s1, n, st)));
    return rc;
}

// exchange of the ranks' pivot records: only the live part (header + n) travels
int exchange(gpx_handle h, const double* rec, double* rec_all, double* rec_win, int64_t n, int minimize, const PivotSinks& k,
             cudaStream_t st) {
    const int64_t live = GPX_PIVOT_HDR + n;
    int rc = gpx_comm_allgather(h, rec, rec_all, live, st);
    if (rc) return rc;
    return launch_select_store(rec_all, h->comm_size, live, n, minimize, rec_win, k, st);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Small problems (configs[0]: 1 000 candidates x 10 000 MC points): the whole greedy IVAR loop as ONE cooperative kernel.
// The multi-launch loop above is bound by launch issue (~12 us per launch, 5 per step); here a step is three grid-wide
// phases separated by grid.sync():
//   A  scores from the resident column sums (same finalisation as ivar_finalize_argmin_kernel) + per-block arg-min
//   B  global arg-min (every block, identical), pivot record, new rows of W_C and W_M, running variances, history
//   C  cov -= w_M[n] w_C[n]^T with the next step's column sums of squares (same layout as gpx_cov_update)
// State conventions at entry and exit are those of the resident engine (cov current, partial sums valid), so the two
// paths can be mixed.  The winner's pivot var_D(p) + noise travels with the block results: it must be read before any
// block starts updating the variances in phase B.
// WT: weighted integration points (s.wM): sum w varM and the weighted column sums, in the same trees; nothing / M.
// ---------------------------------------------------------------------------------------------
namespace {
namespace cg = cooperative_groups;
constexpr int SMALL_NCAP = 1024;   // design points whose pivot column fits the shared-memory buffer
constexpr int SMALL_SEG_PER_WARP = 20;  // COV_MAX_SEG (160) row segments over 8 warps

__device__ __forceinline__ double small_block_sum(double v, double* sm) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sm[w];
    return t;  // every thread holds the same total (fixed order)
}

__device__ __forceinline__ void small_block_argmin(double& v, int64_t& i, double& aux, double* sv, int64_t* si, double* sa) {
    // (value, index) minimum with np.argmin tie-break; aux travels with the winner
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, off);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, i, off);
        const double oa = __shfl_xor_sync(0xffffffffu, aux, off);
        if (gpx_better(ov, oi, v, i, true)) {
            v = ov;
            i = oi;
            aux = oa;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) {
        sv[warp] = v;
        si[warp] = i;
        sa[warp] = aux;
    }
    __syncthreads();
    v = sv[0];
    i = si[0];
    aux = sa[0];
#pragma unroll
    for (int w = 1; w < 8; ++w)
        if (gpx_better(sv[w], si[w], v, i, true)) {
            v = sv[w];
            i = si[w];
            aux = sa[w];
        }
}

template <int FAM, bool WT>
__global__ void __launch_bounds__(256, 2) ivar_small_greedy_kernel(const __grid_constant__ KParams kp, const gpx_ivar_state s,
                                                                 int n_begin, int n_end, double* __restrict__ blk_val,
                                                                 int64_t* __restrict__ blk_idx, double* __restrict__ blk_piv,
                                                                 double* __restrict__ blk_base) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double sm[8], sa[8], s_col[SMALL_NCAP], s_xp[GPX_MAX_DIM], s_part[8][32];
    __shared__ int64_t si[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t nb = gridDim.x, b = blockIdx.x;
    const int64_t M = s.M, C = s.C;
    const int64_t colblocks = (C + 511) / 512;
    const int64_t rows_per_seg = (M + s.nseg - 1) / s.nseg;
    const int64_t cgroups = (C + 31) / 32;
    // sum of var_M for the first step (every block, same order); later steps get it from the blocks' phase-B partials
    double part = 0.0;
    for (int64_t m = tid; m < M; m += 256) {
        if (WT) part = fma(s.wM[m], s.varM[m], part);
        else part += s.varM[m];
    }
    double base_sum = small_block_sum(part, sm);
    for (int n = n_begin; n < n_end; ++n) {
        // ---- phase A: scores of my candidate groups (32 candidates x 8 warps over the row segments), block arg-min ------
        const double base = WT ? base_sum : base_sum / (double)M;     // (1/nMC) sum varMC   experimentalDesign.py:109
        double bv = 0.0, bp = 1.0;
        int64_t bi = -1;
        for (int64_t grp = b; grp < cgroups; grp += nb) {
            const int64_t c = grp * 32 + lane;
            double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
            double den = 1.0;
            if (c < C) {
                // all of this warp's segment partials in one batch of loads (nseg <= 160 = 8 warps x 20)
                const double* wp = s.workspace + c;
                double v[SMALL_SEG_PER_WARP];
#pragma unroll
                for (int u = 0; u < SMALL_SEG_PER_WARP; ++u) {
                    const int g = warp + 8 * u;
                    v[u] = g < s.nseg ? wp[(int64_t)g * s.ldp] : 0.0;
                }
                if (warp == 0) den = s.varC[c] + s.noise;
#pragma unroll
                for (int u = 0; u < SMALL_SEG_PER_WARP; u += 4) {
                    r0 += v[u];
                    r1 += v[u + 1];
                    r2 += v[u + 2];
                    r3 += v[u + 3];
                }
                for (int g = warp + 8 * SMALL_SEG_PER_WARP; g < s.nseg; g += 8) r0 += wp[(int64_t)g * s.ldp];
            }
            __syncthreads();
            s_part[warp][lane] = (r0 + r1) + (r2 + r3);
            __syncthreads();
            if (warp == 0 && c < C) {
                double r = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) r += s_part[w][lane];
                const double red = (den <= s.zero_tol) ? 0.0 : (WT ? r / den : (r / den) / (double)M);
                const double sc = fabs(base - red);                     // np.abs(cost)        experimentalDesign.py:117
                s.scores[c] = sc;
                if (gpx_better(sc, c, bv, bi, true)) {
                    bv = sc;
                    bi = c;
                    bp = den;
                }
            }
        }
        if (warp == 0) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
                const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
                const double oa = __shfl_xor_sync(0xffffffffu, bp, off);
                if (gpx_better(ov, oi, bv, bi, true)) {
                    bv = ov;
                    bi = oi;
                    bp = oa;
                }
            }
            if (lane == 0) {
                blk_val[b] = bv;
                blk_idx[b] = bi;
                blk_piv[b] = bp;
            }
        }
        grid.sync();
        // ---- phase B: the winner (identical in every block), its record, the new rows ---------------------------------
        bv = 0.0;
        bp = 1.0;
        bi = -1;
        for (int64_t q = tid; q < nb; q += 256) {
            const double ov = __ldcg(blk_val + q);
            const int64_t oi = __ldcg(blk_idx + q);
            if (gpx_better(ov, oi, bv, bi, true)) {
                bv = ov;
                bi = oi;
                bp = __ldcg(blk_piv + q);
            }
        }
        small_block_argmin(bv, bi, bp, sm, si, sa);
        const int64_t p = bi;
        const double piv = bp;
        for (int i = tid; i < n; i += 256) s_col[i] = s.Wc[(int64_t)i * s.ldc + p];
        if (tid < GPX_MAX_DIM) s_xp[tid] = tid < kp.d ? s.Xc[tid * s.ldc + p] : 0.0;
        __syncthreads();
        if (b == 0) {
            for (int i = tid; i < n; i += 256)
                if (s.U) s.U[(int64_t)i * s.ldu + n] = s_col[i];
            if (tid == 0) {
                if (s.U) s.U[(int64_t)n * s.ldu + n] = sqrt(piv);
                s.picks[n] = p + s.index_offset;
                if (s.pick_scores) s.pick_scores[n] = bv;
                if (s.pick_pivots) s.pick_pivots[n] = piv;
                s.best[0] = bv;
                s.idx[0] = p;
            }
        }
        const double lnn = piv > 0.0 ? sqrt(piv) : INFINITY;            // non-positive pivot -> zero row (append_row_kernel)
        double vpart = 0.0;
        for (int64_t j = b * 256 + tid; j < C + M; j += nb * 256) {
            const bool cside = j < C;
            const int64_t col = cside ? j : j - C;
            const int64_t ld = cside ? s.ldc : s.ldm;
            double* W = cside ? s.Wc : s.Wm;
            const double* X = cside ? s.Xc : s.Xm;
            double* var = cside ? s.varC : s.varM;
            const double* wp = W + col;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            const double var_old = var[col];
            int i = 0;
            for (; i + 8 <= n; i += 8) {
                double w8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) w8[u] = wp[(int64_t)(i + u) * ld];
#pragma unroll
                for (int u = 0; u < 8; u += 4) {
                    a0 = fma(s_col[i + u], w8[u], a0);
                    a1 = fma(s_col[i + u + 1], w8[u + 1], a1);
                    a2 = fma(s_col[i + u + 2], w8[u + 2], a2);
                    a3 = fma(s_col[i + u + 3], w8[u + 3], a3);
                }
            }
            if (i < n) {
                double w8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) w8[u] = i + u < n ? wp[(int64_t)(i + u) * ld] : 0.0;
#pragma unroll
                for (int u = 0; u < 8; u += 4) {
                    a0 = fma(i + u < n ? s_col[i + u] : 0.0, w8[u], a0);
                    a1 = fma(i + u + 1 < n ? s_col[i + u + 1] : 0.0, w8[u + 1], a1);
                    a2 = fma(i + u + 2 < n ? s_col[i + u + 2] : 0.0, w8[u + 2], a2);
                    a3 = fma(i + u + 3 < n ? s_col[i + u + 3] : 0.0, w8[u + 3], a3);
                }
            }
            const double a = (a0 + a1) + (a2 + a3);
            double k = 0.0;
#pragma unroll
            for (int q = 0; q < GPX_MAX_DIM; ++q)
                if (q < kp.d) kacc_dim<FAM>(k, kp, q, s_xp[q], X[q * ld + col]);
            const double w = (kfinish<FAM>(k, kp) - a) / lnn;
            W[(int64_t)n * ld + col] = w;
            const double nv = var_old - w * w;
            var[col] = nv;
            if (!cside) {
                if (WT) vpart = fma(s.wM[col], nv, vpart);
                else vpart += nv;
            }
        }
        const double vsum = small_block_sum(vpart, sm);
        if (tid == 0) blk_base[b] = vsum;
        grid.sync();
        // ---- phase C: cov -= w_M[n] w_C[n]^T and the column sums of squares of the next step (layout of gpx_cov_update) --
        part = 0.0;
        for (int64_t q = tid; q < nb; q += 256) part += __ldcg(blk_base + q);   // consumed after the covariance pass
        const double* am = s.Wm + (int64_t)n * s.ldm;
        const double* bc = s.Wc + (int64_t)n * s.ldc;
        for (int64_t item = b; item < (int64_t)s.nseg * colblocks; item += nb) {
            const int64_t seg = item / colblocks, c = ((item % colblocks) * 256 + tid) * 2;
            if (c >= C) continue;
            const int64_t m0 = seg * rows_per_seg;
            const int64_t m1 = m0 + rows_per_seg < M ? m0 + rows_per_seg : M;
            const double2 bb = *reinterpret_cast<const double2*>(bc + c);
            double r0 = 0.0, r1 = 0.0;
            double* cp = s.cov + m0 * s.ldcov + c;
            int64_t m = m0;
            for (; m + 8 <= m1; m += 8) {
                double2 v[8];
                double a8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    v[u] = *reinterpret_cast<const double2*>(cp + (int64_t)u * s.ldcov);
                    a8[u] = am[m + u];
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const double a = a8[u];
                    v[u].x = fma(-a, bb.x, v[u].x);
                    v[u].y = fma(-a, bb.y, v[u].y);
                    *reinterpret_cast<double2*>(cp + (int64_t)u * s.ldcov) = v[u];
                    const double w = WT ? s.wM[m + u] : 1.0;
                    r0 = fma(WT ? w * v[u].x : v[u].x, v[u].x, r0);
                    r1 = fma(WT ? w * v[u].y : v[u].y, v[u].y, r1);
                }
                cp += 8 * s.ldcov;
            }
            for (; m < m1; ++m, cp += s.ldcov) {
                double2 v = *reinterpret_cast<const double2*>(cp);
                const double a = am[m];
                v.x = fma(-a, bb.x, v.x);
                v.y = fma(-a, bb.y, v.y);
                *reinterpret_cast<double2*>(cp) = v;
                const double w = WT ? s.wM[m] : 1.0;
                r0 = fma(WT ? w * v.x : v.x, v.x, r0);
                r1 = fma(WT ? w * v.y : v.y, v.y, r1);
            }
            double* dst = s.workspace + seg * s.ldp + c;
            dst[0] = r0;
            if (c + 1 < C) dst[1] = r1;
        }
        base_sum = small_block_sum(part, sm);
        grid.sync();
    }
}

}  // namespace

// Whole greedy IVAR loop in one cooperative launch, for a RESIDENT engine state on one GPU (s->cov != NULL, no
// communicator): steps n_begin .. n_end-1.  Meant for small problems (the covariance M x C should fit the L2 cache);
// correct for any size.  n_end <= 1024.
extern "C" int gpx_ivar_greedy_small(gpx_handle h, const gpx_ivar_state* s, int64_t n_begin, int64_t n_end, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(s != nullptr, GPX_EINVAL, "state is NULL");
    GPX_REQUIRE(n_begin >= 0 && n_end >= n_begin && n_end <= s->ncap && n_end <= SMALL_NCAP, GPX_ESIZE,
                "step range outside the state's capacity or beyond 1024 design points");
    GPX_REQUIRE(s->cov && s->Xm && s->Wm && s->varM && s->Xc && s->Wc && s->varC && s->workspace && s->scores && s->best &&
                    s->idx && s->picks && s->M >= 1 && s->C >= 1 && s->nseg >= 1 && s->ldp >= s->C && s->ldcov >= s->C,
                GPX_EINVAL, "the one-kernel loop needs a complete resident state");
    GPX_REQUIRE((s->ldcov % 2) == 0 && s->ldcov >= s->C + (s->C & 1) && (s->ldc % 2) == 0 && gpx_aligned16(s->cov) &&
                    gpx_aligned16(s->Wc),
                GPX_EALIGN, "cov and W_C must be 16-byte aligned with even leading dimensions");
    GPX_REQUIRE(h->nccl_comm == nullptr || h->comm_size <= 1 || s->rec_all == nullptr, GPX_EINVAL,
                "the one-kernel loop is single-GPU");
    if (n_end == n_begin) return GPX_OK;
    int per_sm = 0;
    cudaError_t e;
#define GPX_SMALL_LAUNCH(F, W)                                                                                           \
    do {                                                                                                                 \
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ivar_small_greedy_kernel<F, W>, 256, 0);              \
        if (e == cudaSuccess) {                                                                                          \
            if (per_sm > 2) per_sm = 2;                                                                                  \
            int blocks = per_sm * (h->sm_count > 0 ? h->sm_count : 148);                                                 \
            if (blocks > 512) blocks = 512;                                                                              \
            KParams kp = h->kp;                                                                                          \
            gpx_ivar_state st = *s;                                                                                      \
            int nb0 = (int)n_begin, ne0 = (int)n_end;                                                                    \
            double* bv = h->red_val;                                                                                     \
            int64_t* bi = h->red_idx;                                                                                    \
            double* bp = h->red_val + 512;                                                                               \
            double* bb = h->red_val + 1024;                                                                              \
            void* args[] = {&kp, &st, &nb0, &ne0, &bv, &bi, &bp, &bb};                                                   \
            e = blocks > 0 ? cudaLaunchCooperativeKernel((const void*)ivar_small_greedy_kernel<F, W>, dim3(blocks), dim3(256), \
                                                         args, 0, (cudaStream_t)stream)                                  \
                           : cudaErrorLaunchOutOfResources;                                                              \
        }                                                                                                                \
    } while (0)
    if (s->wM) GPX_DISPATCH_FAMILY(h->kp.family, GPX_SMALL_LAUNCH(FAM, true));
    else GPX_DISPATCH_FAMILY(h->kp.family, GPX_SMALL_LAUNCH(FAM, false));
#undef GPX_SMALL_LAUNCH
    if (e != cudaSuccess) {
        gpx_set_error("gpx_ivar_greedy_small: %s", cudaGetErrorString(e));
        return (int)e;
    }
    return gpx_check_launch("gpx_ivar_greedy_small");
}

// sizeof of the state structs as this library was compiled: lets a binding verify its own layout
extern "C" int64_t gpx_state_bytes(int which) {
    return which == 0 ? (int64_t)sizeof(gpx_ivar_state) : (which == 1 ? (int64_t)sizeof(gpx_var_state) : -1);
}

extern "C" int gpx_ivar_greedy_run(gpx_handle h, const gpx_ivar_state* s, int64_t n_begin, int64_t n_end, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(s != nullptr, GPX_EINVAL, "state is NULL");
    GPX_REQUIRE(n_begin >= 0 && n_end >= n_begin && n_end <= s->ncap, GPX_EINVAL, "step range outside the state's capacity");
    GPX_REQUIRE(s->Xm && s->Wm && s->varM && s->Xc && s->Wc && s->varC && s->workspace && s->scores && s->best && s->idx &&
                    s->rec && s->picks,
                GPX_EINVAL, "NULL pointer in the state");
    GPX_REQUIRE(s->M >= 1 && s->C >= 1, GPX_EINVAL, "empty point set");
    GPX_REQUIRE(s->cov != nullptr || (s->Ma_rows && s->Cb_rows), GPX_EINVAL, "contraction mode needs the prologue rows");
    const bool sharded = h->nccl_comm != nullptr && h->comm_size > 1 && s->rec_all != nullptr;
    GPX_REQUIRE(!sharded || s->rec_win != nullptr, GPX_EINVAL, "sharded runs need rec_all and rec_win");
    cudaStream_t st = (cudaStream_t)stream;
    const AppendSide sc = {s->Xc, s->C, s->ldc, s->Wc, s->ldc, s->varC};
    const AppendSide sm = {s->Xm, s->M, s->ldm, s->Wm, s->ldm, s->varM};
    GPX_REQUIRE(side_ok(sc) && side_ok(sm), GPX_EALIGN, "factors and coordinates must be 16-byte aligned with even leading dimensions");
    const PivotSinks sinks = {s->U, s->ldu, s->picks, s->pick_scores, s->pick_pivots};
    const PivotSinks none = {nullptr, 0, nullptr, nullptr, nullptr};
    int rc;
    for (int64_t n = n_begin; n < n_end; ++n) {
        if (s->cov) {
            rc = gpx_score_ivar_partials_w(h, s->workspace, s->nseg, s->ldp, s->varM, s->M, s->varC, s->C, s->noise,
                                           s->zero_tol, s->wM, nullptr, s->scores, s->best, s->idx, stream);
        } else {
            rc = gpx_score_ivar_w(h, s->prologue, s->Wm, s->ldm, s->varM, s->Ma_rows, s->M, s->Wc, s->ldc, s->varC, s->Cb_rows,
                                  s->C, n, s->noise, s->zero_tol, s->wM, nullptr, s->workspace, s->scores, s->best, s->idx,
                                  stream);
        }
        if (rc) return rc;
        rc = launch_gather_store(h, s->Wc, s->ldc, n, s->varC, s->Xc, s->ldc, s->best, s->idx, s->index_offset, s->noise, s->rec,
                                 sharded ? 0 : 1, sharded ? none : sinks, st);
        if (rc) return rc;
        const double* win = s->rec;
        if (sharded) {
            rc = exchange(h, s->rec, s->rec_all, s->rec_win, n, 1, sinks, st);
            if (rc) return rc;
            win = s->rec_win;
        }
        rc = launch_append2(h, win, sc, sm, n, st);
        if (rc) return rc;
        if (s->cov) {
            rc = gpx_cov_update_w(h, s->cov, s->ldcov, s->M, s->C, s->Wm + n * s->ldm, s->Wc + n * s->ldc, s->wM, s->workspace,
                                  s->ldp, stream);
            if (rc) return rc;
        }
    }
    return GPX_OK;
}

extern "C" int gpx_var_greedy_run(gpx_handle h, const gpx_var_state* s, int64_t n_begin, int64_t n_end, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(s != nullptr, GPX_EINVAL, "state is NULL");
    GPX_REQUIRE(n_begin >= 0 && n_end >= n_begin && n_end <= s->ncap, GPX_EINVAL, "step range outside the state's capacity");
    GPX_REQUIRE(s->X && s->W && s->var && s->best && s->idx && s->rec && s->picks && s->C >= 1, GPX_EINVAL,
                "NULL pointer in the state");
    const bool sharded = h->nccl_comm != nullptr && h->comm_size > 1 && s->rec_all != nullptr;
    GPX_REQUIRE(!sharded || s->rec_win != nullptr, GPX_EINVAL, "sharded runs need rec_all and rec_win");
    cudaStream_t st = (cudaStream_t)stream;
    const PivotSinks sinks = {nullptr, 0, s->picks, s->pick_scores, s->pick_pivots};
    const PivotSinks none = {nullptr, 0, nullptr, nullptr, nullptr};
    int rc;
    for (int64_t n = n_begin; n < n_end; ++n) {
        rc = gpx_argreduce_impl(h, s->var, s->weights, nullptr, s->C, 0, s->best, s->idx, st);
        if (rc) return rc;
        rc = launch_gather_store(h, s->W, s->ld, n, s->var, s->X, s->ld, s->best, s->idx, s->index_offset, s->noise, s->rec,
                                 sharded ? 0 : 1, sharded ? none : sinks, st);
        if (rc) return rc;
        const double* win = s->rec;
        if (sharded) {
            rc = exchange(h, s->rec, s->rec_all, s->rec_win, n, 0, sinks, st);
            if (rc) return rc;
            win = s->rec_win;
        }
        rc = gpx_append_row(h, GPX_ROW_KERNEL, win, nullptr, s->X, s->C, s->ld, s->W, s->ld, n, s->var, stream);
        if (rc) return rc;
    }
    return GPX_OK;
}
