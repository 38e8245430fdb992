// FP64 tensor-core (DMMA.8x8x4) contractions of the greedy design path.
//
//   T[i,j] = sum_k A[k*lda + i] * B[k*ldb + j]           both operands K-major (row k contiguous)
//
// with an optional *prologue* that evaluates the covariance k(x_i, y_j) inside the same kernel, and three epilogues:
//
//   EPI_IVAR   r[j] += sum_i (k(i,j) - T[i,j])^2          K5: IVAR scoring, experimentalDesign.py:105-117 restated
//   EPI_STORE  out[i,j] = k(i,j) - T[i,j]                  K1+K3: block row of the left-looking TRSM
//   EPI_SUB    C[i,j]  -= T[i,j]                           K2: Cholesky trailing update / materialised TRSM / MI set-up
//
// Prologue forms (GPX_PRO_*):
//   EXPANDED   k = f(e), e = sum_q u_q(i) v_q(j) over the d+2 rows of two *prepared sides* (gpx_prep_side): the d
//              scaled coordinates plus the rows (alpha_i, 1) x (1, beta_j), so that the whole exponent -- including the
//              |x|^2 and |y|^2 terms -- comes out of ONE extra DMMA chunk on the tensor pipe.  Cancellation error
//              ~ eps * max|alpha|: the host only selects it when that is below 1e-11 (after centring), else
//   DIFF       k = f(sum_q a_q (x_q - y_q)^2) from the raw coordinates staged in shared memory (difference form, the
//              arithmetic of kernels.py:121-122 itself): no cancellation, d FP64 operations more per pair.
//
// sm_100a has no f64 kind in tcgen05, so the FP64 tensor path is warp-level mma.sync.m8n8k4 (SASS DMMA.8x8x4)
// fed from shared memory.  Two kernels share the fragment layout:
//
//   ivar_ws_kernel     THE hot kernel (EPI_IVAR on fully padded operands): 128x128 CTA tile, 8 warps of 32x64,
//                      operand chunks by TMA bulk copies completing on mbarriers, no CTA barrier in the main loop,
//                      table-driven exp prologue, butterfly column reduction.
//   dmma_core_kernel   the generic predicated kernel (cp.async ring + __syncthreads, zero-filled edges, 64x128 tile,
//                      2 CTAs per SM) used for EPI_STORE / EPI_SUB and for unpadded IVAR operands.
//
// Rows are padded to 132 doubles and the fragment <-> matrix index map is permuted so that every thread reads
// 2 adjacent doubles per conflict-free LDS.128:
//   i_local = wm*32 + (t>>1)*16 + (lane>>2)*2 + (t&1)            t = 0..3  (A fragments)
//   j_local = wn*64 + (u>>1)*16 + (lane>>2)*2 + (u&1)            u = 0..7  (B fragments, load side)
//   accumulator (t,u,e) sits at column  wn*64 + (u>>1)*16 + ((lane&3)*2+e)*2 + (u&1)
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "gpx_common.cuh"

namespace {

// expanded-form covariance with the table exp.  The table carries the signal variance AND the sign the accumulators
// need (tab[j] = -signal * 2^(j/256)), so these return -k(x,y) without a negation per element.
template <int FAM>
__device__ __forceinline__ double neg_kexpand_tab(double e, const KParams& kp, const double* __restrict__ ntab) {
    if (FAM == GPX_MATERN32) {
        const double t = kp.c0 * sqrt(fmax(e, 0.0));
        return (1.0 + t) * gpx_exp_tab(-t, ntab);
    }
    return gpx_exp_tab<FAM == GPX_MEHLER>(e, ntab);
}

constexpr int BN = 128;
constexpr int BK = 16;
constexpr int STAGES = 4;

enum { EPI_IVAR = 0, EPI_STORE = 1, EPI_SUB = 2 };
enum { PRO_NONE = 0, PRO_EXPANDED = GPX_PRO_EXPANDED, PRO_DIFF = GPX_PRO_DIFF };

// generic kernel geometry: 2 warps along i: 128 threads, 64x128 tile, 2 CTAs/SM (two independent CTAs de-phase the
// barriers and the exp prologue against each other's DMMA stream)
struct Cfg {
    static constexpr int WM = 2;
    static constexpr int NT = WM * 64;
    static constexpr int BM = WM * 32;
    static constexpr int LDA = BM + 4;  // row strides = 4 (mod 16) doubles: conflict-free LDS.128 fragment loads
    static constexpr int LDB = BN + 4;
    static constexpr int STAGE = BK * (LDA + LDB);
    static constexpr int PIECES_A = BK * BM / 2;  // 16-byte pieces per chunk
    static constexpr int PIECES = BK * (BM + BN) / 2;
    static constexpr int PER_THREAD = PIECES / NT;
    static constexpr int A_ITERS = PIECES_A / NT;
    static constexpr int SMEM_DOUBLES = STAGES * STAGE + WM * BN + 256;
    static constexpr size_t SMEM_BYTES = (size_t)SMEM_DOUBLES * sizeof(double);
    static_assert(PIECES % NT == 0 && PIECES_A % NT == 0, "loader mapping");
};

struct CoreArgs {
    const double* A;   // K x I (main operand)
    const double* B;   // K x J
    const double* Ap;  // prologue rows, same column space as A: prepared side (EXPANDED) or raw coordinates (DIFF)
    const double* Bp;  // prologue rows of the B side
    double* out;       // IVAR: partial sums [split][ldo] ; STORE / SUB: row-major I x J
    int64_t lda, ldb, ldo;
    int64_t I, J;
    int K;
    int prows;         // prologue rows to stage: EXPANDED roundup(d+2, 4), DIFF d
    int tiles_per_cta; // IVAR: i-tiles each CTA walks
    int upper_only;    // SUB: update only j >= i (strictly-lower entries untouched) ; ivar_ws_kernel: candidate tiles per wave group
    int ldo_splits;    // ivar_ws_kernel: number of M-splits
    // sub_ws_kernel: operand B is this rank's column slice of a LOWER-triangular matrix distributed block-cyclically
    // (local column j = block j / tri_blk of this rank = global block (j / tri_blk) * tri_world + tri_rank): rows above the
    // first global column of a tile are structurally zero and are skipped.  tri_blk = 0: dense operand.
    int tri_blk, tri_world, tri_rank;
};

__device__ __forceinline__ void cp_async16(double* dst, const double* src, bool ok) {
    const unsigned int d = (unsigned int)__cvta_generic_to_shared(dst);
    const int sz = ok ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <int LDA_, int LDB_>
__device__ __forceinline__ void load_frags(double (&af)[4], double (&bf)[8], const double* pa, const double* pb, int ks) {
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        const double2 v = *reinterpret_cast<const double2*>(pa + ks * 4 * LDA_ + t2 * 16);
        af[t2 * 2] = v.x;
        af[t2 * 2 + 1] = v.y;
    }
#pragma unroll
    for (int u2 = 0; u2 < 4; ++u2) {
        const double2 v = *reinterpret_cast<const double2*>(pb + ks * 4 * LDB_ + u2 * 16);
        bf[u2 * 2] = v.x;
        bf[u2 * 2 + 1] = v.y;
    }
}

__device__ __forceinline__ void mma_tile(double (&acc)[4][8][2], const double (&af)[4], const double (&bf)[8]) {
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int u = 0; u < 8; ++u) dmma(acc[t][u][0], acc[t][u][1], af[t], bf[u]);
}

// Difference-form covariance of the warp's 32x64 accumulator block from coordinates staged in shared memory:
// sa / sb point at row 0 of the staged A / B coordinates, offset to this thread's first i / j (see the index map).
// `tab` is the NEGATED exp table (-signal * 2^(j/256)); on exit acc = -k(i,j).
template <int FAM, int LDA_, int LDB_>
__device__ __forceinline__ void diff_prologue(double (&acc)[4][8][2], const KParams& kp, const double* __restrict__ sa,
                                              const double* __restrict__ sb, const double* __restrict__ tab) {
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int u = 0; u < 8; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;
#pragma unroll 1
    for (int q = 0; q < kp.d; ++q) {
        double x[4], y[8][2];
#pragma unroll
        for (int t2 = 0; t2 < 2; ++t2) {
            const double2 v = *reinterpret_cast<const double2*>(sa + q * LDA_ + t2 * 16);
            x[t2 * 2] = v.x;
            x[t2 * 2 + 1] = v.y;
        }
#pragma unroll
        for (int u2 = 0; u2 < 4; ++u2)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double2 v = *reinterpret_cast<const double2*>(sb + q * LDB_ + u2 * 16 + e * 2);
                y[u2 * 2][e] = v.x;
                y[u2 * 2 + 1][e] = v.y;
            }
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int e = 0; e < 2; ++e) kacc_dim<FAM>(acc[t][u][e], kp, q, x[t], y[u][e]);
    }
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int e = 0; e < 2; ++e) acc[t][u][e] = kfinish_tab<FAM>(acc[t][u][e], kp, tab);  // tab is negated: -k
}

// squares of the warp's accumulator block summed over its 32 rows: butterfly reduce-scatter over the 8 lanes that
// share q4; lane g4 ends up owning columns u = g4, e = 0, 1
__device__ __forceinline__ void column_squares(const double (&acc)[4][8][2], bool full, int64_t i_first, int64_t I, int lane,
                                               double (&rs)[2]) {
    const int g4 = lane >> 2;
    double p[8][2];
#pragma unroll
    for (int u = 0; u < 8; ++u) p[u][0] = p[u][1] = 0.0;
    if (full) {  // every row of the tile is a real integration point: no masking
#pragma unroll
        for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int e = 0; e < 2; ++e) p[u][e] = fma(acc[t][u][e], acc[t][u][e], p[u][e]);
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int64_t i = i_first + (t >> 1) * 16 + g4 * 2 + (t & 1);
            const bool ok = i < I;
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double v = ok ? acc[t][u][e] : 0.0;
                    p[u][e] = fma(v, v, p[u][e]);
                }
        }
    }
    const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
    double h[4][2], q[2][2];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double keep = b4 ? p[u + 4][e] : p[u][e];
            const double send = b4 ? p[u][e] : p[u + 4][e];
            h[u][e] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double keep = b3 ? h[u + 2][e] : h[u][e];
            const double send = b3 ? h[u][e] : h[u + 2][e];
            q[u][e] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const double keep = b2 ? q[1][e] : q[0][e];
        const double send = b2 ? q[0][e] : q[1][e];
        rs[e] += keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
}

template <int FAM, int EPI, int PRO>
__global__ void __launch_bounds__(Cfg::NT, 2)
    dmma_core_kernel(const __grid_constant__ CoreArgs a, const __grid_constant__ KParams kp) {
    using C = Cfg;
    constexpr int WM = C::WM, BM = C::BM, NT = C::NT, LDA = C::LDA, LDB = C::LDB;
    extern __shared__ __align__(16) double smem[];
    double* s_red = smem + STAGES * C::STAGE;
    double* s_tab = s_red + WM * BN;

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int wm = warp % WM, wn = warp / WM;
    const int g4 = lane >> 2, q4 = lane & 3;

    const int64_t j0 = (int64_t)blockIdx.x * BN;
    const int64_t itiles = (a.I + BM - 1) / BM;
    int64_t it_begin, it_end;
    if (EPI == EPI_IVAR) {
        it_begin = (int64_t)blockIdx.y * a.tiles_per_cta;
        it_end = it_begin + a.tiles_per_cta;
        if (it_end > itiles) it_end = itiles;
    } else {
        it_begin = blockIdx.y;
        it_end = it_begin + 1;
        // symmetric update: nothing to do for tiles strictly below the diagonal
        if (a.upper_only && it_begin * BM >= j0 + BN) return;
    }
    const int ntiles = it_end > it_begin ? (int)(it_end - it_begin) : 0;
    const int kch = (a.K + BK - 1) / BK;
    const int T = (PRO != PRO_NONE ? 1 : 0) + kch;  // chunks per tile
    const int G = ntiles * T;

    if (PRO != PRO_NONE) {
        for (int i = tid; i < 256; i += NT) s_tab[i] = -kp.signal * gpx_exp2_tab[i];
    }

    // ---- chunk loader (cp.async ring, 3 chunks in flight) ------------------------------------------
    int is_g = 0, is_tl = 0, is_ch = 0;
    auto issue = [&]() {
        if (is_g < G) {
            const int64_t i0 = (it_begin + is_tl) * BM;
            const double *srcA, *srcB;
            int krows;
            if (PRO != PRO_NONE && is_ch == 0) {
                srcA = a.Ap;
                srcB = a.Bp;
                krows = a.prows;
            } else {
                const int kc = is_ch - (PRO != PRO_NONE ? 1 : 0);
                srcA = a.A + (int64_t)kc * BK * a.lda;
                srcB = a.B + (int64_t)kc * BK * a.ldb;
                krows = a.K - kc * BK;
            }
            double* sA = smem + (is_g % STAGES) * C::STAGE;
            double* sB = sA + BK * LDA;
#pragma unroll
            for (int it = 0; it < C::PER_THREAD; ++it) {
                if (it < C::A_ITERS) {
                    const int p = tid + it * NT;
                    const int row = p / (BM / 2), c2 = (p % (BM / 2)) * 2;
                    const bool ok = (row < krows) && (i0 + c2 < a.I);
                    cp_async16(sA + row * LDA + c2, ok ? srcA + (int64_t)row * a.lda + i0 + c2 : srcA, ok);
                } else {
                    const int p = tid + it * NT - C::PIECES_A;
                    const int row = p / (BN / 2), c2 = (p % (BN / 2)) * 2;
                    const bool ok = (row < krows) && (j0 + c2 < a.J);
                    cp_async16(sB + row * LDB + c2, ok ? srcB + (int64_t)row * a.ldb + j0 + c2 : srcB, ok);
                }
            }
            if (++is_ch == T) {
                is_ch = 0;
                ++is_tl;
            }
        }
        ++is_g;
        cp_async_commit();
    };
    // chunk g+1 landed and visible to all warps; the stage of chunk g-1 is free -> refill it with chunk g+3
    auto midsync = [&]() {
        cp_async_wait<1>();
        __syncthreads();
        issue();
    };

    double acc[4][8][2];
    double rs[2] = {0.0, 0.0};
    double af0[4], bf0[8], af1[4], bf1[8];

    issue();
    issue();
    issue();
    cp_async_wait<2>();
    __syncthreads();

    const int fa = q4 * LDA + wm * 32 + g4 * 2;  // fragment offsets inside a stage
    const int fb = q4 * LDB + wn * 64 + g4 * 2;
    int tl = 0, ch = 0;
    bool pre = false;
    for (int g = 0; g < G; ++g) {
        const int64_t i0 = (it_begin + tl) * BM;
        if (ch == 0) {
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
                for (int u = 0; u < 8; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;
        }
        const double* pa = smem + (g % STAGES) * C::STAGE + fa;
        const double* pb = smem + (g % STAGES) * C::STAGE + BK * LDA + fb;
        int ksteps;
        bool next_full;
        {
            const int kc = ch - (PRO != PRO_NONE ? 1 : 0);
            if (PRO != PRO_NONE && ch == 0) {
                ksteps = PRO == PRO_EXPANDED ? (a.prows >> 2) : 0;
            } else {
                const int rem = a.K - kc * BK;
                ksteps = rem >= BK ? 4 : ((rem + 3) >> 2);
            }
            next_full = (a.K - (kc + 1) * BK) >= BK;
        }
        if (PRO == PRO_DIFF && ch == 0) {
            // covariance in difference form from the staged raw coordinates
            const double* sa = smem + (g % STAGES) * C::STAGE + wm * 32 + g4 * 2;
            const double* sb = smem + (g % STAGES) * C::STAGE + BK * LDA + wn * 64 + q4 * 4;
            diff_prologue<FAM, LDA, LDB>(acc, kp, sa, sb, s_tab);
            midsync();
            pre = false;
        } else if (ksteps == 4) {
            // software-pipelined: fragments of k-step s+1 are fetched while the DMMAs of k-step s issue
            if (!pre) load_frags<LDA, LDB>(af0, bf0, pa, pb, 0);
            load_frags<LDA, LDB>(af1, bf1, pa, pb, 1);
            mma_tile(acc, af0, bf0);
            load_frags<LDA, LDB>(af0, bf0, pa, pb, 2);
            mma_tile(acc, af1, bf1);
            load_frags<LDA, LDB>(af1, bf1, pa, pb, 3);
            mma_tile(acc, af0, bf0);
            midsync();
            const bool np = (ch + 1 < T) && !(PRO != PRO_NONE && ch == 0) && next_full;
            if (np) {
                const double* na = smem + ((g + 1) % STAGES) * C::STAGE + fa;
                const double* nb = smem + ((g + 1) % STAGES) * C::STAGE + BK * LDA + fb;
                load_frags<LDA, LDB>(af0, bf0, na, nb, 0);
            }
            mma_tile(acc, af1, bf1);
            pre = np;
        } else {
#pragma unroll 1
            for (int ks = 0; ks < ksteps; ++ks) {
                if (ks == ksteps - 1) midsync();
                load_frags<LDA, LDB>(af0, bf0, pa, pb, ks);
                mma_tile(acc, af0, bf0);
            }
            if (ksteps == 0) midsync();
            pre = false;
        }

        if (PRO == PRO_EXPANDED && ch == 0) {
            // covariance from the expanded form (alpha, beta ride in the contraction); accumulators become -k so
            // that the main loop yields T - k
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
                for (int u = 0; u < 8; ++u)
#pragma unroll
                    for (int e = 0; e < 2; ++e) acc[t][u][e] = neg_kexpand_tab<FAM>(acc[t][u][e], kp, s_tab);
        }

        if (ch == T - 1) {
            // ---- tile epilogue ---------------------------------------------------------------------
            if (EPI == EPI_IVAR) {
                column_squares(acc, i0 + BM <= a.I, i0 + wm * 32, a.I, lane, rs);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int64_t i = i0 + wm * 32 + (t >> 1) * 16 + g4 * 2 + (t & 1);
                    if (i >= a.I) continue;
#pragma unroll
                    for (int u2 = 0; u2 < 4; ++u2)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int64_t j = j0 + wn * 64 + u2 * 16 + (q4 * 2 + e) * 2;
                            if (j >= a.J) continue;
                            double* dst = a.out + i * a.ldo + j;
                            const double v0 = acc[t][u2 * 2][e], v1 = acc[t][u2 * 2 + 1][e];
                            if (EPI == EPI_STORE) {
                                if (j + 1 < a.J) {
                                    *reinterpret_cast<double2*>(dst) = make_double2(-v0, -v1);
                                } else {
                                    dst[0] = -v0;
                                }
                            } else if (a.upper_only && j < i) {
                                // symmetric update of a diagonal-straddling tile: the strictly-lower part is left untouched
                                if (j + 1 == i && j + 1 < a.J) dst[1] -= v1;
                            } else {
                                if (j + 1 < a.J) {
                                    double2 c = *reinterpret_cast<double2*>(dst);
                                    c.x -= v0;
                                    c.y -= v1;
                                    *reinterpret_cast<double2*>(dst) = c;
                                } else {
                                    dst[0] -= v0;
                                }
                            }
                        }
                }
            }
            ch = 0;
            ++tl;
        } else {
            ++ch;
        }
    }
    cp_async_wait<0>();

    if (EPI == EPI_IVAR) {
        // lane (g4,q4) owns columns u = g4, e = 0,1 of its warp; add the WM i-warps in a fixed order
        __syncthreads();
#pragma unroll
        for (int e = 0; e < 2; ++e) s_red[wm * BN + wn * 64 + (g4 >> 1) * 16 + (q4 * 2 + e) * 2 + (g4 & 1)] = rs[e];
        __syncthreads();
        for (int c = tid; c < BN; c += NT) {
            if (j0 + c < a.J) {
                double r = s_red[c];
#pragma unroll
                for (int w = 1; w < WM; ++w) r += s_red[w * BN + c];
                a.out[(int64_t)blockIdx.y * a.ldo + j0 + c] = r;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// TMA + mbarrier IVAR contraction (the hot kernel): operand chunks arrive by TMA bulk copies
// (cp.async.bulk -> UBLKCP) that complete on mbarriers; the eight warps do LDS.128 + DMMA and take turns at issuing
// the bulk copies of a chunk -- a ninth, dedicated producer warp would put three warps on one sub-partition and cap
// everybody at 168 registers.  No CTA-wide barrier in the main loop.
//
// Ring geometries (template RING) and operand movement (template TMAP), selected per handle (gpx_set_ivar_ring):
//   ring 0  32-row chunks, 3 stages, 1 chunk ahead, one cp.async.bulk (UBLKCP) per operand ROW: 65 copies per chunk
//           issued from one lane of the producing warp (round-1 kernel).
//   ring 1  same ring, but each operand chunk is ONE 2-D tensor-map TMA load (cp.async.bulk.tensor.2d, SASS UTMALDG):
//           the box is 132 columns x 32 rows, so the hardware itself writes the padded, conflict-free 132-double row
//           layout the fragment loads expect, and zero-fills the K tail (rows >= n) and the column overhang.
//   ring 2  24-row chunks, 4 stages, 2 chunks ahead, tensor-map loads: more slack between a chunk's request and its
//           first use.
// Measured and dropped in round 2: holding the second warp group (columns 64-127) one or two 16-row chunks behind the
// first so that one group's exp prologue overlaps the other's DMMA stream -- 174-178 ms against 162.7 ms at n = 255:
// DMMA and DFMA share the FP64 pipe, so there is nothing to overlap, and the extra barrier costs.
// Requires fully padded operands: lda, ldb multiples of 128 covering whole tiles (the engines guarantee it).
// ---------------------------------------------------------------------------------------------
constexpr int WS_BM = 128;
constexpr int WS_LD = 132;

template <int BK_, int STAGES_, int AHEAD_>
struct Ring {
    static constexpr int RBK = BK_;                    // K rows per chunk
    static constexpr int KSTEPS = BK_ / 4;
    static constexpr int STAGE = BK_ * 2 * WS_LD;      // doubles (a multiple of 16: every stage starts 128-byte aligned)
    static constexpr int NSTAGES = STAGES_;            // ring depth
    static constexpr int AHEAD = AHEAD_;               // chunks in flight ahead of the consumers
    static constexpr int SMEM_DOUBLES = STAGES_ * STAGE + 4 * BN + 2 * STAGES_ + 256;
    static constexpr size_t SMEM_BYTES = (size_t)SMEM_DOUBLES * sizeof(double);
    static_assert(AHEAD_ <= STAGES_ - 2, "the refilled stage must have been released a whole chunk ago");
    static_assert((BK_ * WS_LD) % 16 == 0, "operand halves of a stage must be 128-byte aligned for TMA");
};
// Measured on B200, round 1 (n = 2047 / n = 255, C = M = 100k): 16 rows x 6 stages, 3 ahead: 34.18 TFLOP/s / 165.5 ms;
// 32 rows x 3 stages, 1 ahead: 34.70 / 165.3 ms; 32 x 3, 2 ahead: 23.7 / 240 ms (the refilled stage must have been
// released at least one whole chunk ago, or the producing warp blocks on the slowest consumer).
using RingSync = Ring<32, 3, 1>;
using RingDeep = Ring<24, 4, 2>;

// tensor maps of the four operand streams of one IVAR launch (boxes: 132 columns x chunk rows)
struct alignas(64) TmaMaps {
    CUtensorMap a_main, b_main, a_pro, b_pro;
};

// sub_ws_kernel keeps the round-1 ring
constexpr int WS_BK = RingSync::RBK;
constexpr int WS_KSTEPS = RingSync::KSTEPS;
constexpr int WS_STAGE = RingSync::STAGE;
constexpr int WS_STAGES = RingSync::NSTAGES;
constexpr int WS_AHEAD = RingSync::AHEAD;

__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, unsigned int bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned int parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(double* dst, const double* src, unsigned int bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tma_load_2d(double* dst, const CUtensorMap* tm, int col, int row, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(col), "r"(row), "r"(smem_u32(bar))
        : "memory");
}

__device__ __forceinline__ void load_frags_ws(double (&af)[4], double (&bf)[8], const double* pa, const double* pb, int ks) {
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        const double2 v = *reinterpret_cast<const double2*>(pa + ks * 4 * WS_LD + t2 * 16);
        af[t2 * 2] = v.x;
        af[t2 * 2 + 1] = v.y;
    }
#pragma unroll
    for (int u2 = 0; u2 < 4; ++u2) {
        const double2 v = *reinterpret_cast<const double2*>(pb + ks * 4 * WS_LD + u2 * 16);
        bf[u2 * 2] = v.x;
        bf[u2 * 2 + 1] = v.y;
    }
}

template <int FAM, int PRO, class RING, bool TMAP>
__global__ void __launch_bounds__(256, 1) ivar_ws_kernel(const __grid_constant__ CoreArgs a, const __grid_constant__ KParams kp,
                                                         const __grid_constant__ TmaMaps maps) {
    constexpr int BM = WS_BM, LD = WS_LD, NW = 8;
    constexpr int RBK = RING::RBK, NST = RING::NSTAGES, AHEAD = RING::AHEAD;
    extern __shared__ __align__(128) double smem[];
    double* s_red = smem + NST * RING::STAGE;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_red + 4 * BN);
    uint64_t* empty = full + NST;
    double* s_tab = reinterpret_cast<double*>(empty + NST);          // -signal * 2^(j/256)

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    // Rasterisation for L2 reuse: the 1-D grid is walked as  j-group (one wave of candidate tiles) -> M-split -> tile,
    // so the waves that share a group's W_C tiles (re-read once per split) run back to back while every wave streams one
    // W_M slice; DRAM traffic ~ (#groups) x (|W_M| + |W_C group|) instead of (#waves) x (|W_M|/splits + |W_C group|).
    const int64_t jtiles = (a.J + BN - 1) / BN;
    const int64_t gw = a.upper_only;  // group width in tiles (reused field: CTAs per wave), >= 1
    const int64_t per_group = gw * a.ldo_splits;
    const int64_t jg = blockIdx.x / per_group;
    const int64_t rem = blockIdx.x - jg * per_group;
    const int64_t gsz = (jtiles - jg * gw) < gw ? (jtiles - jg * gw) : gw;  // tiles in this (possibly last, short) group
    const int64_t split = rem / gsz;
    const int64_t jt = jg * gw + rem % gsz;
    if (split >= a.ldo_splits) return;  // padding CTAs of a short last group
    const int64_t j0 = jt * BN;
    const int64_t itiles = (a.I + BM - 1) / BM;
    const int64_t it_begin = split * a.tiles_per_cta;
    int64_t it_end = it_begin + a.tiles_per_cta;
    if (it_end > itiles) it_end = itiles;
    const int ntiles = it_end > it_begin ? (int)(it_end - it_begin) : 0;
    const int kch = (a.K + RBK - 1) / RBK;
    const int T = 1 + kch;
    const int G = ntiles * T;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NST; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (tid < 256) s_tab[tid] = -kp.signal * gpx_exp2_tab[tid];
    __syncthreads();

    double rs[2] = {0.0, 0.0};
    const int wm = warp & 3, wn = warp >> 2;
    const int g4 = lane >> 2, q4 = lane & 3;

    // ---- producer step, executed by one warp per chunk; all addresses are warp-uniform so that the bulk
    //      copies issue back to back from one lane (UBLKCP takes uniform registers) -----------------------
    auto produce = [&](int c) {
        if (c >= G) return;
        const int s = c % NST;
        const unsigned int ph = (unsigned int)(c / NST) & 1u;
        mbar_wait(empty + s, ph ^ 1u);
        const int ptl = c / T, pch = c - ptl * T;
        const int64_t i0 = (it_begin + ptl) * BM;
        const double *srcA, *srcB;
        int krows, ksteps;
        if (pch == 0) {
            srcA = a.Ap + i0;
            srcB = a.Bp + j0;
            krows = a.prows;  // EXPANDED: a multiple of 4 (zero rows are part of the prepared side); DIFF: d, no DMMA
            ksteps = PRO == PRO_EXPANDED ? (a.prows >> 2) : 0;
        } else {
            const int kc = pch - 1;
            srcA = a.A + (int64_t)kc * RBK * a.lda + i0;
            srcB = a.B + (int64_t)kc * RBK * a.ldb + j0;
            const int rem = a.K - kc * RBK;
            krows = rem < RBK ? rem : RBK;
            ksteps = rem >= RBK ? RING::KSTEPS : ((rem + 3) >> 2);
        }
        double* stA = smem + s * RING::STAGE;
        double* stB = stA + RBK * LD;
        if (TMAP) {
            // one 2-D tensor-map load per operand: the 132-column box lands as the padded rows the fragment loads expect;
            // rows beyond the operand (K tail) and columns beyond its leading dimension are zero-filled by the TMA unit
            if (lane == 0) {
                const bool pro = pch == 0;
                const int brows = pro ? a.prows : RBK;
                mbar_arrive_expect_tx(full + s, (unsigned int)brows * 2u * LD * 8u);
                tma_load_2d(stA, pro ? &maps.a_pro : &maps.a_main, (int)i0, pro ? 0 : (pch - 1) * RBK, full + s);
                tma_load_2d(stB, pro ? &maps.b_pro : &maps.b_main, (int)j0, pro ? 0 : (pch - 1) * RBK, full + s);
            }
            __syncwarp();
            return;
        }
        if (krows < ksteps * 4) {
            // K tail: rows the DMMAs will read but the operand does not have -> explicit zeros (lane -> column pair)
            for (int r = krows; r < ksteps * 4; ++r) {
                for (int cc = lane * 2; cc < BM; cc += 64) {
                    *reinterpret_cast<double2*>(stA + r * LD + cc) = make_double2(0.0, 0.0);
                    *reinterpret_cast<double2*>(stB + r * LD + cc) = make_double2(0.0, 0.0);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic writes before later TMA writes here
            __syncwarp();
        }
        if (lane == 0) {
            mbar_arrive_expect_tx(full + s, (unsigned int)krows * (BM + BN) * 8u);
#pragma unroll 4
            for (int r = 0; r < krows; ++r) {
                bulk_g2s(stA + r * LD, srcA + (int64_t)r * a.lda, BM * 8u, full + s);
                bulk_g2s(stB + r * LD, srcB + (int64_t)r * a.ldb, BN * 8u, full + s);
            }
        }
        __syncwarp();
    };
    if (warp < AHEAD) produce(warp);

    {
        double acc[4][8][2];
        double af0[4], bf0[8];
        const int fa = q4 * LD + wm * 32 + g4 * 2;
        const int fb = RBK * LD + q4 * LD + wn * 64 + g4 * 2;
        int tl = 0, ch = 0;
        for (int g = 0; g < G; ++g) {
            const int s = g % NST;
            const unsigned int ph = (unsigned int)(g / NST) & 1u;
            const int64_t i0 = (it_begin + tl) * BM;
            if (warp == (g & (NW - 1))) produce(g + AHEAD);
            if (ch == 0 && PRO != PRO_DIFF) {
#pragma unroll
                for (int t = 0; t < 4; ++t)
#pragma unroll
                    for (int u = 0; u < 8; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;
            }
            mbar_wait(full + s, ph);
            const double* pa = smem + s * RING::STAGE + fa;
            const double* pb = smem + s * RING::STAGE + fb;
            if (ch == 0 && PRO == PRO_DIFF) {
                diff_prologue<FAM, LD, LD>(acc, kp, smem + s * RING::STAGE + wm * 32 + g4 * 2,
                                           smem + s * RING::STAGE + RBK * LD + wn * 64 + q4 * 4, s_tab);
            } else {
                int ksteps;
                if (ch == 0) {
                    ksteps = a.prows >> 2;
                } else {
                    const int rem = a.K - (ch - 1) * RBK;
                    ksteps = rem >= RBK ? RING::KSTEPS : ((rem + 3) >> 2);
                }
                // single-buffered fragments: the other warp of the sub-partition covers the LDS latency (double
                // buffering measured identical in round 1: 34.44 vs 34.43 TFLOP/s at n = 4095).  Whole chunks run fully
                // unrolled (constant LDS offsets, no loop arithmetic between the DMMA groups).
                if (ksteps == RING::KSTEPS) {
#pragma unroll
                    for (int ks = 0; ks < RING::KSTEPS; ++ks) {
                        load_frags_ws(af0, bf0, pa, pb, ks);
                        mma_tile(acc, af0, bf0);
                    }
                } else {
#pragma unroll 1
                    for (int ks = 0; ks < ksteps; ++ks) {
                        load_frags_ws(af0, bf0, pa, pb, ks);
                        mma_tile(acc, af0, bf0);
                    }
                }
                if (ch == 0) {
                    // covariance from the expanded form (alpha, beta are two rows of the contraction); accumulators
                    // become -k so that the main loop yields T - k
#pragma unroll
                    for (int t = 0; t < 4; ++t)
#pragma unroll
                        for (int u = 0; u < 8; ++u)
#pragma unroll
                            for (int e = 0; e < 2; ++e) acc[t][u][e] = neg_kexpand_tab<FAM>(acc[t][u][e], kp, s_tab);
                }
            }
            // this warp is done with stage s (all its LDS results have been consumed)
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + s);

            if (ch == T - 1) {
                column_squares(acc, i0 + BM <= a.I, i0 + wm * 32, a.I, lane, rs);
                ch = 0;
                ++tl;
            } else {
                ++ch;
            }
        }
    }

    __syncthreads();
#pragma unroll
    for (int e = 0; e < 2; ++e) s_red[wm * BN + wn * 64 + (g4 >> 1) * 16 + (q4 * 2 + e) * 2 + (g4 & 1)] = rs[e];
    __syncthreads();
    if (tid < BN && j0 + tid < a.J) {
        const double r = ((s_red[tid] + s_red[BN + tid]) + s_red[2 * BN + tid]) + s_red[3 * BN + tid];
        a.out[split * a.ldo + j0 + tid] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// TMA + mbarrier variant of the plain update  C[i,j] -= sum_k A[k,i] B[k,j]  for callers that GUARANTEE fully padded
// operands (every 128-wide tile of A and B readable and finite; the distributed MI set-up does).  Same ring, fragment
// layout and rotating producer as ivar_ws_kernel<RingSync>, one 128x128 tile per CTA, no prologue.
// ---------------------------------------------------------------------------------------------
constexpr int SUBWS_SMEM_DOUBLES = WS_STAGES * WS_STAGE + 2 * WS_STAGES;
constexpr size_t SUBWS_SMEM_BYTES = (size_t)SUBWS_SMEM_DOUBLES * sizeof(double);

template <bool TMAP>
__global__ void __launch_bounds__(256, 1) sub_ws_kernel(const __grid_constant__ CoreArgs a, const __grid_constant__ TmaMaps maps) {
    constexpr int BM = WS_BM, LD = WS_LD, NW = 8;
    extern __shared__ __align__(128) double smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + WS_STAGES * WS_STAGE);
    uint64_t* empty = full + WS_STAGES;

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t j0 = (int64_t)blockIdx.x * BN;
    const int64_t i0 = (int64_t)blockIdx.y * BM;
    if (a.upper_only && i0 >= j0 + BN) return;  // tile strictly below the diagonal of a symmetric update
    // first K chunk that can hold a non-zero of this column tile (lower-triangular B: rows < global column are zero)
    int c_begin = 0;
    if (a.tri_blk > 0) {
        const int64_t gcol = ((j0 / a.tri_blk) * a.tri_world + a.tri_rank) * a.tri_blk + (j0 % a.tri_blk);
        c_begin = (int)(gcol / WS_BK);
    }
    const int c_end = (a.K + WS_BK - 1) / WS_BK;
    const int G = c_end > c_begin ? c_end - c_begin : 0;  // chunks this CTA walks: c_begin + g
    if (G == 0) return;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < WS_STAGES; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    const int wm = warp & 3, wn = warp >> 2;
    const int g4 = lane >> 2, q4 = lane & 3;

    auto produce = [&](int g) {
        if (g >= G) return;
        const int c = c_begin + g;
        const int s = g % WS_STAGES;
        const unsigned int ph = (unsigned int)(g / WS_STAGES) & 1u;
        mbar_wait(empty + s, ph ^ 1u);
        double* stA = smem + s * WS_STAGE;
        double* stB = stA + WS_BK * LD;
        if (TMAP) {
            if (lane == 0) {
                mbar_arrive_expect_tx(full + s, (unsigned int)WS_BK * 2u * LD * 8u);
                tma_load_2d(stA, &maps.a_main, (int)i0, c * WS_BK, full + s);
                tma_load_2d(stB, &maps.b_main, (int)j0, c * WS_BK, full + s);
            }
            __syncwarp();
            return;
        }
        const double* srcA = a.A + (int64_t)c * WS_BK * a.lda + i0;
        const double* srcB = a.B + (int64_t)c * WS_BK * a.ldb + j0;
        const int rem = a.K - c * WS_BK;
        const int krows = rem < WS_BK ? rem : WS_BK;
        const int ksteps = rem >= WS_BK ? WS_KSTEPS : ((rem + 3) >> 2);
        if (krows < ksteps * 4) {
            for (int r = krows; r < ksteps * 4; ++r) {
                for (int cc = lane * 2; cc < BM; cc += 64) {
                    *reinterpret_cast<double2*>(stA + r * LD + cc) = make_double2(0.0, 0.0);
                    *reinterpret_cast<double2*>(stB + r * LD + cc) = make_double2(0.0, 0.0);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            __syncwarp();
        }
        if (lane == 0) {
            mbar_arrive_expect_tx(full + s, (unsigned int)krows * (BM + BN) * 8u);
#pragma unroll 4
            for (int r = 0; r < krows; ++r) {
                bulk_g2s(stA + r * LD, srcA + (int64_t)r * a.lda, BM * 8u, full + s);
                bulk_g2s(stB + r * LD, srcB + (int64_t)r * a.ldb, BN * 8u, full + s);
            }
        }
        __syncwarp();
    };
    if (warp < WS_AHEAD) produce(warp);

    double acc[4][8][2];
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int u = 0; u < 8; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;
    double af0[4], bf0[8];
    const int fa = q4 * LD + wm * 32 + g4 * 2;
    const int fb = WS_BK * LD + q4 * LD + wn * 64 + g4 * 2;
    for (int g = 0; g < G; ++g) {
        const int s = g % WS_STAGES;
        const unsigned int ph = (unsigned int)(g / WS_STAGES) & 1u;
        if (warp == (g & (NW - 1))) produce(g + WS_AHEAD);
        mbar_wait(full + s, ph);
        const double* pa = smem + s * WS_STAGE + fa;
        const double* pb = smem + s * WS_STAGE + fb;
        const int rem = a.K - (c_begin + g) * WS_BK;
        if (rem >= WS_BK) {
#pragma unroll
            for (int ks = 0; ks < WS_KSTEPS; ++ks) {
                load_frags_ws(af0, bf0, pa, pb, ks);
                mma_tile(acc, af0, bf0);
            }
        } else {
            const int ksteps = (rem + 3) >> 2;
#pragma unroll 1
            for (int ks = 0; ks < ksteps; ++ks) {
                load_frags_ws(af0, bf0, pa, pb, ks);
                mma_tile(acc, af0, bf0);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
    }
    // C -= acc, two adjacent columns per 16-byte access
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int64_t i = i0 + wm * 32 + (t >> 1) * 16 + g4 * 2 + (t & 1);
        if (i >= a.I) continue;
#pragma unroll
        for (int u2 = 0; u2 < 4; ++u2)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int64_t j = j0 + wn * 64 + u2 * 16 + (q4 * 2 + e) * 2;
                if (j >= a.J) continue;
                double* dst = a.out + i * a.ldo + j;
                const double v0 = acc[t][u2 * 2][e], v1 = acc[t][u2 * 2 + 1][e];
                if (a.upper_only && j < i) {
                    // symmetric update of a diagonal-straddling tile: the strictly-lower part is left untouched
                    if (j + 1 == i && j + 1 < a.J) dst[1] -= v1;
                } else if (j + 1 < a.J) {
                    double2 c = *reinterpret_cast<double2*>(dst);
                    c.x -= v0;
                    c.y -= v1;
                    *reinterpret_cast<double2*>(dst) = c;
                } else {
                    dst[0] -= v0;
                }
            }
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// rows x ld doubles, row-major, box = 132 columns x box_rows; out-of-range elements read as zero
int make_map(CUtensorMap* m, const double* base, int64_t ld, int64_t rows, int box_rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) {
        gpx_set_error("ivar_ws: cuTensorMapEncodeTiled is not available from this driver");
        return GPX_EINVAL;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)(rows > 0 ? rows : 1)};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    const cuuint32_t box[2] = {(cuuint32_t)WS_LD, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        gpx_set_error("ivar_ws: cuTensorMapEncodeTiled failed with CUresult %d (ld %lld, rows %lld, box rows %d)", (int)r,
                      (long long)ld, (long long)rows, box_rows);
        return GPX_EINVAL;
    }
    return GPX_OK;
}

template <int FAM, int PRO, class RING, bool TMAP>
int launch_ivar_ws_ring(gpx_handle h, const CoreArgs& a, dim3 grid, cudaStream_t st) {
    TmaMaps maps;
    memset(&maps, 0, sizeof(maps));
    int rc;
    if (TMAP) {
        // the K extent of the main maps is the CURRENT design size: rows >= n are zero-filled, never read
        if (a.K > 0) {
            if ((rc = make_map(&maps.a_main, a.A, a.lda, a.K, RING::RBK))) return rc;
            if ((rc = make_map(&maps.b_main, a.B, a.ldb, a.K, RING::RBK))) return rc;
        }
        if ((rc = make_map(&maps.a_pro, a.Ap, a.lda, a.prows, a.prows))) return rc;
        if ((rc = make_map(&maps.b_pro, a.Bp, a.ldb, a.prows, a.prows))) return rc;
    }
    rc = gpx_ensure_smem(h, (const void*)ivar_ws_kernel<FAM, PRO, RING, TMAP>, RING::SMEM_BYTES, "ivar_ws");
    if (rc) return rc;
    ivar_ws_kernel<FAM, PRO, RING, TMAP><<<grid, 256, RING::SMEM_BYTES, st>>>(a, h->kp, maps);
    return gpx_check_launch("ivar_ws");
}

template <int FAM, int PRO>
int launch_ivar_ws(gpx_handle h, const CoreArgs& a, dim3 grid, cudaStream_t st) {
    // every prologue fits one chunk of every ring (EXPANDED <= 16 rows, DIFF <= 16 coordinates, chunks >= 24 rows)
    switch (h->ivar_ring) {
        case 1: return launch_ivar_ws_ring<FAM, PRO, RingSync, true>(h, a, grid, st);
        case 2: return launch_ivar_ws_ring<FAM, PRO, RingDeep, true>(h, a, grid, st);
        default: return launch_ivar_ws_ring<FAM, PRO, RingSync, false>(h, a, grid, st);
    }
}

template <int FAM, int EPI, int PRO>
int launch_core(gpx_handle h, const CoreArgs& a, int64_t jt, int64_t it_or_splits, cudaStream_t st) {
    dim3 grid((unsigned)jt, (unsigned)it_or_splits);
    int rc = gpx_ensure_smem(h, (const void*)dmma_core_kernel<FAM, EPI, PRO>, Cfg::SMEM_BYTES, "dmma core");
    if (rc) return rc;
    dmma_core_kernel<FAM, EPI, PRO><<<grid, Cfg::NT, Cfg::SMEM_BYTES, st>>>(a, h->kp);
    return gpx_check_launch("dmma core");
}

int check_operand(const double* p, int64_t ld, const char* name) {
    if (!gpx_aligned16(p) || (ld & 1)) {
        gpx_set_error("dmma core: operand %s must be 16-byte aligned with an even leading dimension", name);
        return GPX_EALIGN;
    }
    return GPX_OK;
}

// rows of the prologue chunk for this handle's kernel, or < 0 if the form cannot be used
int prologue_rows(gpx_handle h, int prologue) {
    if (prologue == PRO_DIFF) return h->kp.d;
    if (prologue == PRO_EXPANDED && h->kp.d + 2 <= GPX_KROWS) return (h->kp.d + 2 + 3) & ~3;
    return -1;
}

// ---------------------------------------------------------------------------------------------
// INT8 tensor-core IVAR core (tcgen05.mma .kind::i8): the contraction S = W_M^T W_C emulated exactly by fixed-point
// slicing (Ozaki-style).  Each column x = W[:, c] gets a power-of-two scale 2^e_c > max_i |x_i| and the integer
//     Y[i, c] = rint(x_i * 2^(54 - e_c)),   |Y| <= 2^54,
// written as I8_L = 7 balanced base-256 digits  Y = sum_p a_p 256^(6-p),  a_1..a_6 in [-128, 127],  |a_0| <= 64.
// Then  sum_i Y_M Y_C = sum_t D_t 256^(12-t),  D_t = sum_{p+q=t} sum_i a_p(m) b_q(c),  and the kernel keeps the
// diagonals t = 0..6 (28 int8 products per K step): one exact int32 TMEM accumulator per diagonal
// (|D_t| <= (t+1) K 2^14 < 2^31 for K <= 16384).
// Error of one pair, in units u = 2^(e_m + e_c - 54) (so u <= 4 * 2^-54 * max|W_M[:,m]| max|W_C[:,c]|):
//     rounding of the operands     |x~ - x| <= 2^(e - 55) and |x| < 2^e per side: <= K u (1 + 2^-56)
//     dropped diagonals t = 7..12  <= K 2^14 sum_{t>=7} (13 - t) 256^(12 - t) / 2^54 < 6.03 K u
//     the FP64 recombination       one rounding of S (relative 2^-53)
// i.e. |S_i8 - S| <= 7.04 K u + |S| 2^-53, against the FP64 DMMA bound ~ K eps sum_i |W_M[i,m]| |W_C[i,c]|.
// L = 7 is the smallest L for which the bound stays at the FP64 level (L = 6 is 256 times coarser); L = 8 would add
// 8 products per K step and an eighth accumulator (8 x 64 TMEM columns: no room for anything else) for accuracy the
// FP64 epilogue cannot use.  tests/test_ivar_int8_core.py checks the model against exact integer arithmetic, and
// tests/test_ivar_contraction_exact.py checks this kernel against the model bit for bit, pair by pair.
// Domain of the bound: both column maxima >= 2^-1044 (2^(e - 30) > 0) and 2^(e_m + e_c - 60) normal; outside it S_i8
// flushes to 0, which in IVAR (|W| <= sqrt(k) < 2^512) only happens where |S| < 2^-517 and S^2 is not a normal number.
//
// Slices live K-major ([p][column][k], ldk = roundup(n, 64) bytes) in caller scratch (gpx_set_ivar_scratch) and are
// rebuilt from the FP64 factors on every scoring call by ivar_slice_kernel: one streaming pass over W (0.75 ms of the
// 90.7 ms cfg-2 call at n = 255 on a B200, DESIGN.md section 5), so no other producer of W has to know about them.
//
// ivar_i8_kernel: 128 (integration points) x 64 (candidates) tiles, K in 32-byte chunks (SWIZZLE_32B, 4 stages of 42 KB).
//   warp 16    TMA producer: one 3-D tensor-map load per operand and chunk brings all 7 slices.
//   warp 17    MMA issuer (one lane): 10 tcgen05.mma per chunk into the 7 accumulators (7 x 64 of the 512 TMEM columns):
//             each A slice meets a stack of adjacent B slices (N up to 256) and writes several diagonals at once, so a
//             chunk reads 96 KB of operands from smem instead of the 168 KB of 28 separate N = 64 products.
//   warps 0-15 epilogue: warp w owns TMEM lanes 32 (w % 4).. (its integration points) and columns 16 (w / 4)..
//             Per tile it first evaluates -k for its 16 pairs (same prologue arithmetic as the DMMA kernels), then
//             waits for the accumulators, drains them two columns at a time (int64 recombination, one FP64 fma with
//             the scales and -k) into per-thread column sums of (S - k)^2 kept across the CTA's M tiles, and hands
//             TMEM back as soon as the last load has landed.  The 7 accumulators leave no room for a second TMEM
//             buffer, so this is the overlap there is: the next tile's MMAs run under the -k work of that tile.
//   At 18 warps the register file allows 96 registers a thread; 16 epilogue warps beat 8 (168 registers) because
//   the -k work is latency bound (cfg-2 n = 255 call on a B200 at 1000 W: 92.2 ms against 97.7 ms, DESIGN.md 5).
//   Kernel time at cfg-2 n = 255 (B200, 1000 W, 1965 MHz; DESIGN.md 5): 89.9 ms with 28 MMAs per K step and 64-byte
//   chunks x 2, 68.0 ms now.  The MMA/TMA stream alone (epilogue handing TMEM back at once) takes 47.9 ms and TMA alone
//   46.5 ms: 32-byte boxes cost the TMA more than 64-byte ones (29.8 ms), but the 64-byte ring fits only 2 stages
//   (69.8 ms).  What is left above the stream is the TMEM drain, during which the MMAs wait.
// Determinism: fixed M-split grid and rasterisation as ivar_ws_kernel; per-column summation order independent of the
// candidate's position in its tile.
// ---------------------------------------------------------------------------------------------
constexpr int I8_L = 7;
constexpr int I8_BM = 128;
constexpr int I8_BN = 64;
constexpr int I8_BK = 32;                                  // bytes of K per chunk = one MMA K step = the swizzle span
constexpr int I8_A_BYTES = I8_L * I8_BM * I8_BK;           // 28672
constexpr int I8_B_BYTES = I8_L * I8_BN * I8_BK;           // 14336
constexpr int I8_STAGE = I8_A_BYTES + I8_B_BYTES;          // multiple of 1024
constexpr int I8_STAGES = 4;
constexpr int I8_EPI_WARPS = 16;                        // 4 per TMEM lane quarter
constexpr int I8_EPI_COLS = 4 * I8_BN / I8_EPI_WARPS;  // columns per epilogue thread
constexpr int I8_THREADS = (I8_EPI_WARPS + 2) * 32;
constexpr int I8_KMAX = GPX_I8_MAX_N;
// smem: ring | neg. exp table | column prologue rows | column scales | reduction | barriers | tmem address
constexpr size_t I8_SMEM_BYTES =
    1024 + (size_t)I8_STAGES * I8_STAGE + 256 * 8 + GPX_KROWS * I8_BN * 8 + I8_BN * 8 + 4 * I8_BN * 8 + 16 * 8 + 16;

struct I8Maps {
    CUtensorMap a, b;
};

struct I8Args {
    const double* Ap;  // prologue rows of the integration points (ld lda) and of the candidates (ld ldb)
    const double* Bp;
    const double* fa;  // per-column scales 2^(e - 30)
    const double* fb;
    double* out;
    int64_t lda, ldb, ldo;
    int64_t I, J;
    int K;
    int np;            // prologue rows read: EXPANDED d + 2, DIFF d
    int tiles_per_cta, group_w, splits;
};

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}

// K-major operand, 32-byte swizzle: 8-row core groups 256 bytes apart (SBO), LBO unused, descriptor version 1,
// layout type 6
__device__ __forceinline__ uint64_t i8_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)6 << 61);
}
// kind::i8: D s32, A and B signed, both K-major, M = 128, N = 64 nq
template <int NQ>
__device__ __forceinline__ void i8_mma(uint32_t dtm, uint64_t ad, uint64_t bd, uint32_t acc) {
    constexpr uint32_t idesc =
        (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NQ * I8_BN >> 3) << 17) | ((uint32_t)(I8_BM >> 4) << 24);
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(dtm),
        "l"(ad), "l"(bd), "r"(idesc), "r"(acc)
        : "memory");
}
// One K step of the 7 diagonals: A slice p against the stack of B slices q0 .. q0 + nq - 1 (adjacent in smem with the
// uniform core-group stride, so one operand of N = 64 nq) writes a_p^T b_q into D_{p+q}, which sit 64 TMEM columns
// apart.  N <= 256 splits the 28 slice products into these 10 MMAs; the p = 0 pair covers all 448 columns and comes
// first, so it alone carries the tile's first-step overwrite.
template <int P, int Q0, int NQ>
__device__ __forceinline__ void i8_mma_stack(uint32_t tmem, uint32_t sa, uint32_t sb, uint32_t first) {
    i8_mma<NQ>(tmem + (P + Q0) * I8_BN, i8_desc(sa + P * (I8_BM * I8_BK)), i8_desc(sb + Q0 * (I8_BN * I8_BK)),
               P != 0 || !first);
}
__device__ __forceinline__ void i8_mma_kstep(uint32_t tmem, uint32_t sa, uint32_t sb, uint32_t first) {
    i8_mma_stack<0, 0, 4>(tmem, sa, sb, first);
    i8_mma_stack<0, 4, 3>(tmem, sa, sb, first);
    i8_mma_stack<1, 0, 4>(tmem, sa, sb, first);
    i8_mma_stack<1, 4, 2>(tmem, sa, sb, first);
    i8_mma_stack<2, 0, 4>(tmem, sa, sb, first);
    i8_mma_stack<2, 4, 1>(tmem, sa, sb, first);
    i8_mma_stack<3, 0, 4>(tmem, sa, sb, first);
    i8_mma_stack<4, 0, 3>(tmem, sa, sb, first);
    i8_mma_stack<5, 0, 2>(tmem, sa, sb, first);
    i8_mma_stack<6, 0, 1>(tmem, sa, sb, first);
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, int (&v)[2]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];\n" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// |v| < 2^51 -> exact double without the conversion unit
__device__ __forceinline__ double i64_to_f64(int64_t v) {
    return __longlong_as_double(0x4338000000000000LL + v) - 6755399441055744.0;
}

template <int FAM, int PRO>
__global__ void __launch_bounds__(I8_THREADS, 1) ivar_i8_kernel(const __grid_constant__ I8Args a, const __grid_constant__ KParams kp,
                                                                const __grid_constant__ I8Maps maps) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* ring = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    double* s_tab = reinterpret_cast<double*>(ring + I8_STAGES * I8_STAGE);
    double* s_colp = s_tab + 256;               // [GPX_KROWS][I8_BN]
    double* s_fb = s_colp + GPX_KROWS * I8_BN;  // [I8_BN]
    double* s_red = s_fb + I8_BN;               // [4][I8_BN]
    uint64_t* full = reinterpret_cast<uint64_t*>(s_red + 4 * I8_BN);
    uint64_t* empty = full + I8_STAGES;
    uint64_t* acc_full = empty + I8_STAGES;
    uint64_t* acc_empty = acc_full + 1;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(acc_empty + 1);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // rasterisation of ivar_ws_kernel: j-group -> M-split -> tile
    const int64_t jtiles = (a.J + I8_BN - 1) / I8_BN;
    const int64_t gw = a.group_w;
    const int64_t per_group = gw * a.splits;
    const int64_t jg = blockIdx.x / per_group;
    const int64_t rem = blockIdx.x - jg * per_group;
    const int64_t gsz = (jtiles - jg * gw) < gw ? (jtiles - jg * gw) : gw;
    const int64_t split = rem / gsz;
    const int64_t jt = jg * gw + rem % gsz;
    if (split >= a.splits) return;
    const int64_t j0 = jt * I8_BN;
    const int64_t itiles = (a.I + I8_BM - 1) / I8_BM;
    const int64_t it_begin = split * a.tiles_per_cta;
    int64_t it_end = it_begin + a.tiles_per_cta;
    if (it_end > itiles) it_end = itiles;
    const int ntiles = it_end > it_begin ? (int)(it_end - it_begin) : 0;
    const int kch = (a.K + I8_BK - 1) / I8_BK;

    if (tid == 0) {
        for (int s = 0; s < I8_STAGES; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, 1);
        }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, I8_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == I8_EPI_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(s_tmem)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    if (tid < 256) s_tab[tid] = -kp.signal * gpx_exp2_tab[tid];
    for (int i = tid; i < a.np * I8_BN; i += I8_THREADS) {
        const int q = i / I8_BN, c = i - q * I8_BN;
        s_colp[i] = j0 + c < a.J ? a.Bp[(int64_t)q * a.ldb + j0 + c] : 0.0;
    }
    if (tid < I8_BN) s_fb[tid] = j0 + tid < a.J ? a.fb[j0 + tid] : 0.0;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem;

    if (warp == I8_EPI_WARPS) {
        // ---- TMA producer ----
        if (lane == 0) {
            int s = 0;
            unsigned ph = 0;
            for (int tl = 0; tl < ntiles; ++tl) {
                const int i0 = (int)((it_begin + tl) * I8_BM);
                for (int kc = 0; kc < kch; ++kc, s = s + 1 == I8_STAGES ? 0 : s + 1, ph ^= s == 0) {
                    mbar_wait(empty + s, ph ^ 1u);
                    mbar_arrive_expect_tx(full + s, (unsigned)I8_STAGE);
                    unsigned char* st = ring + s * I8_STAGE;
                    tma_load_3d(st, &maps.a, kc * I8_BK, i0, 0, full + s);
                    tma_load_3d(st + I8_A_BYTES, &maps.b, kc * I8_BK, (int)j0, 0, full + s);
                }
            }
        }
    } else if (warp == I8_EPI_WARPS + 1) {
        // ---- MMA issuer ----
        if (lane == 0) {
            const uint32_t ring_s = smem_u32(ring);
            int s = 0;
            unsigned ph = 0;
            for (int tl = 0; tl < ntiles; ++tl) {
                if (tl > 0) {
                    mbar_wait(acc_empty, (unsigned)(tl - 1) & 1u);  // the epilogue has read the previous tile
                    tc_fence_after();
                }
                for (int kc = 0; kc < kch; ++kc, s = s + 1 == I8_STAGES ? 0 : s + 1, ph ^= s == 0) {
                    mbar_wait(full + s, ph);
                    tc_fence_after();
                    const uint32_t sa = ring_s + s * I8_STAGE, sb = sa + I8_A_BYTES;
                    i8_mma_kstep(tmem, sa, sb, kc == 0);
                    tc_commit(empty + s);
                }
                tc_commit(acc_full);
            }
        }
    } else {
        // ---- epilogue ----
        const int quad = warp & 3, c00 = (warp >> 2) * I8_EPI_COLS;
        const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16) + c00;
        double p[I8_EPI_COLS];
#pragma unroll
        for (int j = 0; j < I8_EPI_COLS; ++j) p[j] = 0.0;
        for (int tl = 0; tl < ntiles; ++tl) {
            const int64_t m = (it_begin + tl) * I8_BM + quad * 32 + lane;
            const bool mok = m < a.I;
            // -k of the thread's pairs, evaluated while the tensor cores work on this tile (and, from the second tile
            // on, right after the previous tile's accumulators were handed back)
            double nk[I8_EPI_COLS];
#pragma unroll
            for (int j = 0; j < I8_EPI_COLS; ++j) nk[j] = 0.0;
            for (int q = 0; q < a.np; ++q) {
                const double x = mok ? a.Ap[(int64_t)q * a.lda + m] : 0.0;
                const double* y = s_colp + q * I8_BN + c00;
#pragma unroll
                for (int j = 0; j < I8_EPI_COLS; ++j) {
                    if (PRO == PRO_EXPANDED) nk[j] = fma(x, y[j], nk[j]);
                    else kacc_dim<FAM>(nk[j], kp, q, x, y[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < I8_EPI_COLS; ++j)
                nk[j] = PRO == PRO_EXPANDED ? neg_kexpand_tab<FAM>(nk[j], kp, s_tab) : kfinish_tab<FAM>(nk[j], kp, s_tab);
            const double fm = mok ? a.fa[m] : 0.0;
            mbar_wait(acc_full, (unsigned)tl & 1u);
            tc_fence_after();
#pragma unroll
            for (int cb = 0; cb < I8_EPI_COLS; cb += 2) {
                int d[I8_L][2];
#pragma unroll
                for (int t = 0; t < I8_L; ++t) tmem_ld2(trow + t * I8_BN + cb, d[t]);
                tmem_wait_ld();
                if (cb == I8_EPI_COLS - 2) {
                    // every accumulator of this tile is in registers: hand TMEM back to the MMA issuer
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty);
                }
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int64_t hi = ((int64_t)d[0][j] << 24) + ((int64_t)d[1][j] << 16) + ((int64_t)d[2][j] << 8) + d[3][j];
                    const int64_t lo = ((int64_t)d[4][j] << 16) + ((int64_t)d[5][j] << 8) + d[6][j];
                    // S - k with S = (D_0..3 2^24 + D_4..6) (fm fb): the scale product inside one fma with -k
                    const double R = fma(i64_to_f64(hi), 0x1p24, i64_to_f64(lo));
                    const double v = mok ? __fma_rn(R, __dmul_rn(fm, s_fb[c00 + cb + j]), nk[cb + j]) : 0.0;
                    p[cb + j] = fma(v, v, p[cb + j]);
                }
            }
        }
        // column sums over the warp's 32 rows, pairing lanes 16, 8, 4, 2, 1 apart: a reduce-scatter that leaves
        // lane l with column c00 + l % I8_EPI_COLS (lanes 16 apart hold the same sum when a warp has 16 columns)
#pragma unroll
        for (int st = 0; st < 5; ++st) {
            const int off = 16 >> st;
            if (off >= I8_EPI_COLS) {
#pragma unroll
                for (int j = 0; j < I8_EPI_COLS; ++j) p[j] += __shfl_xor_sync(0xffffffffu, p[j], off);
                continue;
            }
            const bool up = (lane & off) != 0;
#pragma unroll
            for (int j = 0; j < off; ++j) {
                const double keep = up ? p[j + off] : p[j];
                const double send = up ? p[j] : p[j + off];
                p[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
        }
        if (lane < I8_EPI_COLS) s_red[quad * I8_BN + c00 + lane] = p[0];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == I8_EPI_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tmem) : "memory");
    }
    if (tid < I8_BN && j0 + tid < a.J) {
        const double r = ((s_red[tid] + s_red[I8_BN + tid]) + s_red[2 * I8_BN + tid]) + s_red[3 * I8_BN + tid];
        a.out[split * a.ldo + j0 + tid] = r;
    }
}

// digits of one side: S[p][c][k] (int8, ldk bytes per column, slice stride sstride) and f[c] = 2^(e_c - 30)
// block: 32 columns x 8 row lanes
__global__ void __launch_bounds__(256) ivar_slice_kernel(const double* __restrict__ W, int64_t ldw, int n, int64_t ncols,
                                                         int8_t* __restrict__ S, int64_t ldk, int64_t sstride,
                                                         double* __restrict__ f) {
    __shared__ double s_mx[8][32];
    __shared__ __align__(16) int8_t s_dig[I8_L][32][64];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t c = (int64_t)blockIdx.x * 32 + tx;
    const bool cok = c < ncols;
    double mx = 0.0;
    if (cok)
        for (int i = ty; i < n; i += 8) mx = fmax(mx, fabs(W[(int64_t)i * ldw + c]));
    s_mx[ty][tx] = mx;
    __syncthreads();
    mx = s_mx[0][tx];
#pragma unroll
    for (int r = 1; r < 8; ++r) mx = fmax(mx, s_mx[r][tx]);
    int e = 0;
    if (mx > 0.0) frexp(mx, &e);  // mx < 2^e
    if (ty == 0 && cok) f[c] = ldexp(1.0, e - 30);
    const int kpad = (n + 63) & ~63;
    for (int i0 = 0; i0 < kpad; i0 += 64) {
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int i = i0 + ty + 8 * r;
            long long Y = 0;
            if (cok && i < n) Y = llrint(ldexp(W[(int64_t)i * ldw + c], 54 - e));
#pragma unroll
            for (int pp = I8_L - 1; pp > 0; --pp) {
                const int dg = (int)((Y + 128) & 255) - 128;
                s_dig[pp][tx][ty + 8 * r] = (int8_t)dg;
                Y = (Y - dg) >> 8;
            }
            s_dig[0][tx][ty + 8 * r] = (int8_t)Y;
        }
        __syncthreads();
        // 7 x 32 runs of 64 bytes -> 16-byte stores
        for (int v = threadIdx.x; v < I8_L * 32 * 4; v += 256) {
            const int pp = v / 128, col = (v / 4) & 31, part = v & 3;
            const int64_t cc = (int64_t)blockIdx.x * 32 + col;
            if (cc < ncols)
                *reinterpret_cast<int4*>(S + pp * sstride + cc * ldk + i0 + part * 16) =
                    *reinterpret_cast<const int4*>(&s_dig[pp][col][part * 16]);
        }
    }
}

// 3-D map over the slices of one side: dims {n (K bytes), ncols, 7}, box {32, rows, 7}, 32-byte swizzle
int make_i8_map(CUtensorMap* m, const int8_t* base, int64_t ldk, int64_t n, int64_t ncols, int64_t sstride, int box_rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) {
        gpx_set_error("ivar_i8: cuTensorMapEncodeTiled is not available from this driver");
        return GPX_EINVAL;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)n, (cuuint64_t)ncols, (cuuint64_t)I8_L};
    const cuuint64_t strides[2] = {(cuuint64_t)ldk, (cuuint64_t)sstride};
    const cuuint32_t box[3] = {(cuuint32_t)I8_BK, (cuuint32_t)box_rows, (cuuint32_t)I8_L};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        gpx_set_error("ivar_i8: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
        return GPX_EINVAL;
    }
    return GPX_OK;
}

// scratch layout for one call: [slices of M][slices of C][fa][fb]; returns the bytes needed
int64_t i8_layout(int64_t M, int64_t C, int64_t n, int64_t* ldk, int64_t* sm, int64_t* sc) {
    *ldk = (n + 63) & ~(int64_t)63;
    *sm = ((M + I8_BM - 1) / I8_BM * I8_BM) * *ldk;
    *sc = ((C + I8_BM - 1) / I8_BM * I8_BM) * *ldk;
    return I8_L * (*sm + *sc) + 8 * (((M + 1) & ~(int64_t)1) + ((C + 1) & ~(int64_t)1)) + 256;
}

}  // namespace

// number of i-splits for the IVAR grid: fill the machine in whole waves
static int ivar_splits_for(gpx_handle h, int64_t M, int64_t C, int bm, int bn = BN) {
    const int64_t jt = (C + bn - 1) / bn;
    const int64_t itl = (M + bm - 1) / bm;
    const int sms = h->sm_count > 0 ? h->sm_count : 148;
    int best = 1;
    double best_eff = -1.0;
    for (int s = 1; s <= 32 && s <= itl; ++s) {
        const int64_t tps = (itl + s - 1) / s;
        const int64_t seff = (itl + tps - 1) / tps;  // splits that actually have work
        if (seff != s) continue;
        const int64_t ctas = jt * s;
        const int64_t waves = (ctas + sms - 1) / sms;
        // time ~ waves * tiles-per-cta ; ideal = jt*itl / sms
        const double eff = (double)(jt * itl) / (double)(waves * sms * tps);
        if (eff > best_eff + 1e-9) {
            best_eff = eff;
            best = s;
        }
    }
    return best;
}
int gpx_ivar_splits(gpx_handle, int64_t, int64_t) { return 32; }  // workspace bound: never more than 32 splits

// INT8 core: slice both factors into the handle's scratch, then one ivar_i8_kernel launch (same workspace contract as
// ivar_ws_kernel: partial column sums per M-split)
static int launch_ivar_i8(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* Ma_rows, int64_t M,
                          const double* Wc, int64_t ldc, const double* Cb_rows, int64_t C, int64_t n, double* partial,
                          int64_t ldp, int* nsplit_out, cudaStream_t st) {
    int64_t ldk, sm, sc;
    i8_layout(M, C, n, &ldk, &sm, &sc);
    int8_t* Sm = reinterpret_cast<int8_t*>(((uintptr_t)h->i8_scratch + 127) & ~(uintptr_t)127);
    int8_t* Sc = Sm + I8_L * sm;
    double* fa = reinterpret_cast<double*>(Sc + I8_L * sc);
    double* fb = fa + ((M + 1) & ~(int64_t)1);
    ivar_slice_kernel<<<(unsigned)((M + 31) / 32), 256, 0, st>>>(Wm, ldm, (int)n, M, Sm, ldk, sm, fa);
    int rc = gpx_check_launch("ivar_slice");
    if (rc) return rc;
    ivar_slice_kernel<<<(unsigned)((C + 31) / 32), 256, 0, st>>>(Wc, ldc, (int)n, C, Sc, ldk, sc, fb);
    if ((rc = gpx_check_launch("ivar_slice"))) return rc;
    I8Maps maps;
    memset(&maps, 0, sizeof(maps));
    if ((rc = make_i8_map(&maps.a, Sm, ldk, n, M, sm, I8_BM))) return rc;
    if ((rc = make_i8_map(&maps.b, Sc, ldk, n, C, sc, I8_BN))) return rc;
    const int splits = ivar_splits_for(h, M, C, I8_BM, I8_BN);
    const int64_t itl = (M + I8_BM - 1) / I8_BM;
    const int64_t jt = (C + I8_BN - 1) / I8_BN;
    I8Args a;
    a.Ap = Ma_rows;
    a.Bp = Cb_rows;
    a.fa = fa;
    a.fb = fb;
    a.out = partial;
    a.lda = ldm;
    a.ldb = ldc;
    a.ldo = ldp;
    a.I = M;
    a.J = C;
    a.K = (int)n;
    a.np = prologue == PRO_DIFF ? h->kp.d : h->kp.d + 2;
    a.tiles_per_cta = (int)((itl + splits - 1) / splits);
    a.group_w = h->sm_count > 0 ? h->sm_count : 148;
    a.splits = splits;
    *nsplit_out = splits;
    const dim3 grid((unsigned)(jt * splits), 1u);
#define GPX_I8_LAUNCH(F, P)                                                                                        \
    do {                                                                                                           \
        if ((rc = gpx_ensure_smem(h, (const void*)ivar_i8_kernel<F, P>, I8_SMEM_BYTES, "ivar_i8"))) return rc;    \
        ivar_i8_kernel<F, P><<<grid, I8_THREADS, I8_SMEM_BYTES, st>>>(a, h->kp, maps);                            \
    } while (0)
    if (prologue == PRO_DIFF) {
        GPX_DISPATCH_FAMILY(h->kp.family, GPX_I8_LAUNCH(FAM, PRO_DIFF));
    } else {
        GPX_DISPATCH_FAMILY(h->kp.family, GPX_I8_LAUNCH(FAM, PRO_EXPANDED));
    }
#undef GPX_I8_LAUNCH
    return gpx_check_launch("ivar_i8");
}

int gpx_launch_core_ivar(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* Ma_rows, int64_t M,
                         const double* Wc, int64_t ldc, const double* Cb_rows, int64_t C, int64_t n, double* partial,
                         int64_t ldp, int* nsplit_out, cudaStream_t st) {
    int rc;
    const int prows = prologue_rows(h, prologue);
    GPX_REQUIRE(prows >= 0, GPX_ESIZE, "prologue must be GPX_PRO_DIFF, or GPX_PRO_EXPANDED with d <= GPX_KROWS - 2");
    if ((rc = check_operand(Ma_rows, ldm, "Ma_rows"))) return rc;
    if ((rc = check_operand(Cb_rows, ldc, "Cb_rows"))) return rc;
    if (n > 0) {
        if ((rc = check_operand(Wm, ldm, "Wm"))) return rc;
        if ((rc = check_operand(Wc, ldc, "Wc"))) return rc;
    }
    // the TMA path reads whole 128-wide tiles: operands must be padded to full tiles (the engines do that);
    // anything else goes through the predicated cp.async core
    const bool tma = (ldm % WS_BM) == 0 && (ldc % BN) == 0 && ldm >= (M + WS_BM - 1) / WS_BM * WS_BM &&
                     ldc >= (C + BN - 1) / BN * BN;
    if (tma && h->ivar_core == GPX_CORE_I8 && n > 0 && n <= I8_KMAX) {
        int64_t ldk, sm, sc;
        if (i8_layout(M, C, n, &ldk, &sm, &sc) <= h->i8_scratch_bytes)
            return launch_ivar_i8(h, prologue, Wm, ldm, Ma_rows, M, Wc, ldc, Cb_rows, C, n, partial, ldp, nsplit_out, st);
    }
    const int bm = tma ? WS_BM : Cfg::BM;
    const int splits = ivar_splits_for(h, M, C, bm);
    const int64_t itl = (M + bm - 1) / bm;
    CoreArgs a;
    a.A = Wm;
    a.B = Wc;
    a.Ap = Ma_rows;
    a.Bp = Cb_rows;
    a.out = partial;
    a.lda = ldm;
    a.ldb = ldc;
    a.ldo = ldp;
    a.I = M;
    a.J = C;
    a.K = (int)n;
    a.prows = prows;
    a.tiles_per_cta = (int)((itl + splits - 1) / splits);
    a.upper_only = 0;
    a.ldo_splits = 0;
    a.tri_blk = a.tri_world = a.tri_rank = 0;
    *nsplit_out = splits;
    if (tma) {
        const int64_t jt = (C + BN - 1) / BN;
        // one CTA per SM: a group is one wave of candidate tiles (their W_C tiles must stay L2-resident)
        const int64_t gw = (int64_t)(h->sm_count > 0 ? h->sm_count : 148);
        const int64_t groups = (jt + gw - 1) / gw;
        a.upper_only = (int)gw;
        a.ldo_splits = splits;
        // a group of g tiles owns g*splits consecutive CTAs; only the last group can be short, and the kernel's index
        // decode needs nothing beyond it, so the grid is exactly jt*splits CTAs (round 1 padded the last group to
        // gw*splits slots: 2 520 CTAs that exited at once per cfg-1 step, ~25 us of launch work)
        (void)groups;
        dim3 grid((unsigned)(jt * splits), 1u);
        if (prologue == PRO_DIFF) {
            GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_ivar_ws<FAM, PRO_DIFF>(h, a, grid, st)));
        } else {
            GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_ivar_ws<FAM, PRO_EXPANDED>(h, a, grid, st)));
        }
        return rc;
    }
    if (prologue == PRO_DIFF) {
        GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_core<FAM, EPI_IVAR, PRO_DIFF>(h, a, (C + BN - 1) / BN, splits, st)));
    } else {
        GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_core<FAM, EPI_IVAR, PRO_EXPANDED>(h, a, (C + BN - 1) / BN, splits, st)));
    }
    return rc;
}

int gpx_launch_core_store(gpx_handle h, int prologue, const double* A, int64_t lda, const double* Ap, int64_t I,
                          const double* B, int64_t ldb, const double* Bp, int64_t J, int64_t K, double* out, int64_t ldo,
                          cudaStream_t st) {
    int rc;
    const int prows = prologue_rows(h, prologue);
    GPX_REQUIRE(prows >= 0, GPX_ESIZE, "prologue must be GPX_PRO_DIFF, or GPX_PRO_EXPANDED with d <= GPX_KROWS - 2");
    if ((rc = check_operand(Ap, lda, "Ap"))) return rc;
    if ((rc = check_operand(Bp, ldb, "Bp"))) return rc;
    if ((rc = check_operand(out, ldo, "out"))) return rc;
    if (K > 0) {
        if ((rc = check_operand(A, lda, "A"))) return rc;
        if ((rc = check_operand(B, ldb, "B"))) return rc;
    }
    CoreArgs a;
    a.A = A;
    a.B = B;
    a.Ap = Ap;
    a.Bp = Bp;
    a.out = out;
    a.lda = lda;
    a.ldb = ldb;
    a.ldo = ldo;
    a.I = I;
    a.J = J;
    a.K = (int)K;
    a.prows = prows;
    a.tiles_per_cta = 1;
    a.upper_only = 0;
    a.ldo_splits = 0;
    a.tri_blk = a.tri_world = a.tri_rank = 0;
    const int64_t jt = (J + BN - 1) / BN, it = (I + Cfg::BM - 1) / Cfg::BM;
    if (prologue == PRO_DIFF) {
        GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_core<FAM, EPI_STORE, PRO_DIFF>(h, a, jt, it, st)));
    } else {
        GPX_DISPATCH_FAMILY(h->kp.family, rc = (launch_core<FAM, EPI_STORE, PRO_EXPANDED>(h, a, jt, it, st)));
    }
    return rc;
}

extern "C" int gpx_dgemm_tn_sub(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                                int64_t ldc, int64_t I, int64_t J, int64_t K, int upper_only, void* stream) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    GPX_REQUIRE(I >= 0 && J >= 0 && K >= 0, GPX_EINVAL, "negative size");
    if (I == 0 || J == 0 || K == 0) return GPX_OK;
    GPX_REQUIRE(A && B && C, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE((I + 63) / 64 <= 65535, GPX_ESIZE, "I too large for one launch");
    int rc;
    if ((rc = check_operand(A, lda, "A"))) return rc;
    if ((rc = check_operand(B, ldb, "B"))) return rc;
    if ((rc = check_operand(C, ldc, "C"))) return rc;
    CoreArgs a;
    a.A = A;
    a.B = B;
    a.Ap = a.Bp = nullptr;
    a.out = C;
    a.lda = lda;
    a.ldb = ldb;
    a.ldo = ldc;
    a.I = I;
    a.J = J;
    a.K = (int)K;
    a.prows = 0;
    a.tiles_per_cta = 1;
    a.upper_only = upper_only;
    a.ldo_splits = 0;
    a.tri_blk = a.tri_world = a.tri_rank = 0;
    return launch_core<GPX_SE, EPI_SUB, PRO_NONE>(h, a, (J + BN - 1) / BN, (I + Cfg::BM - 1) / Cfg::BM, (cudaStream_t)stream);
}

// Same update for operands the CALLER guarantees to be fully padded (every 128-wide tile of A's I columns and B's J
// columns readable and finite, lda/ldb multiples of 128 or at least covering the rounded-up extents): TMA + mbarrier kernel,
// one 2-D tensor-map load per operand chunk.  tri_blk > 0 declares B the local column slice of a lower-triangular matrix
// in a block-cyclic distribution (see CoreArgs): its structurally-zero leading rows are skipped per column tile.
static int dgemm_tn_sub_ws(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                           int64_t I, int64_t J, int64_t K, int upper_only, int tri_blk, int tri_world, int tri_rank,
                           void* stream) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    GPX_REQUIRE(I >= 0 && J >= 0 && K >= 0, GPX_EINVAL, "negative size");
    if (I == 0 || J == 0 || K == 0) return GPX_OK;
    GPX_REQUIRE(A && B && C, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE((I + WS_BM - 1) / WS_BM <= 65535, GPX_ESIZE, "I too large for one launch");
    int rc;
    if ((rc = check_operand(A, lda, "A"))) return rc;
    if ((rc = check_operand(B, ldb, "B"))) return rc;
    if ((rc = check_operand(C, ldc, "C"))) return rc;
    GPX_REQUIRE(lda >= (I + WS_BM - 1) / WS_BM * WS_BM && ldb >= (J + BN - 1) / BN * BN, GPX_EALIGN,
                "padded variant needs leading dimensions that cover whole 128-wide tiles");
    GPX_REQUIRE(tri_blk == 0 || (tri_blk % BN == 0 && tri_world >= 1 && tri_rank >= 0 && tri_rank < tri_world), GPX_EINVAL,
                "block-cyclic description: blk must be a multiple of 128, 0 <= rank < world");
    CoreArgs a;
    a.A = A;
    a.B = B;
    a.Ap = a.Bp = nullptr;
    a.out = C;
    a.lda = lda;
    a.ldb = ldb;
    a.ldo = ldc;
    a.I = I;
    a.J = J;
    a.K = (int)K;
    a.prows = 0;
    a.tiles_per_cta = 1;
    a.upper_only = upper_only;
    a.ldo_splits = 0;
    a.tri_blk = tri_blk;
    a.tri_world = tri_world;
    a.tri_rank = tri_rank;
    dim3 grid((unsigned)((J + BN - 1) / BN), (unsigned)((I + WS_BM - 1) / WS_BM));
    TmaMaps maps;
    memset(&maps, 0, sizeof(maps));
    if (encode_tiled() && make_map(&maps.a_main, A, lda, K, WS_BK) == GPX_OK && make_map(&maps.b_main, B, ldb, K, WS_BK) == GPX_OK) {
        if ((rc = gpx_ensure_smem(h, (const void*)sub_ws_kernel<true>, SUBWS_SMEM_BYTES, "sub_ws"))) return rc;
        sub_ws_kernel<true><<<grid, 256, SUBWS_SMEM_BYTES, (cudaStream_t)stream>>>(a, maps);
    } else {
        if ((rc = gpx_ensure_smem(h, (const void*)sub_ws_kernel<false>, SUBWS_SMEM_BYTES, "sub_ws"))) return rc;
        sub_ws_kernel<false><<<grid, 256, SUBWS_SMEM_BYTES, (cudaStream_t)stream>>>(a, maps);
    }
    return gpx_check_launch("gpx_dgemm_tn_sub_padded");
}

extern "C" int gpx_dgemm_tn_sub_padded(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                                       int64_t ldc, int64_t I, int64_t J, int64_t K, int upper_only, void* stream) {
    return dgemm_tn_sub_ws(h, A, lda, B, ldb, C, ldc, I, J, K, upper_only, 0, 0, 0, stream);
}

extern "C" int gpx_dgemm_tn_sub_lower(gpx_handle h, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                                      int64_t ldc, int64_t I, int64_t J, int64_t K, int blk, int world, int rank, void* stream) {
    GPX_REQUIRE(blk > 0, GPX_EINVAL, "blk must be positive");
    return dgemm_tn_sub_ws(h, A, lda, B, ldb, C, ldc, I, J, K, 0, blk, world, rank, stream);
}

// ---------------------------------------------------------------------------------------------
// K5 + K7: IVAR scores of every candidate and their arg-min.  The finalisation (sum the M-splits, apply the
// pinv null-direction rule, |base - reduction|) and the first level of the arg-min share one kernel; the last block
// to finish reduces the per-block winners (np.argmin order: lowest index wins ties).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ivar_finalize_argmin_kernel(const double* __restrict__ partial, int nsplit, int64_t ldp,
                                                                    const double* __restrict__ varC,
                                                                    const double* __restrict__ sumVarM, int64_t M, int64_t C,
                                                                    double noise, double zero_tol,
                                                                    const uint8_t* __restrict__ mask, double* __restrict__ score,
                                                                    double* red_val, int64_t* red_idx, unsigned int* counter,
                                                                    double* best, int64_t* idx) {
    __shared__ double sv[8];
    __shared__ int64_t si[8];
    __shared__ bool last;
    const double base = sumVarM[0] / (double)M;            // (1/nMC) sum varMC   experimentalDesign.py:109
    double bv = 0.0;
    int64_t bi = -1;
    for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < C; c += (int64_t)gridDim.x * 256) {
        double r = 0.0;
        for (int s = 0; s < nsplit; ++s) r += partial[(int64_t)s * ldp + c];
        const double den = varC[c] + noise;
        const double red = (den <= zero_tol) ? 0.0 : (r / den) / (double)M;
        const double sc = fabs(base - red);                // np.abs(cost)        experimentalDesign.py:117
        score[c] = sc;
        if (!(mask && mask[c]) && gpx_better(sc, c, bv, bi, true)) {
            bv = sc;
            bi = c;
        }
    }
    gpx_warp_argreduce(bv, bi, true);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        sv[warp] = bv;
        si[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? sv[lane] : 0.0;
        bi = lane < 8 ? si[lane] : -1;
        gpx_warp_argreduce(bv, bi, true);
        if (lane == 0) {
            red_val[blockIdx.x] = bv;
            red_idx[blockIdx.x] = bi;
            __threadfence();
            last = (atomicAdd(counter, 1u) == gridDim.x - 1);
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
        if (gpx_better(ov, oi, bv, bi, true)) {
            bv = ov;
            bi = oi;
        }
    }
    gpx_warp_argreduce(bv, bi, true);
    if (lane == 0) {
        sv[warp] = bv;
        si[warp] = bi;
    }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? sv[lane] : 0.0;
        bi = lane < 8 ? si[lane] : -1;
        gpx_warp_argreduce(bv, bi, true);
        if (lane == 0) {
            best[0] = bv;
            idx[0] = bi;
            *counter = 0u;
        }
    }
}

static int ivar_finalize_argmin(gpx_handle h, const double* partial, int nsplit, int64_t ldp, const double* varC, int64_t M,
                                int64_t C, double noise, double zero_tol, const uint8_t* mask, double* score_out, double* best,
                                int64_t* idx, cudaStream_t st) {
    int64_t blocks = (C + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    // slots [0, 1024) and ticket 0 of the handle scratch, like gpx_argreduce (never concurrent on one handle)
    ivar_finalize_argmin_kernel<<<(unsigned)blocks, 256, 0, st>>>(partial, nsplit, ldp, varC, h->scal, M, C, noise, zero_tol,
                                                                 mask, score_out, h->red_val, h->red_idx, h->red_counter, best,
                                                                 idx);
    return gpx_check_launch("gpx_score_ivar finalize");
}

// ring / operand movement of the hot kernel: 0 = 32-row chunks x 3 stages, per-row bulk copies; 1 = same ring, one 2-D
// tensor-map load per operand chunk; 2 = 24-row chunks x 4 stages, 2 ahead, tensor-map loads.
// Default GPX_DEFAULT_IVAR_RING, or the GPX_IVAR_RING environment variable.
extern "C" int gpx_set_ivar_ring(gpx_handle h, int ring) {
    GPX_REQUIRE(h != nullptr && ring >= 0 && ring <= 2, GPX_EINVAL, "ring must be 0, 1 or 2");
    h->ivar_ring = ring;
    return GPX_OK;
}

extern "C" int gpx_set_ivar_core(gpx_handle h, int core) {
    GPX_REQUIRE(h != nullptr && (core == GPX_CORE_DMMA || core == GPX_CORE_I8), GPX_EINVAL,
                "core must be GPX_CORE_DMMA or GPX_CORE_I8");
    h->ivar_core = core;
    return GPX_OK;
}

extern "C" int64_t gpx_ivar_scratch_bytes(gpx_handle h, int64_t M, int64_t C, int64_t n_max) {
    if (!h || M < 0 || C < 0 || n_max < 0) return 0;
    int64_t ldk, sm, sc;
    return i8_layout(M, C, n_max, &ldk, &sm, &sc);
}

extern "C" int gpx_set_ivar_scratch(gpx_handle h, void* scratch, int64_t bytes) {
    GPX_REQUIRE(h != nullptr && bytes >= 0 && (scratch != nullptr || bytes == 0), GPX_EINVAL, "bad scratch");
    h->i8_scratch = scratch;
    h->i8_scratch_bytes = bytes;
    return GPX_OK;
}

extern "C" int64_t gpx_score_ivar_workspace(gpx_handle h, int64_t M, int64_t C) {
    if (!h || M < 0 || C < 0) return 0;
    const int64_t ldp = (C + 1) & ~(int64_t)1;
    return (int64_t)gpx_ivar_splits(h, M, C) * ldp;
}

extern "C" int gpx_score_ivar(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* varM,
                              const double* Ma_rows, int64_t M, const double* Wc, int64_t ldc, const double* varC,
                              const double* Cb_rows, int64_t C, int64_t n, double noise, double zero_tol, const uint8_t* mask,
                              double* workspace, double* score_out, double* best, int64_t* idx, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(M >= 1 && C >= 1 && n >= 0, GPX_EINVAL, "bad sizes");
    GPX_REQUIRE(varM && Ma_rows && varC && Cb_rows && workspace && score_out && best && idx, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE(n == 0 || (Wm && Wc), GPX_EINVAL, "W is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = gpx_sum_impl(h, varM, M, h->scal, st);
    if (rc) return rc;
    const int64_t ldp = (C + 1) & ~(int64_t)1;
    int nsplit = 1;
    rc = gpx_launch_core_ivar(h, prologue, Wm, ldm, Ma_rows, M, Wc, ldc, Cb_rows, C, n, workspace, ldp, &nsplit, st);
    if (rc) return rc;
    return ivar_finalize_argmin(h, workspace, nsplit, ldp, varC, M, C, noise, zero_tol, mask, score_out, best, idx, st);
}

// IVAR scores from per-segment column sums of squares (resident-covariance mode): same finalisation + arg-min
extern "C" int gpx_score_ivar_partials(gpx_handle h, const double* partial, int nseg, int64_t ldp, const double* varM, int64_t M,
                                       const double* varC, int64_t C, double noise, double zero_tol, const uint8_t* mask,
                                       double* score_out, double* best, int64_t* idx, void* stream) {
    GPX_REQUIRE(h && partial && varM && varC && score_out && best && idx && nseg >= 1 && M >= 1 && C >= 1, GPX_EINVAL,
                "bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = gpx_sum_impl(h, varM, M, h->scal, st);
    if (rc) return rc;
    return ivar_finalize_argmin(h, partial, nseg, ldp, varC, M, C, noise, zero_tol, mask, score_out, best, idx, st);
}

// cov[m,c] = k(m,c) - sum_{i<n} Wm[i,m] Wc[i,c] for a GIVEN design (DMMA contraction with the Gram prologue, stored)
extern "C" int gpx_cov_from_factors(gpx_handle h, int prologue, const double* Wm, int64_t ldm, const double* Ma_rows, int64_t M,
                                    const double* Wc, int64_t ldc, const double* Cb_rows, int64_t C, int64_t n, double* cov,
                                    int64_t ldcov, void* stream) {
    GPX_NEED_KERNEL(h);
    GPX_REQUIRE(M >= 1 && C >= 1 && n >= 0 && cov && Ma_rows && Cb_rows, GPX_EINVAL, "bad arguments");
    GPX_REQUIRE((M + 63) / 64 <= 65535, GPX_ESIZE, "M too large for one launch");
    return gpx_launch_core_store(h, prologue, Wm, ldm, Ma_rows, M, Wc, ldc, Cb_rows, C, n, cov, ldcov, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Yard-sticks for bench.py: raw DMMA and DFMA issue rates (no memory traffic)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bench_dmma_kernel(int64_t iters, double* sink) {
    double c[16][2];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i][0] = c[i][1] = 0.0;
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
    for (int64_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) dmma(c[i][0], c[i][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i][0] + c[i][1];
    if (s == 123.456) sink[0] = s;
}

__global__ void __launch_bounds__(256) bench_dfma_kernel(int64_t iters, double* sink) {
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) c[i] = i;
    const double a = 1.0 + threadIdx.x * 1e-9, b = 1e-9;
    for (int64_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) c[i] = fma(c[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += c[i];
    if (s == 123.456) sink[0] = s;
}

// each launch: sm_count*4 CTAs of 8 warps; flops = ctas*8 warps*iters*16 DMMA*512  (DFMA: ctas*256 thr*iters*16*2)
extern "C" int gpx_bench_dmma(gpx_handle h, int64_t iters, double* sink, void* stream) {
    GPX_REQUIRE(h && sink && iters > 0, GPX_EINVAL, "bad arguments");
    bench_dmma_kernel<<<h->sm_count * 4, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    return gpx_check_launch("gpx_bench_dmma");
}
extern "C" int gpx_bench_dfma(gpx_handle h, int64_t iters, double* sink, void* stream) {
    GPX_REQUIRE(h && sink && iters > 0, GPX_EINVAL, "bad arguments");
    bench_dfma_kernel<<<h->sm_count * 4, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    return gpx_check_launch("gpx_bench_dfma");
}
