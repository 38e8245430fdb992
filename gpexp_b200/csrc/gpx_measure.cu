// Closed-form IVAR over a box or Gaussian measure for squared-exponential and Mehler kernels: the measure's constants, the
// kernel products Phi(x, y) = int k(t, x) k(t, y) dmu(t), the Z-row append, the Psi-row forward substitution and the
// scoring pass.  The Monte-Carlo contraction of the other IVAR path is not used: every greedy step here is append-only or
// rank-1 and moves O(n C) doubles.
#include <float.h>
#include <math.h>
#include <string.h>

#include "gpx_common.cuh"

// ---------------------------------------------------------------------------------------------
// Per-dimension factor of the box measure.  With u = (lo - m) / cl, v = (hi - m) / cl (u < v):
//     I(m) = J(u, v) / (v - u),   J(u, v) = int_u^v e^{-t^2} dt = e^E F
// E <= 0 joins the exponent sum of Phi, so that a far tail costs one exp and no product of underflowing factors.
//   narrow    (v - u <= 1 and |c| (v - u) <= 1, c = (u + v) / 2): J = e^{-c^2} int_{|s| <= h} e^{-(2c + s) s} ds by 10-point
//             Gauss-Legendre, h = (v - u) / 2.  |(2c + s) s| <= 5/4 there, so the rule's error is below 1e-16 relative;
//             this is where both erf and erfc differences cancel (cl much longer than the box).
//   straddle  (u <= 0 <= v): sqrt(pi)/2 (erf(v) + erf(-u)), two terms of one sign.
//   one side  a = min(|u|, |v|), b = max(|u|, |v|) (J(u, v) = J(-v, -u)):
//             a < 1/2: sqrt(pi)/2 (erf(b) - erf(a)); here b - a > 1 (else "narrow"), so erf(b) >= 2.2 (erf(b) - erf(a)).
//             a >= 1/2: sqrt(pi)/2 e^{-a^2} (erfcx(a) - e^{-(b - a)(b + a)} erfcx(b)), the erfc difference without its
//             tails; (b - a)(b + a) > 2 outside "narrow", so the bracket keeps more than 1 - e^-2 of erfcx(a).
// MEAN returns J / (v - u) instead, for a width that may be 0 (Mehler with t = 0): "narrow" then gives the Gauss-Legendre
// mean itself, never 0 / 0, and every other branch has width > 0.
// ---------------------------------------------------------------------------------------------
template <bool MEAN>
__device__ __forceinline__ double box_tail_j(double u, double v, double width, double& E) {
    const double SQRTPI_2 = 0.88622692545275801365;
    const double c = 0.5 * (u + v);
    if (width <= 1.0 && fabs(c) * width <= 1.0) {
        const double x[5] = {0x1.30e507891e27ap-3, 0x1.bbcc009016adcp-2, 0x1.5bdb9228de198p-1, 0x1.bae995e9cb2f3p-1,
                             0x1.f2a3e062af2d8p-1};
        const double w[5] = {0x1.2e9de7014d6eep-2, 0x1.13baa7a559c01p-2, 0x1.c0b059d00bc30p-3, 0x1.32138c878efdep-3,
                             0x1.1115f8b62dc1fp-4};
        const double h = 0.5 * width;
        double sum = 0.0;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const double s = h * x[k];
            sum = fma(w[k], exp(-(2.0 * c + s) * s) + exp((2.0 * c - s) * s), sum);
        }
        E = -c * c;
        return MEAN ? 0.5 * sum : h * sum;
    }
    E = 0.0;
    double j;
    const double a = fmin(fabs(u), fabs(v)), b = fmax(fabs(u), fabs(v));
    if (u <= 0.0 && v >= 0.0) {
        j = SQRTPI_2 * (erf(v) + erf(-u));
    } else if (a < 0.5) {
        j = SQRTPI_2 * (erf(b) - erf(a));
    } else {
        E = -a * a;
        j = SQRTPI_2 * (erfcx(a) - exp(-width * (a + b)) * erfcx(b));
    }
    return MEAN ? j / width : j;
}

// one dimension of Phi(x, y): exponent sum S and bounded factor F.  Mehler, with t = t_q, r = 1 - t^2:
//     k(z, x) k(z, y) = r^-1 exp(m^2 - t^2 (x - y)^2 / (4 r)) exp(-(t z - m)^2 / r)
// so the box factor is J((t lo - m) / sqrt(r), (t hi - m) / sqrt(r)) / width with m^2 joining the exponent, and the Gaussian
// one is the closed-form quadratic g2 m^2 + g1 m + g0 (MParams), whose arrangement avoids cancelling m^2 against
// (m - t mean)^2 / g.
template <int FAM, int KIND>
__device__ __forceinline__ void phi_dim(const MParams& mp, int q, double x, double y, double& S, double& F) {
    static_assert(FAM == GPX_SE || FAM == GPX_MEHLER, "the closed-form measure is for SE and Mehler kernels");
    const double df = x - y;
    S = fma(-df * df, mp.a4[q], S);
    const double m = 0.5 * (x + y);
    if (FAM == GPX_SE && KIND == GPX_MEASURE_GAUSS) {
        const double t = (m - mp.p0[q]) * mp.rs[q];
        S = fma(-t, t, S);
    } else if (FAM == GPX_SE) {
        double E;
        F *= box_tail_j<false>((mp.p0[q] - m) * mp.rs[q], (mp.p1[q] - m) * mp.rs[q], mp.width[q], E);
        S += E;
    } else if (KIND == GPX_MEASURE_GAUSS) {
        S += fma(fma(mp.g2[q], m, mp.g1[q]), m, mp.g0[q]);
    } else {
        double E;
        F *= box_tail_j<true>((mp.p0[q] - m) * mp.rs[q], (mp.p1[q] - m) * mp.rs[q], mp.width[q], E);
        S += fma(m, m, E);
    }
}

// one exp for the whole exponent; a value below 2^-1022 is flushed to 0, as gpx_gram's table exp flushes k
__device__ __forceinline__ double phi_finish(const MParams& mp, double S, double F) {
    const double v = mp.pref * F * exp(S);
    return fabs(v) < DBL_MIN ? 0.0 : v;
}

template <int FAM, int KIND>
__device__ __forceinline__ double phi_eval(const MParams& mp, const double* __restrict__ X, int64_t ldx, int64_t i,
                                           const double* __restrict__ Y, int64_t ldy, int64_t j) {
    double S = 0.0, F = 1.0;
#pragma unroll 1
    for (int q = 0; q < mp.d; ++q) phi_dim<FAM, KIND>(mp, q, X[q * ldx + i], Y[q * ldy + j], S, F);
    return phi_finish(mp, S, F);
}

#define GPX_DISPATCH_MEASURE(kind, ...)                \
    do {                                               \
        if ((kind) == GPX_MEASURE_BOX) {               \
            constexpr int KIND = GPX_MEASURE_BOX;      \
            __VA_ARGS__;                               \
        } else {                                       \
            constexpr int KIND = GPX_MEASURE_GAUSS;    \
            __VA_ARGS__;                               \
        }                                              \
    } while (0)

// the kernel families gpx_set_measure accepts (it rejects every other one)
#define GPX_DISPATCH_MEASURE_FAMILY(fam, kind, ...)                \
    do {                                                           \
        if ((fam) == GPX_MEHLER) {                                 \
            constexpr int FAM = GPX_MEHLER;                        \
            GPX_DISPATCH_MEASURE(kind, __VA_ARGS__);               \
        } else {                                                   \
            constexpr int FAM = GPX_SE;                            \
            GPX_DISPATCH_MEASURE(kind, __VA_ARGS__);               \
        }                                                          \
    } while (0)

#define GPX_NEED_MEASURE(h)                                                                                 \
    do {                                                                                                    \
        GPX_NEED_KERNEL(h);                                                                                 \
        GPX_REQUIRE((h)->has_measure, GPX_ENOKERNEL, "gpx_set_measure has not been called for this kernel"); \
    } while (0)

// int_lo^hi exp(c x^2) dx = e^K G for the box prior of a Mehler kernel (c = t / (1 + t), an erf for c < 0 and a
// Dawson / erfi form for c > 0), as one composite 10-point Gauss-Legendre rule of the positive integrand
// e^{c x^2 - K} = e^{c d (d + 2 xr)}, d = x - xr, K = c xr^2 its largest exponent on [lo, hi] (xr = +-max|x| for c > 0,
// the point nearest 0 for c < 0).  Nodes are placed in d, so that their rounding is relative to the distance from the
// peak, not to |x|.  Only the part of [lo, hi] where the exponent exceeds -50 is integrated: the rest adds less than
// e^-50 relative.  Panels of half-width <= 1/2 min(|c|^-1/2, 1 / (|c| max |x|)) keep the exponent's slope within 1 and
// its curvature within 1/4 per panel, where the rule is exact to rounding; the panel sums are added with Neumaier
// compensation.  NaN when the panel count is not finite and below 2^20 (an overflowing box).
static double mehler_box_integral(double c, double lo, double hi, double& K) {
    static const double X[5] = {0x1.30e507891e27ap-3, 0x1.bbcc009016adcp-2, 0x1.5bdb9228de198p-1, 0x1.bae995e9cb2f3p-1,
                                0x1.f2a3e062af2d8p-1};
    static const double W[5] = {0x1.2e9de7014d6eep-2, 0x1.13baa7a559c01p-2, 0x1.c0b059d00bc30p-3, 0x1.32138c878efdep-3,
                                0x1.1115f8b62dc1fp-4};
    const double T = 50.0;
    K = 0.0;
    if (c == 0.0) return hi - lo;
    double xk, xr[2], a[2], b[2];
    int pieces = 0;
    if (c > 0.0) {
        xk = fmax(fabs(lo), fabs(hi));
        const double xt = sqrt(fmax(0.0, xk * xk - T / c));
        if (lo < -xt) {
            xr[pieces] = -xk;
            a[pieces] = lo;
            b[pieces++] = fmin(hi, -xt);
        }
        if (hi > xt) {
            xr[pieces] = xk;
            a[pieces] = fmax(lo, xt);
            b[pieces++] = hi;
        }
    } else {
        xk = lo > 0.0 ? lo : (hi < 0.0 ? hi : 0.0);
        const double xt = sqrt(xk * xk - T / c);
        xr[0] = xk;
        a[0] = fmax(lo, -xt);
        b[0] = fmin(hi, xt);
        pieces = 1;
    }
    // K = c xr^2 rounded, and its rounding error (exact products by fma) folded into G: e^K is then off by at most the
    // rounding of exp, not by |K| ulp
    const double cx = c * xk;
    K = cx * xk;
    const double Klo = fma(fma(c, xk, -cx), xk, fma(cx, xk, -K));
    double sum = 0.0, comp = 0.0;
    for (int p = 0; p < pieces; ++p) {
        const double xm = fmax(fabs(a[p]), fabs(b[p]));
        const double h = 0.5 * fmin(1.0 / sqrt(fabs(c)), 1.0 / (fabs(c) * xm));
        const double panels = ceil((b[p] - a[p]) / (2.0 * h));
        if (!(panels <= 1048576.0)) return NAN;
        const int np = panels < 1.0 ? 1 : (int)panels;
        const double da = a[p] - xr[p], hp = (b[p] - a[p]) / (2.0 * np), x2 = 2.0 * xr[p];
        for (int k = 0; k < np; ++k) {
            const double mid = da + (2 * k + 1) * hp;
            double panel = 0.0;
            for (int i = 0; i < 5; ++i) {
                const double d0 = mid - hp * X[i], d1 = mid + hp * X[i];
                panel += W[i] * (exp(c * (d0 * (d0 + x2))) + exp(c * (d1 * (d1 + x2))));
            }
            const double term = hp * panel, t = sum + term;
            comp += fabs(sum) >= fabs(term) ? (sum - t) + term : (term - t) + sum;
            sum = t;
        }
    }
    return (sum + comp) * exp(Klo);
}

extern "C" int gpx_set_measure(gpx_handle h, int kind, int d, const double* p0, const double* p1) {
    GPX_NEED_KERNEL(h);
    const int fam = h->kp.family;
    GPX_REQUIRE(fam == GPX_SE || fam == GPX_MEHLER, GPX_EINVAL,
                "a closed-form measure needs a squared-exponential or Mehler kernel");
    GPX_REQUIRE(kind == GPX_MEASURE_BOX || kind == GPX_MEASURE_GAUSS, GPX_EINVAL, "unknown measure kind");
    GPX_REQUIRE(d == h->kp.d, GPX_EINVAL, "measure dimension differs from the kernel's");
    GPX_REQUIRE(p0 != nullptr && p1 != nullptr, GPX_EINVAL, "NULL parameter array");
    MParams mp;
    memset(&mp, 0, sizeof(mp));
    mp.kind = kind;
    mp.d = d;
    const double s = h->kp.signal;
    double pref = fam == GPX_SE ? s * s : 1.0;
    double prior = fam == GPX_SE ? s : 1.0;
    for (int q = 0; q < d; ++q) {
        GPX_REQUIRE(isfinite(p0[q]) && isfinite(p1[q]), GPX_EINVAL, "measure parameters must be finite");
        if (kind == GPX_MEASURE_BOX) {
            GPX_REQUIRE(p0[q] < p1[q], GPX_EINVAL, "box needs lower < upper in every dimension");
        } else {
            GPX_REQUIRE(p1[q] > 0.0, GPX_EINVAL, "Gaussian measure needs std > 0 in every dimension");
        }
        if (fam == GPX_MEHLER) {
            // t = kp.b / 2 exactly; r = 1 - t^2 as (1 - t)(1 + t), within 2 ulp also for t near 1
            const double t = 0.5 * h->kp.b[q], r = (1.0 - t) * (1.0 + t);
            mp.a4[q] = 0.25 * t * t / r;
            if (kind == GPX_MEASURE_BOX) {
                const double len = p1[q] - p0[q];
                GPX_REQUIRE(isfinite(len), GPX_EINVAL, "box width overflows");
                mp.rs[q] = 1.0 / sqrt(r);
                mp.p0[q] = t >= 0.0 ? t * p0[q] : t * p1[q];
                mp.p1[q] = t >= 0.0 ? t * p1[q] : t * p0[q];
                mp.width[q] = fabs(t) * len * mp.rs[q];
                pref /= r;
                // s_q = r^-1/2 / (hi - lo) int_lo^hi e^{c x^2} dx
                double K;
                const double G = mehler_box_integral(t / (1.0 + t), p0[q], p1[q], K);
                prior *= G / (len * sqrt(r)) * exp(K);
            } else {
                const double sd2 = p1[q] * p1[q], mu = p0[q];
                const double g = fma(2.0 * t * t, sd2, r);
                mp.g2[q] = t * t * fma(2.0, sd2, -1.0) / g;
                mp.g1[q] = 2.0 * t * mu / g;
                mp.g0[q] = -(t * t) * (mu * mu) / g;
                pref /= sqrt(r * g);
                // s_q = r^-1/2 (1 - 2 c std^2)^-1/2 exp(c mean^2 / (1 - 2 c std^2)), c = t / (1 + t), written through
                // num = (1 + t)(1 - 2 c std^2) = 1 + t - 2 t std^2
                const double num = fma(-2.0 * t, sd2, 1.0 + t);
                GPX_REQUIRE(num > 0.0, GPX_EINVAL,
                            "Gaussian measure too wide for the Mehler kernel: int k(x, x) dmu is infinite unless "
                            "std^2 < (1 + t) / (2 t) in every dimension");
                prior *= exp(t * mu * mu / num) / sqrt((1.0 - t) * num);
            }
            continue;
        }
        const double a = h->kp.a[q];  // cl_q^-2
        mp.a4[q] = 0.25 * a;
        if (kind == GPX_MEASURE_BOX) {
            mp.rs[q] = sqrt(a);
            mp.p0[q] = p0[q];
            mp.p1[q] = p1[q];
            mp.width[q] = (p1[q] - p0[q]) * mp.rs[q];
            GPX_REQUIRE(isfinite(mp.width[q]), GPX_EINVAL, "box width overflows");
            pref /= mp.width[q];
        } else {
            const double g = fma(2.0 * p1[q] * p1[q], a, 1.0);  // 1 + 2 std^2 / cl^2
            GPX_REQUIRE(isfinite(g), GPX_EINVAL, "Gaussian std overflows");
            mp.rs[q] = sqrt(a / g);                              // 1 / sqrt(cl^2 + 2 std^2)
            mp.p0[q] = p0[q];
            mp.p1[q] = p1[q];
            pref /= sqrt(g);
        }
    }
    GPX_REQUIRE(isfinite(pref) && isfinite(prior) && prior > 0.0, GPX_EINVAL,
                "int k(x, x) dmu or the Phi prefactor is not a finite positive double for this kernel and measure");
    mp.pref = pref;
    mp.prior = prior;
    h->mp = mp;
    h->has_measure = true;
    return GPX_OK;
}

// ---------------------------------------------------------------------------------------------
// Phi(X_i, Y_j) cross block and diagonal.  Per element: d evaluations of erf / erfcx (box) or one FMA chain (Gaussian)
// and one exp; the coordinates are re-read from L1 for every row rather than kept in a per-dimension register array.
// ---------------------------------------------------------------------------------------------
template <int FAM, int KIND>
__global__ void __launch_bounds__(256) phi_gram_kernel(const __grid_constant__ MParams mp, const double* __restrict__ X,
                                                       int64_t nx, int64_t ldx, const double* __restrict__ Y, int64_t ny,
                                                       int64_t ldy, double* __restrict__ out, int64_t ld) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= ny) return;
    for (int64_t i = blockIdx.y; i < nx; i += gridDim.y) out[i * ld + j] = phi_eval<FAM, KIND>(mp, X, ldx, i, Y, ldy, j);
}

extern "C" int gpx_phi_gram(gpx_handle h, const double* X, int64_t nx, int64_t ldx, const double* Y, int64_t ny,
                            int64_t ldy, double* out, int64_t ld, void* stream) {
    GPX_NEED_MEASURE(h);
    GPX_REQUIRE(nx >= 0 && ny >= 0 && ld >= ny, GPX_EINVAL, "bad sizes");
    if (nx == 0 || ny == 0) return GPX_OK;
    GPX_REQUIRE(X && Y && out, GPX_EINVAL, "NULL pointer");
    const dim3 grid((unsigned)((ny + 255) / 256), (unsigned)(nx < 65535 ? nx : 65535));
    GPX_DISPATCH_MEASURE_FAMILY(h->kp.family, h->mp.kind, (phi_gram_kernel<FAM, KIND><<<grid, 256, 0, (cudaStream_t)stream>>>(h->mp, X, nx, ldx, Y, ny,
                                                                                                     ldy, out, ld)));
    return gpx_check_launch("gpx_phi_gram");
}

template <int FAM, int KIND>
__global__ void __launch_bounds__(256) phi_diag_kernel(const __grid_constant__ MParams mp, const double* __restrict__ X,
                                                       int64_t n, int64_t ldx, double* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j < n) out[j] = phi_eval<FAM, KIND>(mp, X, ldx, j, X, ldx, j);
}

extern "C" int gpx_phi_diag(gpx_handle h, const double* X, int64_t n, int64_t ldx, double* out, void* stream) {
    GPX_NEED_MEASURE(h);
    GPX_REQUIRE(n >= 0, GPX_EINVAL, "negative size");
    if (n == 0) return GPX_OK;
    GPX_REQUIRE(X && out, GPX_EINVAL, "NULL pointer");
    GPX_DISPATCH_MEASURE_FAMILY(h->kp.family, h->mp.kind, (phi_diag_kernel<FAM, KIND><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
                                          h->mp, X, n, ldx, out)));
    return gpx_check_launch("gpx_phi_diag");
}

// ---------------------------------------------------------------------------------------------
// Z-row append: Z[n, j] = (Phi(x_p, Y_j) - sum_{i<n} rec.col[i] Z[i, j]) / sqrt(rec[2]), the W-row recurrence of
// gpx_append_row with Phi as the source term and no running variance.  Two adjacent columns per thread (16-byte
// streaming loads), the pivot's W column in shared memory.  Reads 8 n ncols bytes.  A non-positive pivot appends a zero
// row, as gpx_append_row does.
// ---------------------------------------------------------------------------------------------
template <int FAM, int KIND>
__global__ void __launch_bounds__(128) phi_append_kernel(const __grid_constant__ MParams mp, const double* __restrict__ rec,
                                                         const double* __restrict__ Y, int64_t ncols, int64_t ldy,
                                                         double* __restrict__ Z, int64_t ldz, int n) {
    extern __shared__ double sl[];
    for (int i = threadIdx.x; i < n; i += 128) sl[i] = rec[GPX_PIVOT_HDR + i];
    const int64_t j = ((int64_t)blockIdx.x * 128 + threadIdx.x) * 2;
    const bool active = j < ncols, two = j + 1 < ncols;
    double s0 = 0.0, s1 = 0.0;
    // the pivot's coordinates are rec[3 .. 3+d), read as a one-column coordinate array
    if (active) s0 = phi_eval<FAM, KIND>(mp, rec + 3, 1, 0, Y, ldy, j);
    if (two) s1 = phi_eval<FAM, KIND>(mp, rec + 3, 1, 0, Y, ldy, j + 1);
    const double lnn = rec[2] > 0.0 ? sqrt(rec[2]) : INFINITY;
    __syncthreads();
    if (!active) return;
    double a0 = 0.0, a1 = 0.0;
    const double* zp = Z + j;
#pragma unroll 8
    for (int i = 0; i < n; ++i) {
        const double2 z = __ldcs(reinterpret_cast<const double2*>(zp + (int64_t)i * ldz));
        a0 = fma(sl[i], z.x, a0);
        a1 = fma(sl[i], z.y, a1);
    }
    double* dst = Z + (int64_t)n * ldz + j;
    dst[0] = (s0 - a0) / lnn;
    dst[1] = two ? (s1 - a1) / lnn : 0.0;
}

extern "C" int gpx_phi_append_row(gpx_handle h, const double* rec, const double* Y, int64_t ncols, int64_t ldy, double* Z,
                                  int64_t ldz, int64_t n, void* stream) {
    GPX_NEED_MEASURE(h);
    GPX_REQUIRE(ncols >= 0 && n >= 0, GPX_EINVAL, "negative size");
    if (ncols == 0) return GPX_OK;
    GPX_REQUIRE(rec && Y && Z, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE((ldz % 2) == 0 && ldz >= ncols + (ncols & 1) && gpx_aligned16(Z), GPX_EALIGN,
                "Z must be 16-byte aligned with an even leading dimension covering an even column count");
    const size_t smem = (size_t)(n > 0 ? n : 1) * sizeof(double);
    GPX_REQUIRE(smem <= 200 * 1024, GPX_ESIZE, "design size exceeds the shared-memory column buffer (25600)");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((ncols + 255) / 256);
    GPX_DISPATCH_MEASURE_FAMILY(h->kp.family, h->mp.kind, {
        if (smem > 48 * 1024) {
            const int rc = gpx_ensure_smem(h, (const void*)phi_append_kernel<FAM, KIND>, 200 * 1024, "phi_append_row");
            if (rc) return rc;
        }
        phi_append_kernel<FAM, KIND><<<grid, 128, smem, st>>>(h->mp, rec, Y, ncols, ldy, Z, ldz, (int)n);
    });
    return gpx_check_launch("gpx_phi_append_row");
}

// ---------------------------------------------------------------------------------------------
// Psi row n (one block):  U^T x = b,  b_k = Z[n, cols[k] - offset] (k <= n),  Psi[n, k] = Psi[k, n] = x_k.
// Blocked by 32 columns: warp 0 solves the 32 x 32 diagonal triangle in registers (shuffles, no barrier), then every
// thread subtracts the block's contribution from the rest of b.  Two barriers and one dependent global load per 32
// columns.  A non-positive or NaN diagonal entry (the zero row of a dependent pivot) gives x = 0.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) psi_row_kernel(const double* __restrict__ U, int64_t ldu, const double* __restrict__ Z,
                                                      int64_t ldz, const int64_t* __restrict__ cols, int64_t offset, int n,
                                                      double* __restrict__ Psi, int64_t ldpsi) {
    extern __shared__ double b[];
    const int nn = n + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < nn; k += 256) b[k] = Z[(int64_t)n * ldz + (cols[k] - offset)];
    for (int j0 = 0; j0 < nn; j0 += 32) {
        const int nb = nn - j0 < 32 ? nn - j0 : 32;
        __syncthreads();
        if (warp == 0) {
            const bool live = lane < nb;
            const int jl = j0 + lane;
            double ucol[32];
#pragma unroll
            for (int r = 0; r < 32; ++r) ucol[r] = (live && r <= lane) ? U[(int64_t)(j0 + r) * ldu + jl] : 0.0;
            double bl = live ? b[jl] : 0.0;
            double x = 0.0;
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                if (lane == r) x = ucol[r] > 0.0 ? bl / ucol[r] : 0.0;
                const double xr = __shfl_sync(0xffffffffu, x, r);
                if (lane > r) bl = fma(-ucol[r], xr, bl);
            }
            if (live) {
                b[jl] = x;
                Psi[(int64_t)n * ldpsi + jl] = x;
                Psi[(int64_t)jl * ldpsi + n] = x;
            }
        }
        __syncthreads();
        for (int k = j0 + 32 + threadIdx.x; k < nn; k += 256) {
            double acc = b[k];
            for (int r = 0; r < nb; ++r) acc = fma(-U[(int64_t)(j0 + r) * ldu + k], b[j0 + r], acc);
            b[k] = acc;
        }
    }
}

extern "C" int gpx_psi_row(gpx_handle h, const double* U, int64_t ldu, const double* Z, int64_t ldz, const int64_t* cols,
                           int64_t index_offset, int64_t n, double* Psi, int64_t ldpsi, void* stream) {
    GPX_REQUIRE(h != nullptr, GPX_EINVAL, "handle is NULL");
    GPX_REQUIRE(n >= 0 && ldu > n && ldpsi > n, GPX_EINVAL, "bad sizes");
    GPX_REQUIRE(U && Z && cols && Psi, GPX_EINVAL, "NULL pointer");
    const size_t smem = (size_t)(n + 1) * sizeof(double);
    GPX_REQUIRE(smem <= 200 * 1024, GPX_ESIZE, "design size exceeds the shared-memory buffer (25599)");
    if (smem > 48 * 1024) {
        const int rc = gpx_ensure_smem(h, (const void*)psi_row_kernel, 200 * 1024, "psi_row");
        if (rc) return rc;
    }
    psi_row_kernel<<<1, 256, smem, (cudaStream_t)stream>>>(U, ldu, Z, ldz, cols, index_offset, (int)n, Psi, ldpsi);
    return gpx_check_launch("gpx_psi_row");
}

// ---------------------------------------------------------------------------------------------
// Scoring pass, one column per thread, and its arg-min.  UPDATE first brings Y = Psi W up to date with the last append
// (row n-1 of W and Psi):  Y[i, c] += Psi[i, n-1] W[n-1, c] for i < n-1 and Y[n-1, c] = sum_{j<n} Psi[n-1, j] W[j, c].
// Then, from the stored rows,
//     q_c = Phi_cc - 2 sum_i W[i,c] Z[i,c] + sum_i W[i,c] Y[i,c]     (= int cov_D(x, c)^2 dmu)
//     score_c = |s - tr Psi - q_c / (varC_c + noise)|,  reduction 0 where varC_c + noise <= zero_tol (as the MC path)
// Reads 3n doubles per candidate, writes n with UPDATE.  Every block sums the diagonal of Psi in the same order, so
// tr Psi (and the scores) are run-to-run identical.  cost (nullable) receives s - tr Psi, the cost of the design itself.
// ---------------------------------------------------------------------------------------------
template <bool UPDATE>
__global__ void __launch_bounds__(256) ivar_measure_score_kernel(const double* __restrict__ W, const double* __restrict__ Z,
                                                                 double* __restrict__ Y, int64_t ld,
                                                                 const double* __restrict__ phic,
                                                                 const double* __restrict__ varC, int64_t C, int n,
                                                                 const double* __restrict__ Psi, int64_t ldpsi, double prior,
                                                                 double noise, double zero_tol, double* __restrict__ cost,
                                                                 double* __restrict__ score, double* red_val, int64_t* red_idx,
                                                                 unsigned int* counter, double* best, int64_t* idx) {
    extern __shared__ double sp[];
    __shared__ double sv[8];
    __shared__ int64_t si[8];
    __shared__ double s_base;
    __shared__ bool last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (UPDATE)
        for (int i = threadIdx.x; i < n; i += 256) sp[i] = Psi[(int64_t)(n - 1) * ldpsi + i];
    if (warp == 0) {
        double t = 0.0;
        for (int i = lane; i < n; i += 32) t += Psi[(int64_t)i * ldpsi + i];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (lane == 0) {
            s_base = prior - t;
            if (cost && blockIdx.x == 0) cost[0] = s_base;
        }
    }
    __syncthreads();
    const double base = s_base;
    double bv = 0.0;
    int64_t bi = -1;
    for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < C; c += (int64_t)gridDim.x * 256) {
        double wz = 0.0, wy = 0.0;
        if (n > 0) {
            const double* wc = W + c;
            const double* zc = Z + c;
            double* yc = Y + c;
            const double wl = wc[(int64_t)(n - 1) * ld];
            double ynew = 0.0;
#pragma unroll 4
            for (int i = 0; i < n - 1; ++i) {
                const double w = __ldcs(wc + (int64_t)i * ld);
                const double z = __ldcs(zc + (int64_t)i * ld);
                double y;
                if (UPDATE) {
                    y = fma(sp[i], wl, yc[(int64_t)i * ld]);
                    __stcs(yc + (int64_t)i * ld, y);
                    ynew = fma(sp[i], w, ynew);
                } else {
                    y = __ldcs(yc + (int64_t)i * ld);
                }
                wz = fma(w, z, wz);
                wy = fma(w, y, wy);
            }
            double yl;
            if (UPDATE) {
                yl = fma(sp[n - 1], wl, ynew);
                yc[(int64_t)(n - 1) * ld] = yl;
            } else {
                yl = yc[(int64_t)(n - 1) * ld];
            }
            wz = fma(wl, zc[(int64_t)(n - 1) * ld], wz);
            wy = fma(wl, yl, wy);
        }
        const double q = fma(-2.0, wz, phic[c]) + wy;
        const double den = varC[c] + noise;
        const double red = (den <= zero_tol) ? 0.0 : q / den;
        const double sc = fabs(base - red);
        score[c] = sc;
        if (gpx_better(sc, c, bv, bi, true)) {
            bv = sc;
            bi = c;
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

extern "C" int gpx_ivar_measure_score(gpx_handle h, const double* W, const double* Z, double* Y, int64_t ld,
                                      const double* phic, const double* varC, int64_t C, int64_t n, int update,
                                      const double* Psi, int64_t ldpsi, double noise, double zero_tol, double* cost,
                                      double* score_out, double* best, int64_t* idx, void* stream) {
    GPX_NEED_MEASURE(h);
    GPX_REQUIRE(C >= 1 && n >= 0 && ld >= C && (n == 0 || ldpsi >= n), GPX_EINVAL, "bad sizes");
    GPX_REQUIRE(phic && varC && score_out && best && idx, GPX_EINVAL, "NULL pointer");
    GPX_REQUIRE(n == 0 || (W && Z && Y && Psi), GPX_EINVAL, "W, Z, Y or Psi is NULL");
    GPX_REQUIRE(!update || n >= 1, GPX_EINVAL, "update needs an appended row");
    const size_t smem = update ? (size_t)n * sizeof(double) : 0;
    GPX_REQUIRE(smem <= 200 * 1024, GPX_ESIZE, "design size exceeds the shared-memory Psi row (25600)");
    int64_t blocks = (C + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    cudaStream_t st = (cudaStream_t)stream;
    // slots [0, 1024) and ticket 0 of the handle scratch, like gpx_argreduce (never concurrent on one handle)
    if (update) {
        if (smem > 48 * 1024) {
            const int rc = gpx_ensure_smem(h, (const void*)ivar_measure_score_kernel<true>, 200 * 1024, "ivar_measure_score");
            if (rc) return rc;
        }
        ivar_measure_score_kernel<true><<<(unsigned)blocks, 256, smem, st>>>(W, Z, Y, ld, phic, varC, C, (int)n, Psi, ldpsi,
                                                                            h->mp.prior, noise, zero_tol, cost, score_out,
                                                                            h->red_val, h->red_idx, h->red_counter, best, idx);
    } else {
        ivar_measure_score_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(W, Z, Y, ld, phic, varC, C, (int)n, Psi, ldpsi,
                                                                          h->mp.prior, noise, zero_tol, cost, score_out,
                                                                          h->red_val, h->red_idx, h->red_counter, best, idx);
    }
    return gpx_check_launch("gpx_ivar_measure_score");
}
