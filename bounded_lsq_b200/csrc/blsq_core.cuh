// Per-problem mathematics of the bounded trust-region least-squares hot path.
//
// Everything here is written once as __host__ __device__ templates on the
// parameter count N.  The CUDA kernels (blsq_kernels.cu) call these from one
// thread per problem; tests/host_emul compiles the very same header with g++
// so the branch logic can be checked against the oracle without a GPU.  The
// host build is test infrastructure only -- the product never loads it.
//
// Reference being restated (nmayorov/bounded-lsq):
//   bounds.py:24-149        step_size_to_bound, find_active_constraints,
//                           make_strictly_feasible, scaling_vector
//   trust_region.py:11-152  intersect_trust_region, solve_lsq_trust_region
//   trf.py:15-170,238-344   1-D quadratics, reflected/gradient step, the
//                           step selection and ratio test of the TRF loop
//   dogbox.py:9-97,164-251  find_intersection, dogleg_step,
//                           constrained_cauchy_step, dogbox loop body
//
// Arithmetic rules: the file is compiled with -fmad=false (nvcc) /
// -ffp-contract=off (g++), so `a*b+c` is two roundings exactly as NumPy does
// it; fused multiply-adds appear only where fma() is written out (dot
// products and rotations of the dense tail, where the reference itself goes
// through BLAS and has no defined summation order).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define BLSQ_HD __host__ __device__ __forceinline__

#define BLSQ_UNROLL _Pragma("unroll")
#else
#define BLSQ_HD inline
#define BLSQ_UNROLL
#endif

// tools/phase_probe.py builds a variant with -DBLSQ_PHASE_CLOCKS: cycles per
// phase of trf_round_impl, summed over all threads (never in the shipped .so)
#if defined(BLSQ_PHASE_CLOCKS) && defined(__CUDACC__)
static __device__ unsigned long long blsq_phase_acc[32];
#endif
#if defined(BLSQ_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
#define BLSQ_PHASE_BEGIN long long ph_ = clock64()
#define BLSQ_PHASE(k)                                                          \
    do {                                                                       \
        long long c_ = clock64();                                              \
        atomicAdd(&blsq_phase_acc[k], (unsigned long long)(c_ - ph_));         \
        atomicAdd(&blsq_phase_acc[16 + k], 1ull);                              \
        ph_ = clock64();                                                       \
    } while (0)
#else
#define BLSQ_PHASE_BEGIN
#define BLSQ_PHASE(k)
#endif

namespace blsq {

static constexpr double EPS = 2.220446049250313e-16;
static constexpr double SQRT_EPS = 1.4901161193847656e-08;

// status codes kept per problem while a solve is in flight
static constexpr int ST_RUNNING = -1;
// reference raises ValueError from intersect_trust_region
// (trust_region.py:28-35); the host turns these into the same exceptions
static constexpr int ST_ERR_TR_ZERO = -101;      // "`s` is zero."
static constexpr int ST_ERR_TR_OUTSIDE = -102;   // "`x` is not within the trust region."

BLSQ_HD double dinf() { return HUGE_VAL; }
BLSQ_HD double dnan() { return HUGE_VAL - HUGE_VAL; }

// NumPy's maximum/minimum propagate NaN (bounds.py:43, dogbox.py:20-21)
BLSQ_HD double np_max(double a, double b) {
    if (a != a) return a;
    if (b != b) return b;
    return a >= b ? a : b;          // ties keep the first operand, like NumPy
}
BLSQ_HD double np_min(double a, double b) {
    if (a != a) return a;
    if (b != b) return b;
    return a <= b ? a : b;
}
BLSQ_HD int isign(double v) { return (v > 0) - (v < 0); }
BLSQ_HD bool finite_d(double v) { return fabs(v) <= 1.79769313486231570815e+308; }

template <int N>
BLSQ_HD double dot(const double* a, const double* b) {
    double s = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) s = fma(a[i], b[i], s);
    return s;
}
template <int N>
BLSQ_HD double norm2(const double* a) { return sqrt(dot<N>(a, a)); }

// ---------------------------------------------------------------------------
// bounds.py -- every function below is bit-exact with NumPy
// ---------------------------------------------------------------------------

// bounds.py:24-48.  hits may be nullptr.
template <int N>
BLSQ_HD double step_size_to_bound(const double* x, const double* d,
                                  const double* lb, const double* ub,
                                  int* hits) {
    double t[N];
    double tmin = dinf();
    bool has_nan = false;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        if (d[i] != 0) {
            t[i] = np_max((lb[i] - x[i]) / d[i], (ub[i] - x[i]) / d[i]);
        } else {
            t[i] = dinf();
        }
        if (t[i] != t[i]) has_nan = true;
        if (!(tmin < t[i])) tmin = t[i];   // NumPy: ties take the later element
    }
    if (has_nan) tmin = dnan();          // np.min propagates NaN
    if (hits) {
        BLSQ_UNROLL
        for (int i = 0; i < N; i++)
            hits[i] = (t[i] == tmin) ? isign(d[i]) : 0;
    }
    return tmin;
}

// bounds.py:51-76
BLSQ_HD int active_constraint(double x, double lb, double ub, double rtol) {
    double below = x - lb;
    double above = ub - x;
    if (below < above)
        return -(int)(below < rtol * np_max(1.0, fabs(lb)));
    return (int)(above < rtol * np_max(1.0, fabs(ub)));
}

// bounds.py:79-103 (lower rule first, upper rule second, both on the input x)
BLSQ_HD double strictly_feasible(double x, double lb, double ub, double rstep) {
    double y = x;
    if (x <= lb)
        y = (rstep == 0) ? nextafter(lb, ub) : lb + rstep * (1 + fabs(lb));
    if (x >= ub)
        y = (rstep == 0) ? nextafter(ub, lb) : ub - rstep * (1 + fabs(ub));
    return y;
}

// bounds.py:106-149
BLSQ_HD void cl_scaling(double x, double g, double lb, double ub, double& v,
                        double& jv) {
    v = 1.0;
    jv = 0.0;
    if (g < 0 && finite_d(ub)) { v = ub - x; jv = -1.0; }
    if (g > 0 && finite_d(lb)) { v = x - lb; jv = 1.0; }
}

// ---------------------------------------------------------------------------
// trust_region.py
// ---------------------------------------------------------------------------

// trust_region.py:11-44.  Returns 0, or the ST_ERR_* code where the
// reference raises.
template <int N>
BLSQ_HD int intersect_trust_region(const double* x, const double* s,
                                   double Delta, double& t_lo, double& t_hi) {
    double a = dot<N>(s, s);
    if (a == 0) return ST_ERR_TR_ZERO;
    double b = dot<N>(x, s);
    double c = dot<N>(x, x) - Delta * Delta;
    if (c > 0) return ST_ERR_TR_OUTSIDE;
    double disc = sqrt(b * b - a * c);
    double q = -(b + copysign(disc, b));
    double r1 = q / a;
    double r2 = c / q;
    if (r1 < r2) { t_lo = r1; t_hi = r2; } else { t_lo = r2; t_hi = r1; }
    return 0;
}

// trust_region.py:47-53
template <int N>
BLSQ_HD void phi_and_derivative(double alpha, const double* suf,
                                const double* s, double Delta, double& phi,
                                double& dphi) {
    double nn = 0.0, dd = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        double den = s[i] * s[i] + alpha;
        double q = suf[i] / den;
        nn = fma(q, q, nn);
        dd += (suf[i] * suf[i]) / (den * den * den);
    }
    double pn = sqrt(nn);
    phi = pn - Delta;
    dphi = -dd / pn;
}

// trust_region.py:56-152.  Vt is row-major N x N, ROW j = right singular
// vector j (i.e. V transposed); suf = s * (U^T f).  The singular values need not be sorted: the
// rank test uses min/max, everything else is a sum over j.  alpha is the
// warm start on entry and the LM parameter on exit.
template <int N>
BLSQ_HD void solve_lsq_trust_region(int m, const double* suf, const double* s,
                                    const double* Vt, double Delta,
                                    double& alpha, double* p,
                                    bool zero_col = true) {
    double smin = s[0], smax = s[0];
    BLSQ_UNROLL
    for (int i = 1; i < N; i++) {
        smin = s[i] < smin ? s[i] : smin;
        smax = s[i] > smax ? s[i] : smax;
    }
    bool full_rank = (m >= N) && (smin > EPS * m * smax);
    double w[N];
    if (full_rank) {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) w[j] = (suf[j] / s[j]) / s[j];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            double acc = 0.0;
            BLSQ_UNROLL
            for (int j = 0; j < N; j++) acc = fma(Vt[j * N + i], w[j], acc);
            p[i] = -acc;
        }
        if (norm2<N>(p) <= Delta) { alpha = 0.0; return; }
    }
    double hi = norm2<N>(suf) / Delta;
    double lo = 0.0;
    double phi, dphi;
    if (full_rank) {
        phi_and_derivative<N>(0.0, suf, s, Delta, phi, dphi);
        lo = -phi / dphi;
    }
    if (!full_rank && alpha == 0) {
        double a1 = 0.001 * hi, a2 = sqrt(lo * hi);
        alpha = a1 > a2 ? a1 : a2;
    }
    for (int it = 0; it < 10; it++) {
        if (alpha < lo || alpha > hi) {
            double a1 = 0.001 * hi, a2 = sqrt(lo * hi);
            alpha = a1 > a2 ? a1 : a2;
        }
        phi_and_derivative<N>(alpha, suf, s, Delta, phi, dphi);
        if (fabs(phi) < 0.01 * Delta) break;
        if (phi < 0) hi = alpha;
        double q = phi / dphi;
        double cand = alpha - q;
        lo = lo > cand ? lo : cand;
        alpha -= (phi + Delta) * q / Delta;
    }
    // An EXACTLY zero singular value of a matrix WITHOUT a zero column
    // (duplicate columns: the Gram-Schmidt / Jacobi route keeps the zero LAPACK
    // would return as ~1e-16 s_max) makes |p(alpha)| < Delta for every
    // alpha > 0: no root, and the iteration above can leave alpha negative.
    // The reference never sees this (its noise-level s_min gives the root a
    // bracket); take the minimum-norm end of the bracket.  A zero COLUMN
    // (Beale at x0) gives the reference an exact zero too and is left alone.
    if (smin == 0.0 && !zero_col && !(alpha > 0.0)) {
        double a1 = 0.001 * hi, a2 = sqrt(lo * hi);
        alpha = a1 > a2 ? a1 : a2;
    }
    BLSQ_UNROLL
    for (int j = 0; j < N; j++) w[j] = suf[j] / (s[j] * s[j] + alpha);
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        double acc = 0.0;
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) acc = fma(Vt[j * N + i], w[j], acc);
        p[i] = -acc;
    }
    if (phi > 0) {
        double sc = Delta / norm2<N>(p);
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) p[i] *= sc;
    }
}

// ---------------------------------------------------------------------------
// Dense n x n tail: packed upper-triangular R (row-major, row i holds columns
// i..N-1), Givens fold-in of a diagonal block, one-sided Jacobi SVD.
// ---------------------------------------------------------------------------

template <int N>
BLSQ_HD constexpr int tri_index(int i, int j) {   // i <= j
    return i * N - (i * (i - 1)) / 2 + (j - i);
}
template <int N>
struct Tri { static constexpr int size = N * (N + 1) / 2; };

// y = R * s for packed upper-triangular R
template <int N>
BLSQ_HD void tri_matvec(const double* R, const double* s, double* y) {
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        double acc = 0.0;
        BLSQ_UNROLL
        for (int j = i; j < N; j++) acc = fma(R[tri_index<N>(i, j)], s[j], acc);
        y[i] = acc;
    }
}

BLSQ_HD double rsqrt_d(double x) {
#if defined(__CUDA_ARCH__)
    return rsqrt(x);
#else
    return 1.0 / sqrt(x);
#endif
}

// One-sided (Hestenes) Jacobi SVD of the N x N matrix A (row-major, in
// place), run on the ROWS of A, i.e. on the columns of A^T.  For the upper
// triangles this is fed, A^T is lower triangular, which is the orientation in
// which one-sided Jacobi converges fastest (Drmac & Veselic).  With
//   A = U S V^T :  rows of A  ->  s_j * v_j^T   (right singular vectors)
//                  b          ->  U^T b         (same rotations applied to b)
// so neither U nor V is accumulated.  High relative accuracy; the order of
// the singular values is whatever falls out (callers do not depend on it).
template <int N>
BLSQ_HD void jacobi_rows(double* A, double* b) {
    if (N == 1) return;
    for (int sweep = 0; sweep < 40; sweep++) {
        bool rotated = false;
        BLSQ_UNROLL
        for (int p = 0; p < N - 1; p++) {
            BLSQ_UNROLL
            for (int q = p + 1; q < N; q++) {
                double al = 0.0, be = 0.0, ga = 0.0;
                BLSQ_UNROLL
                for (int i = 0; i < N; i++) {
                    double ap = A[p * N + i], aq = A[q * N + i];
                    al = fma(ap, ap, al);
                    be = fma(aq, aq, be);
                    ga = fma(ap, aq, ga);
                }
                if (ga == 0.0 || ga * ga <= (EPS * EPS) * (al * be)) continue;
                rotated = true;
                double zeta = (be - al) / (2.0 * ga);
                double t = copysign(1.0, zeta) /
                           (fabs(zeta) + sqrt(fma(zeta, zeta, 1.0)));
                double c = rsqrt_d(fma(t, t, 1.0));
                double sn = c * t;
                BLSQ_UNROLL
                for (int i = 0; i < N; i++) {
                    double ap = A[p * N + i], aq = A[q * N + i];
                    A[p * N + i] = fma(c, ap, -(sn * aq));
                    A[q * N + i] = fma(sn, ap, c * aq);
                }
                double bp = b[p], bq = b[q];
                b[p] = fma(c, bp, -(sn * bq));
                b[q] = fma(sn, bp, c * bq);
            }
        }
        if (!rotated) break;
    }
}

// Factorisation of the hat-space augmented matrix (trf.py:264-274):
//   [ J_h ; diag(sqrt(diag_h)) ]  with  J_h = Q * (R * diag(d)),
// so its singular values / right vectors are those of the 2N x N matrix
// [R*diag(d); diag(sq)].  The diagonal block is folded into the triangle by
// Givens rotations (which also act on [qtf; 0]), then Jacobi runs on N x N.
// Outputs: s, Vt (row j = right singular vector j), suf = s * (U^T f_aug),
// and Rh = R*diag(d) (packed) for the quadratic-model evaluations
// (trf.py:69-74,100-102).
template <int N>
BLSQ_HD void hat_fold(const double* R, const double* qtf, const double* d,
                      const double* diag_h, double* Rh, double* A, double* b) {
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        b[i] = qtf[i];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            if (j >= i) {
                double v = R[tri_index<N>(i, j)] * d[j];
                Rh[tri_index<N>(i, j)] = v;
                A[i * N + j] = v;
            } else {
                A[i * N + j] = 0.0;
            }
        }
    }
    // fold row k of diag(sqrt(diag_h)) into the triangle
    BLSQ_UNROLL
    for (int k = 0; k < N; k++) {
        double e = sqrt(diag_h[k]);
        if (e == 0.0) continue;
        double row[N];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) row[j] = (j == k) ? e : 0.0;
        double bz = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            if (i < k) continue;
            double x = row[i];
            if (x == 0.0) continue;
            double a = A[i * N + i];
            double r = sqrt(fma(a, a, x * x));
            double c = a / r, sn = x / r;
            BLSQ_UNROLL
            for (int j = 0; j < N; j++) {
                if (j < i) continue;
                double aj = A[i * N + j], rj = row[j];
                A[i * N + j] = fma(c, aj, sn * rj);
                row[j] = fma(-sn, aj, c * rj);
            }
            double bi = b[i];
            b[i] = fma(c, bi, sn * bz);
            bz = fma(-sn, bi, c * bz);
        }
    }
}

// Jacobi on the folded triangle and extraction of s, Vt, suf (see hat_svd)
template <int N>
BLSQ_HD void hat_finish(double* A, double* b, double* s, double* Vt, double* suf) {
    jacobi_rows<N>(A, b);
    BLSQ_UNROLL
    for (int j = 0; j < N; j++) {
        double nn = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) nn = fma(A[j * N + i], A[j * N + i], nn);
        s[j] = sqrt(nn);
        suf[j] = s[j] * b[j];
        double inv = (s[j] > 0.0) ? 1.0 / s[j] : 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) Vt[j * N + i] = A[j * N + i] * inv;
    }
}

template <int N>
BLSQ_HD void hat_svd(const double* R, const double* qtf, const double* d,
                     const double* diag_h, double* Rh, double* s, double* Vt,
                     double* suf) {
    double A[N * N];
    double b[N];
    hat_fold<N>(R, qtf, d, diag_h, Rh, A, b);
    hat_finish<N>(A, b, s, Vt, suf);
}

// Gauss-Newton shortcut of solve_lsq_trust_region (trust_region.py:108-117)
// on the folded triangle A (upper triangular) and b = top of Q'^T f_aug:
// the reference takes p = -V (uf / s) and returns (p, 0.0) when the matrix has
// full rank and |p| <= Delta.  Here p = -A^-1 b through the explicit
// triangular inverse T, and full rank is CERTIFIED by the bound
// cond(A) <= |A|_F |T|_F (so s_min / s_max > EPS m with a factor 4 to spare).
// Returns false -- and the caller falls back to the SVD route -- when the
// certificate fails, the step is longer than Delta, or |p| is within 1e-9 of
// Delta (so that the accept / Levenberg-Marquardt decision is always taken by
// the reference's own arithmetic).  ~95 % of the C2 trust-region solves are
// Gauss-Newton steps (oracle count), none of them needs the Jacobi sweeps.
template <int N>
BLSQ_HD bool gn_shortcut(const double* A, const double* b, int m, double Delta,
                         double* p_h) {
    if (m < N) return false;
    double T[N * N];
    double fa = 0.0, ft = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        const double aii = A[i * N + i];
        if (!(aii != 0.0)) return false;
        T[i * N + i] = 1.0 / aii;
    }
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            if (j < i) continue;
            fa = fma(A[i * N + j], A[i * N + j], fa);
            if (j > i) {
                double acc = 0.0;
                BLSQ_UNROLL
                for (int k = 0; k < N; k++) {
                    if (k < i || k >= j) continue;
                    acc = fma(T[i * N + k], A[k * N + j], acc);
                }
                T[i * N + j] = -acc * T[j * N + j];
            }
            ft = fma(T[i * N + j], T[i * N + j], ft);
        }
    }
    const double em = EPS * m;
    if (!(fa * ft * (em * em) < 0.0625)) return false;     // also rejects NaN / inf
    // p = -A^-1 b by back substitution; the quotient by a_ii is the correctly
    // rounded one (reciprocal + one FMA correction, Markstein), so that for
    // n = 1 the step is bit for bit the reference's -V (uf / s) = -b / a
    // (its own test_diff_step compares two solves with assert_equal)
    double nn = 0.0;
    BLSQ_UNROLL
    for (int ii = 0; ii < N; ii++) {
        const int i = N - 1 - ii;
        double num = -b[i];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            if (j <= i) continue;
            num = fma(-A[i * N + j], p_h[j], num);
        }
        const double r = T[i * N + i];
        double q = num * r;
        q = fma(fma(-q, A[i * N + i], num), r, q);
        p_h[i] = q;
        nn = fma(q, q, nn);
    }
    return sqrt(nn) <= Delta * (1.0 - 1e-9);
}

// ---------------------------------------------------------------------------
// trf.py 1-D quadratic helpers
// ---------------------------------------------------------------------------

// trf.py:15-34
BLSQ_HD double minimize_quadratic(double a, double b, double lo, double hi) {
    double t0 = lo, t1 = hi;
    double y0 = a * (t0 * t0) + b * t0;
    double y1 = a * (t1 * t1) + b * t1;
    double tb = t0, yb = y0;
    if (y1 < yb) { tb = t1; yb = y1; }
    if (a != 0) {
        double ext = -0.5 * b / a;
        if (lo <= ext && ext <= hi) {
            double y2 = a * (ext * ext) + b * ext;
            if (y2 < yb) { tb = ext; yb = y2; }
        }
    }
    return tb;
}

// trf.py:37-76 with J replaced by the triangular factor Rh (same values:
// |J_h s| = |Rh s|, (J_h s0).(J_h s) = (Rh s0).(Rh s)).
template <int N>
BLSQ_HD void build_quadratic_1d(const double* Rh, const double* diag,
                                const double* g, const double* s,
                                const double* s0, double& a, double& b) {
    double v[N];
    tri_matvec<N>(Rh, s, v);
    double sd = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) sd = fma(s[i] * diag[i], s[i], sd);
    a = 0.5 * (dot<N>(v, v) + sd);
    b = dot<N>(g, s);
    if (s0) {
        double u[N];
        tri_matvec<N>(Rh, s0, u);
        double s0d = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) s0d = fma(s0[i] * diag[i], s[i], s0d);
        b += dot<N>(u, v) + s0d;
    }
}

// trf.py:79-102 for one step
template <int N>
BLSQ_HD double evaluate_quadratic(const double* Rh, const double* diag,
                                  const double* g, const double* s) {
    double v[N];
    tri_matvec<N>(Rh, s, v);
    double sd = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) sd = fma(diag[i], s[i] * s[i], sd);
    return 0.5 * (dot<N>(v, v) + sd) + dot<N>(s, g);
}

// ---------------------------------------------------------------------------
// TRF: one problem, one round  (trf.py:238-352 cut as judge -> linearise ->
// propose; see DESIGN.md "Batched rounds")
// ---------------------------------------------------------------------------

// Records are laid out in blocks that start at multiples of 4 doubles (32
// bytes): every block moves with 256-bit loads / stores (LDG.E.256 on sm_100a,
// a whole DRAM sector per instruction) and can be fetched on its own when the
// round needs it, instead of the whole record sitting in registers.
// LinRec: the record produced by the linearise kernel for the trial point.
template <int N>
struct LinRec {
    static constexpr int NT = N * (N + 1) / 2;
    static constexpr int R = 0;
    static constexpr int QTF = NT;
    static constexpr int G = NT + N;
    static constexpr int OBJ = NT + 2 * N;
    static constexpr int SIZE = (NT + 2 * N + 1 + 3) & ~3;     // multiple of 4
};

template <int N>
struct TrfState {
    // layout of one problem's record in the state array (doubles)
    static constexpr int NT = N * (N + 1) / 2;
    static constexpr int NP = (N + 3) & ~3;
    static constexpr int X = 0;            // accepted point
    static constexpr int XNEW = NP;        // trial point in flight
    static constexpr int SCALE = 2 * NP;   // 1/scaling, or running 'jac' scale
    static constexpr int R = 3 * NP;       // linearisation at X: same layout as LinRec
    static constexpr int QTF = R + NT;
    static constexpr int G = QTF + N;      // J^T f at X
    static constexpr int OBJ = G + N;      // f.f at X
    static constexpr int SCAL = R + LinRec<N>::SIZE;   // scalar block (8 doubles)
    static constexpr int DELTA = SCAL;
    static constexpr int ALPHA = SCAL + 1;
    static constexpr int PRED = SCAL + 2;   // predicted reduction of the trial
    static constexpr int CORR = SCAL + 3;   // step_h.diag_h.step_h
    static constexpr int NSTEPH = SCAL + 4; // |step_h|
    static constexpr int NSTEP = SCAL + 5;  // |step|
    static constexpr int GNORM = SCAL + 6;  // optimality at the last linearise
    static constexpr int SIZE = SCAL + 8;
};

struct SolveParams {
    double ftol, xtol, gtol;
    int max_nfev;
    int m;
    int jac_scaling;     // 1: scaling='jac' (running minimum of 1/colnorm)
};

// istate layout (int32 per problem).  IS_ONB / IS_MARKS pack one 2-bit
// field per coordinate (0, 1 = lower, 2 = upper): dogbox's on_bound and the
// bound hits of the trial in flight; IS_FREE is the free-set bitmask of the
// trial with tr_hit in bit 30.  TRF uses only the first three.
enum { IS_STATUS = 0, IS_NFEV = 1, IS_NJEV = 2, IS_ONB = 3, IS_MARKS = 4,
       IS_FREE = 5, IS_SIZE = 8 };

// One TRF round for one problem.  `lin` is the linearisation at the trial
// point XNEW (or at the strictly feasible start when first != 0).
// Returns true when a new trial point was written to st[XNEW].
// MODE 0: the whole round in one piece: Gauss-Newton shortcut, else the SVD
// route.  MODE 1: the same, but returns TRF_DEFER (state updated, no trial
// written) instead of entering the SVD route.  MODE 2: resume a deferred
// problem: skip the judge / accept part (already done by MODE 1; `lin` is not
// read) and propose through the SVD.  Returns 0 (finished / no trial), 1 (new
// trial in st[XNEW]) or TRF_DEFER.
enum { TRF_DEFER = 2 };

// ---- block moves: 256-bit on the device when K % 4 == 0 (p 32-byte aligned) ----
template <int K>
BLSQ_HD void ld_block(const double* p, double* d) {
#if defined(__CUDA_ARCH__)
    if (K % 4 == 0) {
        BLSQ_UNROLL
        for (int i = 0; i < K; i += 4)
            asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(d[i]), "=d"(d[i + 1]), "=d"(d[i + 2]), "=d"(d[i + 3])
                         : "l"(p + i));
        return;
    }
#endif
    BLSQ_UNROLL
    for (int i = 0; i < K; i++) d[i] = p[i];
}
template <int K>
BLSQ_HD void st_block(double* p, const double* v) {
#if defined(__CUDA_ARCH__)
    if (K % 4 == 0) {
        BLSQ_UNROLL
        for (int i = 0; i < K; i += 4)
            asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p + i), "d"(v[i]),
                         "d"(v[i + 1]), "d"(v[i + 2]), "d"(v[i + 3])
                         : "memory");
        return;
    }
#endif
    BLSQ_UNROLL
    for (int i = 0; i < K; i++) p[i] = v[i];
}

// Packed-triangle versions of hat_fold / gn_shortcut (same arithmetic as the
// N x N forms above up to the Givens coefficients, which come from one
// reciprocal square root instead of a square root and two divisions).
// A: packed upper triangle (tri_index), in: R * diag(d); out: the triangle of
// the QR factor of [R diag(d); diag(sqrt(diag_h))].  b: in Q^T f, out: rotated.
template <int N>
BLSQ_HD void hat_fold_packed(double* A, double* b, const double* diag_h) {
    BLSQ_UNROLL
    for (int k = 0; k < N; k++) {
        double e = sqrt(diag_h[k]);
        if (e == 0.0) continue;
        double row[N];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) row[j] = (j == k) ? e : 0.0;
        double bz = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            if (i < k) continue;
            double x = row[i];
            if (x == 0.0) continue;
            double a = A[tri_index<N>(i, i)];
            double rinv = rsqrt_d(fma(a, a, x * x));
            double c = a * rinv, sn = x * rinv;
            BLSQ_UNROLL
            for (int j = 0; j < N; j++) {
                if (j < i) continue;
                double aj = A[tri_index<N>(i, j)], rj = row[j];
                A[tri_index<N>(i, j)] = fma(c, aj, sn * rj);
                row[j] = fma(-sn, aj, c * rj);
            }
            double bi = b[i];
            b[i] = fma(c, bi, sn * bz);
            bz = fma(-sn, bi, c * bz);
        }
    }
}

template <int N>
BLSQ_HD bool gn_shortcut_packed(const double* A, const double* b, int m, double Delta,
                                double* p_h) {
    if (m < N) return false;
    double T[Tri<N>::size];
    double fa = 0.0, ft = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        const double aii = A[tri_index<N>(i, i)];
        if (!(aii != 0.0)) return false;
        T[tri_index<N>(i, i)] = 1.0 / aii;
    }
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            if (j < i) continue;
            const double aij = A[tri_index<N>(i, j)];
            fa = fma(aij, aij, fa);
            if (j > i) {
                double acc = 0.0;
                BLSQ_UNROLL
                for (int k = 0; k < N; k++) {
                    if (k < i || k >= j) continue;
                    acc = fma(T[tri_index<N>(i, k)], A[tri_index<N>(k, j)], acc);
                }
                T[tri_index<N>(i, j)] = -acc * T[tri_index<N>(j, j)];
            }
            ft = fma(T[tri_index<N>(i, j)], T[tri_index<N>(i, j)], ft);
        }
    }
    const double em = EPS * m;
    if (!(fa * ft * (em * em) < 0.0625)) return false;     // also rejects NaN / inf
    double nn = 0.0;
    BLSQ_UNROLL
    for (int ii = 0; ii < N; ii++) {
        const int i = N - 1 - ii;
        double num = -b[i];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            if (j <= i) continue;
            num = fma(-A[tri_index<N>(i, j)], p_h[j], num);
        }
        const double r = T[tri_index<N>(i, i)];
        double q = num * r;
        q = fma(fma(-q, A[tri_index<N>(i, i)], num), r, q);   // correctly rounded quotient
        p_h[i] = q;
        nn = fma(q, q, nn);
    }
    return sqrt(nn) <= Delta * (1.0 - 1e-9);
}

// y = R (d o s) for the packed triangle R: J_h s in the rotated frame
template <int N>
BLSQ_HD void tri_matvec_d(const double* R, const double* d, const double* s, double* y) {
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        double acc = 0.0;
        BLSQ_UNROLL
        for (int j = i; j < N; j++) {
            // R[i][j] * d[j] is the entry of R diag(d) (J_h in the rotated frame)
            acc = fma(R[tri_index<N>(i, j)] * d[j], s[j], acc);
        }
        y[i] = acc;
    }
}

template <int N>
BLSQ_HD double evaluate_quadratic_d(const double* R, const double* d, const double* diag,
                                    const double* g, const double* s) {
    double v[N];
    tri_matvec_d<N>(R, d, s, v);
    double sd = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) sd = fma(diag[i], s[i] * s[i], sd);
    return 0.5 * (dot<N>(v, v) + sd) + dot<N>(s, g);
}

template <int N>
BLSQ_HD void build_quadratic_1d_d(const double* R, const double* d, const double* diag,
                                  const double* g, const double* s, const double* s0,
                                  double& a, double& b) {
    double v[N];
    tri_matvec_d<N>(R, d, s, v);
    double sd = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) sd = fma(s[i] * diag[i], s[i], sd);
    a = 0.5 * (dot<N>(v, v) + sd);
    b = dot<N>(g, s);
    if (s0) {
        double u[N];
        tri_matvec_d<N>(R, d, s0, u);
        double s0d = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) s0d = fma(s0[i] * diag[i], s[i], s0d);
        b += dot<N>(u, v) + s0d;
    }
}

// One TRF round for one problem, working on the records IN MEMORY: `sp` the
// state record (TrfState layout), `lp` the linearisation record of the trial
// point (LinRec), both 32-byte aligned.  Blocks are loaded when the round gets
// to them and stored when they change, so the live register set stays small
// (the first version held all 39 + 20 doubles of an N = 4 problem in
// registers from the first to the last instruction: 128 registers plus 528-860
// bytes of spills, profiles/r1_c2_round_kernel_ncu.md).  ist: the first four
// istate words in registers (status, nfev, njev, -).
template <int N, int MODE>
BLSQ_HD int trf_round_impl(double* sp, int* ist, const double* lp,
                           const double* x0, const double* lb, const double* ub,
                           const double* scaling, const SolveParams& P, int first,
                           double* xout = nullptr) {
    typedef TrfState<N> S;
    typedef LinRec<N> L;
    constexpr int NP = S::NP;
    int status = ST_RUNNING;     // pending status set by the inner loop
    bool adopt = false;
    BLSQ_PHASE_BEGIN;
    double sc[8];                // DELTA ALPHA PRED CORR NSTEPH NSTEP GNORM -
    ld_block<8>(sp + S::SCAL, sc);
    double blk[L::SIZE];         // R, QTF, G, OBJ of the point the round works at
    double x[NP];
    if (MODE == 2) {
        first = 0;               // scale / Delta / alpha are in the state already
        ld_block<NP>(sp + S::X, x);
        ld_block<L::SIZE>(sp + S::R, blk);
    } else if (first) {
        // trf.py:201-235
        ist[IS_NFEV] = 1;
        ist[IS_NJEV] = 0;
        adopt = true;
        sc[1] = 0.0;             // alpha
        ld_block<L::SIZE>(lp, blk);
    } else {
        // judge the trial (trf.py:310-344)
        ld_block<L::SIZE>(lp, blk);
        ld_block<NP>(sp + S::X, x);
        int nfev = ++ist[IS_NFEV];
        double obj = sp[S::OBJ];
        double obj_new = blk[L::OBJ];
        double actual = obj - obj_new;
        double pred = sc[2];
        double ratio = (pred > 0) ? (actual - sc[3]) / pred : 0.0;
        double nsh = sc[4];
        double Delta = sc[0];
        if (ratio < 0.25) {
            double Dn = 0.25 * nsh;
            sc[1] *= Delta / Dn;
            sc[0] = Dn;
        } else if (ratio > 0.75 && nsh > 0.95 * Delta) {
            sc[0] = Delta * 2.0;
            sc[1] *= 0.5;
        }
        bool f_ok = fabs(actual) < P.ftol * obj && ratio > 0.25;
        double xn = norm2<N>(x);
        bool x_ok = sc[5] < P.xtol * (SQRT_EPS > xn ? SQRT_EPS : xn);
        if (f_ok && x_ok) status = 4;
        else if (f_ok) status = 2;
        else if (x_ok) status = 3;
        adopt = actual > 0;                       // trf.py:346
        if (nfev >= P.max_nfev) {
            // trf.py:238,354-358: budget exhausted -> status 0 whatever the
            // inner loop decided; an accepted last step is still taken and
            // its Jacobian counted (trf.py:346-352)
            if (adopt) {
                ld_block<NP>(sp + S::XNEW, x);
                st_block<NP>(sp + S::X, x);
                st_block<L::SIZE>(sp + S::R, blk);
                ist[IS_NJEV]++;
            }
            st_block<8>(sp + S::SCAL, sc);
            ist[IS_STATUS] = 0;
            return 0;
        }
    }
    if (adopt) {
        // the trial becomes the point; R, QTF, G, OBJ are contiguous and in the
        // same order in both records
        ld_block<NP>(sp + S::XNEW, x);
        st_block<NP>(sp + S::X, x);
        st_block<L::SIZE>(sp + S::R, blk);
        ist[IS_NJEV]++;
    } else if (MODE != 2) {
        ld_block<L::SIZE>(sp + S::R, blk);        // rejected: back to the old factor
    }
    if (first && 1 >= P.max_nfev) {          // `while nfev < max_nfev` never entered
        sc[6] = dnan();
        st_block<8>(sp + S::SCAL, sc);
        ist[IS_STATUS] = 0;
        return 0;
    }

    BLSQ_PHASE(0);
    // ---- linearise (trf.py:239-277) at x ----
    const double* Rm = blk + L::R;
    double scale[NP], d[N], g_h[N], diag_h[N], v[N];
    double l[N], u[N];
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) { l[i] = lb[i]; u[i] = ub[i]; }
    if (P.jac_scaling) {
        // trf.py:216-221 (first) / 239-242 (running minimum); the column
        // norms of J are those of its triangular factor
        if (!first) ld_block<NP>(sp + S::SCALE, scale);
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            double nn = 0.0;
            BLSQ_UNROLL
            for (int i = 0; i <= j; i++) {
                double r = Rm[tri_index<N>(i, j)];
                nn = fma(r, r, nn);
            }
            double cn = sqrt(nn);
            if (first) {
                if (cn == 0) cn = 1.0;
                scale[j] = 1.0 / cn;
            } else {
                scale[j] = np_min(scale[j], 1.0 / cn);
            }
        }
        BLSQ_UNROLL
        for (int j = N; j < NP; j++) scale[j] = 0.0;
        if (MODE != 2) st_block<NP>(sp + S::SCALE, scale);
    } else if (first) {
        BLSQ_UNROLL
        for (int j = 0; j < NP; j++) scale[j] = (j < N) ? 1.0 / scaling[j] : 0.0;
        st_block<NP>(sp + S::SCALE, scale);
    } else {
        ld_block<NP>(sp + S::SCALE, scale);
    }
    double g_norm = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        double jv;
        const double gi = blk[L::G + i];
        cl_scaling(x[i], gi, l[i], u[i], v[i], jv);
        d[i] = sqrt(v[i]) * scale[i];
        g_h[i] = d[i] * gi;
        diag_h[i] = gi * jv * (scale[i] * scale[i]);
        double gv = fabs(gi * v[i]);
        if (gv > g_norm || gv != gv) g_norm = gv;
    }
    if (first) {
        // trf.py:223-226: Delta from the ORIGINAL x0
        double q[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) q[i] = x0[i] / (scale[i] * sqrt(v[i]));
        double D0 = norm2<N>(q);
        sc[0] = (D0 == 0) ? 1.0 : D0;
    }
    sc[6] = g_norm;
    if (g_norm < P.gtol) status = 1;              // trf.py:252-254 (overrides)
    if (status != ST_RUNNING) {
        st_block<8>(sp + S::SCAL, sc);
        ist[IS_STATUS] = status;
        return 0;
    }

    double theta = 1.0 - g_norm;
    if (theta < 0.995) theta = 0.995;

    BLSQ_PHASE(1);
    // ---- propose (trf.py:284-308) ----
    const double Delta = sc[0];
    double alpha = sc[1];
    double p_h[N], p[N];
    {
        double A[S::NT], b[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            b[i] = blk[L::QTF + i];
            BLSQ_UNROLL
            for (int j = i; j < N; j++)
                A[tri_index<N>(i, j)] = Rm[tri_index<N>(i, j)] * d[j];
        }
        hat_fold_packed<N>(A, b, diag_h);
        BLSQ_PHASE(2);
        // every mode takes the same decision with the same arithmetic, so the
        // result does not depend on how the driver splits the work
        if (MODE != 2 && gn_shortcut_packed<N>(A, b, P.m, Delta, p_h)) {
            alpha = 0.0;                           // trust_region.py:117
            BLSQ_PHASE(3);
        } else if (MODE == 1) {
            st_block<8>(sp + S::SCAL, sc);         // Delta / alpha of the judge, g_norm
            return TRF_DEFER;
        } else {
            // does the hat-space matrix have an exactly zero column?
            bool zero_col = false;
            double Af[N * N];
            BLSQ_UNROLL
            for (int j = 0; j < N; j++) {
                bool z = true;
                BLSQ_UNROLL
                for (int i = 0; i < N; i++) {
                    Af[i * N + j] = (i <= j) ? A[tri_index<N>(i <= j ? i : j, j)] : 0.0;
                    if (i <= j) z = z && (Af[i * N + j] == 0.0);
                }
                zero_col = zero_col || z;
            }
            double sv[N], Vt[N * N], suf[N];
            BLSQ_PHASE(4);
            hat_finish<N>(Af, b, sv, Vt, suf);
            BLSQ_PHASE(5);
            solve_lsq_trust_region<N>(P.m, suf, sv, Vt, Delta, alpha, p_h, zero_col);
            BLSQ_PHASE(6);
        }
    }
    sc[1] = alpha;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) p[i] = d[i] * p_h[i];
    int hits[N];
    double to_bound = step_size_to_bound<N>(x, p, l, u, hits);
    double step_h[N];
    double qbest;
    if (to_bound >= 1) {
        double tb = theta * to_bound;
        double f = tb < 1 ? tb : 1;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) step_h[i] = p_h[i] * f;
        qbest = evaluate_quadratic_d<N>(Rm, d, diag_h, g_h, step_h);
    } else {
        // find_reflected_step, trf.py:105-156 (the hits are those of to_bound)
        double stride_p = to_bound;
        double r_h[N], r[N], x_edge[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            r_h[i] = hits[i] ? -p_h[i] : p_h[i];
            r[i] = d[i] * r_h[i];
            p[i] *= stride_p;
            p_h[i] *= stride_p;
            x_edge[i] = x[i] + p[i];
        }
        double t_lo, to_tr;
        int err = intersect_trust_region<N>(p_h, r_h, Delta, t_lo, to_tr);
        if (err) {
            st_block<8>(sp + S::SCAL, sc);
            ist[IS_STATUS] = err;
            return 0;
        }
        double tb2 = step_size_to_bound<N>(x_edge, r, l, u, nullptr);
        tb2 *= theta;
        double hi = tb2 < to_tr ? tb2 : to_tr;          // Python min(a, b)
        double lo = (hi > 0) ? (1 - theta) * stride_p / hi : -1.0;
        double refl[N];
        bool have_r = false;
        if (lo <= hi) {
            double a, b;
            build_quadratic_1d_d<N>(Rm, d, diag_h, g_h, r_h, p_h, a, b);
            double t = minimize_quadratic(a, b, lo, hi);
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) refl[i] = p_h[i] + r_h[i] * t;
            have_r = true;
        }
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) p_h[i] *= theta;
        if (!have_r) {
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) refl[i] = p_h[i];
        }
        // find_gradient_step, trf.py:159-170
        double ng[N], ngd[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) { ng[i] = -g_h[i]; ngd[i] = ng[i] * d[i]; }
        double tbg = step_size_to_bound<N>(x, ngd, l, u, nullptr);
        tbg *= theta;
        double ttr = Delta / norm2<N>(g_h);
        double hig = tbg < ttr ? tbg : ttr;
        double ag, bg;
        build_quadratic_1d_d<N>(Rm, d, diag_h, g_h, ng, nullptr, ag, bg);
        double tg = minimize_quadratic(ag, bg, 0.0, hig);
        double c_h[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) c_h[i] = -tg * g_h[i];
        // trf.py:300-305: argmin, first minimum wins
        double q0 = evaluate_quadratic_d<N>(Rm, d, diag_h, g_h, p_h);
        double q1 = evaluate_quadratic_d<N>(Rm, d, diag_h, g_h, refl);
        double q2 = evaluate_quadratic_d<N>(Rm, d, diag_h, g_h, c_h);
        int k = 0;
        qbest = q0;
        if (q1 < qbest) { k = 1; qbest = q1; }
        if (q2 < qbest) { k = 2; qbest = q2; }
        BLSQ_UNROLL
        for (int i = 0; i < N; i++)
            step_h[i] = (k == 0) ? p_h[i] : (k == 1 ? refl[i] : c_h[i]);
    }
    BLSQ_PHASE(7);
    double xn[NP];
    double corr = 0.0, nsh2 = 0.0, ns2 = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        const double stp = d[i] * step_h[i];
        corr = fma(step_h[i] * diag_h[i], step_h[i], corr);
        nsh2 = fma(step_h[i], step_h[i], nsh2);
        ns2 = fma(stp, stp, ns2);
        xn[i] = strictly_feasible(x[i] + stp, l[i], u[i], 0.0);
    }
    BLSQ_UNROLL
    for (int i = N; i < NP; i++) xn[i] = 0.0;
    st_block<NP>(sp + S::XNEW, xn);
    if (xout) st_block<N>(xout, xn);       // the trial point handed to the callbacks
    sc[2] = -2 * qbest;
    sc[3] = corr;
    sc[4] = sqrt(nsh2);
    sc[5] = sqrt(ns2);
    st_block<8>(sp + S::SCAL, sc);
    BLSQ_PHASE(8);
    return 1;
}

// One TRF round the way the two-kernel device path runs it: Gauss-Newton
// shortcut first, SVD route for the problems that need it.
template <int N>
BLSQ_HD bool trf_round(double* st, int* ist, const double* lin,
                       const double* x0, const double* lb, const double* ub,
                       const double* scaling, const SolveParams& P, int first) {
    // host emulation: exercise the deferred path the way the two kernels do
    int rc = trf_round_impl<N, 1>(st, ist, lin, x0, lb, ub, scaling, P, first);
    if (rc == TRF_DEFER)
        rc = trf_round_impl<N, 2>(st, ist, lin, x0, lb, ub, scaling, P, first);
    return rc == 1;
}

// ---------------------------------------------------------------------------
// dogbox.py
// ---------------------------------------------------------------------------

// dogbox.py:9-35 for one coordinate; flags bit0 orig_l, bit1 orig_u,
// bit2 tr_l, bit3 tr_u
BLSQ_HD int find_intersection(double x, double tr, double lb, double ub,
                              double& lo, double& hi) {
    double lo_c = lb - x, hi_c = ub - x;
    lo = np_max(lo_c, -tr);
    hi = np_min(hi_c, tr);
    return (int)(lo == lo_c) | ((int)(hi == hi_c) << 1) |
           ((int)(lo == -tr) << 2) | ((int)(hi == tr) << 3);
}

template <int N>
struct DogState {
    static constexpr int NT = N * (N + 1) / 2;
    static constexpr int X = 0;
    static constexpr int XNEW = N;
    static constexpr int SCALE = 2 * N;
    static constexpr int R = 3 * N;
    static constexpr int QTF = R + NT;
    static constexpr int G = QTF + N;
    static constexpr int OBJ = G + N;
    static constexpr int DELTA = OBJ + 1;
    static constexpr int PRED = OBJ + 2;
    static constexpr int NSTEP = OBJ + 3;   // |step/scale|_inf of the trial
    static constexpr int GNORM = OBJ + 4;
    static constexpr int SIZE = OBJ + 5;
};

// The fields are shifted as unsigned: coordinate 15 owns bits 30-31, and
// 2 << 30 on a signed int (or a right shift of a negative word) is not well
// defined.
BLSQ_HD int get2(int word, int i) {      // decode 2-bit field -> -1/0/+1
    unsigned v = ((unsigned)word >> (2 * i)) & 3u;
    return v == 1u ? -1 : (v == 2u ? 1 : 0);
}
BLSQ_HD int put2(int i, int val) {       // val in -1/0/+1
    return (int)((unsigned)(val < 0 ? 1 : (val > 0 ? 2 : 0)) << (2 * i));
}

// dogleg_step / constrained_cauchy_step over the free coordinates
// (dogbox.py:38-97).  Coordinates with free[i]==0 are ignored (the reference
// works on gathered sub-vectors; masks give the same arithmetic because every
// reduction here is a min / any / all).
template <int N>
BLSQ_HD void dog_box_geometry(const double* x, const double* tr,
                              const double* lb, const double* ub,
                              const bool* free_, double* lo, double* hi,
                              int* flags) {
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        if (free_[i]) flags[i] = find_intersection(x[i], tr[i], lb[i], ub[i],
                                                   lo[i], hi[i]);
        else { flags[i] = 0; lo[i] = 0; hi[i] = 0; }
    }
}

template <int N>
BLSQ_HD bool in_box(const double* s, const double* lo, const double* hi,
                    const bool* free_) {
    bool ok = true;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++)
        if (free_[i]) ok = ok && (s[i] >= lo[i]) && (s[i] <= hi[i]);
    return ok;
}

// step_size_to_bound restricted to the free coordinates
template <int N>
BLSQ_HD double step_to_box(const double* x, const double* d, const double* lo,
                           const double* hi, const bool* free_, int* hits) {
    double t[N];
    double tmin = dinf();
    bool has_nan = false;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        if (!free_[i]) { t[i] = dinf(); continue; }
        if (d[i] != 0)
            t[i] = np_max((lo[i] - x[i]) / d[i], (hi[i] - x[i]) / d[i]);
        else
            t[i] = dinf();
        if (t[i] != t[i]) has_nan = true;
        if (!(tmin < t[i])) tmin = t[i];   // NumPy: ties take the later element
    }
    if (has_nan) tmin = dnan();
    BLSQ_UNROLL
    for (int i = 0; i < N; i++)
        hits[i] = (free_[i] && t[i] == tmin) ? isign(d[i]) : 0;
    return tmin;
}

template <int N>
BLSQ_HD void hit_bookkeeping(const int* hits, const int* flags,
                             const bool* free_, int* marks, bool& tr_hit) {
    tr_hit = false;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        marks[i] = 0;
        if (!free_[i]) continue;
        if (hits[i] < 0 && (flags[i] & 1)) marks[i] = -1;
        if (hits[i] > 0 && (flags[i] & 2)) marks[i] = 1;
        if ((hits[i] < 0 && (flags[i] & 4)) || (hits[i] > 0 && (flags[i] & 8)))
            tr_hit = true;
    }
}

// One dogbox round for one problem (dogbox.py:164-267).
template <int N>
BLSQ_HD bool dogbox_round(double* st, int* ist, const double* lin,
                          const double* x0, const double* lb,
                          const double* ub, const double* scaling,
                          const SolveParams& P, int first) {
    typedef DogState<N> S;
    typedef LinRec<N> L;
    int status = ST_RUNNING;
    bool adopt;
    double l[N], u[N];
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) { l[i] = lb[i]; u[i] = ub[i]; }
    if (first) {
        ist[IS_NFEV] = 1;
        ist[IS_NJEV] = 0;
        adopt = true;
        int onb = 0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            int ob = 0;
            if (x0[i] == l[i]) ob = -1;
            if (x0[i] == u[i]) ob = 1;
            onb |= put2(i, ob);
            st[S::X + i] = x0[i];
        }
        ist[IS_ONB] = onb;
    } else {
        int nfev = ++ist[IS_NFEV];
        double obj = st[S::OBJ];
        double obj_new = lin[L::OBJ];
        double actual = obj - obj_new;
        double pred = st[S::PRED];
        double ratio = (pred > 0) ? actual / pred : 0.0;
        bool tr_hit = (ist[IS_FREE] >> 30) & 1;
        if (ratio < 0.25) st[S::DELTA] = 0.25 * st[S::NSTEP];
        else if (ratio > 0.75 && tr_hit) st[S::DELTA] *= 2.0;
        bool f_ok = fabs(actual) < P.ftol * obj && ratio > 0.25;
        double xs = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            double q = fabs(st[S::X + i] / st[S::SCALE + i]);
            if (q > xs || q != q) xs = q;
        }
        bool x_ok = st[S::DELTA] < P.xtol * (SQRT_EPS > xs ? SQRT_EPS : xs);
        if (f_ok && x_ok) status = 4;
        else if (f_ok) status = 2;
        else if (x_ok) status = 3;
        adopt = actual > 0;
        if (adopt) {
            // dogbox.py:253-267
            int onb = ist[IS_ONB], marks = ist[IS_MARKS], fr = ist[IS_FREE];
            int onb_new = 0;
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) {
                int ob = ((fr >> i) & 1) ? get2(marks, i) : get2(onb, i);
                onb_new |= put2(i, ob);
                double xi = st[S::XNEW + i];
                if (ob == -1) xi = l[i];
                if (ob == 1) xi = u[i];
                st[S::X + i] = xi;
            }
            ist[IS_ONB] = onb_new;
        }
        if (nfev >= P.max_nfev) {
            if (adopt) {
                BLSQ_UNROLL
                for (int i = 0; i < L::OBJ + 1; i++) st[S::R + i] = lin[i];
                ist[IS_NJEV]++;
            }
            ist[IS_STATUS] = 0;
            return false;
        }
    }
    if (adopt) {
        BLSQ_UNROLL
        for (int i = 0; i < L::OBJ + 1; i++) st[S::R + i] = lin[i];
        ist[IS_NJEV]++;
    }
    if (first && 1 >= P.max_nfev) {
        st[S::GNORM] = dnan();
        ist[IS_STATUS] = 0;
        return false;
    }

    // ---- linearise (dogbox.py:165-199) ----
    double x[N], g[N], scale[N];
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) { x[i] = st[S::X + i]; g[i] = st[S::G + i]; }
    if (P.jac_scaling) {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            double nn = 0.0;
            BLSQ_UNROLL
            for (int i = 0; i <= j; i++) {
                double r = st[S::R + tri_index<N>(i, j)];
                nn = fma(r, r, nn);
            }
            double cn = sqrt(nn);
            if (first) {
                if (cn == 0) cn = 1.0;
                scale[j] = 1.0 / cn;
            } else {
                scale[j] = np_min(st[S::SCALE + j], 1.0 / cn);
            }
            st[S::SCALE + j] = scale[j];
        }
    } else if (first) {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            scale[j] = 1.0 / scaling[j];
            st[S::SCALE + j] = scale[j];
        }
    } else {
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) scale[j] = st[S::SCALE + j];
    }
    if (first) {
        double D0 = 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            double q = fabs(x0[i] / scale[i]);
            if (q > D0 || q != q) D0 = q;
        }
        st[S::DELTA] = (D0 == 0) ? 1.0 : D0;
    }
    int onb = ist[IS_ONB];
    bool free_[N];
    int nfree = 0, fr_bits = 0;
    double g_norm = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        free_[i] = !(get2(onb, i) * g[i] < 0);
        if (free_[i]) {
            nfree++;
            fr_bits |= 1 << i;
            double ga = fabs(g[i]);
            if (ga > g_norm || ga != ga) g_norm = ga;
        }
    }
    st[S::GNORM] = g_norm;           // all active -> 0.0 (dogbox.py:182-184)
    if (nfree == 0 || g_norm < P.gtol) status = 1;
    if (status != ST_RUNNING) {
        ist[IS_STATUS] = status;
        return false;
    }

    // newton_step = lstsq(J_free, -f) (dogbox.py:197): minimum-norm solution
    // through the SVD of R[:, free], singular values <= eps*max(m,n_free)*smax
    // dropped (numpy.linalg.lstsq rcond=None).
    double A[N * N], bq[N];
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        bq[i] = st[S::QTF + i];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++)
            A[i * N + j] = (j >= i && free_[j])
                               ? st[S::R + tri_index<N>(i, j)] : 0.0;
    }
    double newton[N], cauchy[N];
    // No variable on a bound and full rank certified (cond(R) <= |R|_F |R^-1|_F
    // with a factor 4 to spare against numpy's rcond = eps * max(m, n)): the
    // minimum-norm solution is the least-squares solution -R^-1 Q^T f and no
    // singular value is dropped -- no SVD needed (see gn_shortcut).
    if (!(nfree == N && gn_shortcut<N>(A, bq, P.m, dinf(), newton))) {
        jacobi_rows<N>(A, bq);          // rows: s_j v_j^T ; bq: U^T (Q^T f)
        double sv2[N], smax2 = 0.0;
        BLSQ_UNROLL
        for (int j = 0; j < N; j++) {
            double nn = 0.0;
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) nn = fma(A[j * N + i], A[j * N + i], nn);
            sv2[j] = nn;                 // s_j^2
            if (nn > smax2) smax2 = nn;
        }
        int mx = P.m > nfree ? P.m : nfree;
        double cut = EPS * mx * sqrt(smax2);
        double w[N];
        BLSQ_UNROLL
        for (int j = 0; j < N; j++)
            w[j] = (sqrt(sv2[j]) > cut) ? bq[j] / sv2[j] : 0.0;
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) {
            double acc = 0.0;
            BLSQ_UNROLL
            for (int j = 0; j < N; j++) acc = fma(A[j * N + i], w[j], acc);
            newton[i] = free_[i] ? -acc : 0.0;
        }
    }
    // cauchy = -(g.g)/(Jg.Jg) g  (dogbox.py:198-199), |J_free g| = |R g_free|
    double gf[N], Jg[N];
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) gf[i] = free_[i] ? g[i] : 0.0;
    tri_matvec<N>(st + S::R, gf, Jg);
    double cc = -dot<N>(gf, gf) / dot<N>(Jg, Jg);
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) cauchy[i] = cc * gf[i];

    // ---- propose (dogbox.py:203-223) ----
    double Delta = st[S::DELTA];
    double tr[N], lo[N], hi[N];
    int flags[N], hits[N], marks[N];
    bool tr_hit = false;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) tr[i] = Delta * scale[i];
    dog_box_geometry<N>(x, tr, l, u, free_, lo, hi, flags);
    double step[N];
    if (in_box<N>(newton, lo, hi, free_)) {
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) { step[i] = newton[i]; marks[i] = 0; }
    } else {
        double cz[N], zero[N], diff[N];
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) { cz[i] = cauchy[i]; zero[i] = 0.0; }
        if (!in_box<N>(cz, lo, hi, free_)) {
            double beta = step_to_box<N>(zero, cz, lo, hi, free_, hits);
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) cz[i] = beta * cz[i];
        }
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) diff[i] = newton[i] - cz[i];
        double t = step_to_box<N>(cz, diff, lo, hi, free_, hits);
        hit_bookkeeping<N>(hits, flags, free_, marks, tr_hit);
        BLSQ_UNROLL
        for (int i = 0; i < N; i++) step[i] = free_[i] ? cz[i] + t * diff[i] : 0.0;
    }
    // predicted reduction (dogbox.py:208-209): |J s|^2 = |R s|^2, Js.f = s.g
    double Js[N];
    tri_matvec<N>(st + S::R, step, Js);
    double JsJs = dot<N>(Js, Js);
    double Jsf = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) Jsf = fma(step[i], gf[i], Jsf);
    double pred = -JsJs - 2 * Jsf;
    if (pred <= 0) {
        // constrained_cauchy_step; the stale Js keeps pred <= 0 (Q-D3)
        if (in_box<N>(cauchy, lo, hi, free_)) {
            tr_hit = false;
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) { step[i] = cauchy[i]; marks[i] = 0; }
        } else {
            double zero[N];
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) zero[i] = 0.0;
            double beta = step_to_box<N>(zero, cauchy, lo, hi, free_, hits);
            hit_bookkeeping<N>(hits, flags, free_, marks, tr_hit);
            BLSQ_UNROLL
            for (int i = 0; i < N; i++) step[i] = free_[i] ? beta * cauchy[i] : 0.0;
        }
    }
    int mk = 0;
    double ns = 0.0;
    BLSQ_UNROLL
    for (int i = 0; i < N; i++) {
        mk |= put2(i, marks[i]);
        st[S::XNEW + i] = x[i] + step[i];
        double q = fabs(step[i] / scale[i]);
        if (q > ns || q != q) ns = q;
    }
    ist[IS_MARKS] = mk;
    ist[IS_FREE] = fr_bits | ((int)tr_hit << 30);
    st[S::PRED] = pred;
    st[S::NSTEP] = ns;
    return true;
}

// ---------------------------------------------------------------------------
// 2-point finite differences (least_squares.py:357-365 -> scipy _numdiff):
// step h for one coordinate after the bound adjustment.
// ---------------------------------------------------------------------------
BLSQ_HD double fd2_step(double x, double lb, double ub, double rel_step) {
    double sgn = (x >= 0) ? 1.0 : -1.0;
    double h_def = SQRT_EPS * sgn * np_max(1.0, fabs(x));
    double h = h_def;
    if (rel_step == rel_step) {               // user diff_step given
        h = rel_step * sgn * fabs(x);
        double dx = (x + h) - x;
        if (dx == 0) h = h_def;
    }
    // with lb=-inf, ub=+inf the adjustment below is the identity, which is
    // what scipy's "all bounds infinite" early return gives
    double below = x - lb, above = ub - x;
    double xp = x + h;
    bool violated = (xp < lb) || (xp > ub);
    bool fitting = fabs(h) <= np_max(below, above);
    double out = h;
    if (violated && fitting) out = -h;
    if (!fitting) out = (above >= below) ? above : -below;
    return out;
}

// 3-point scheme (scipy _compute_absolute_step + _adjust_scheme_to_bounds with
// '2-sided', num_steps = 1): central difference where both x - h and x + h fit,
// else a one-sided 3-point stencil x + h, x + 2h (h possibly negative and
// shrunk to half the room), else central again with h = the smaller distance.
BLSQ_HD double fd3_step(double x, double lb, double ub, double rel_step, bool& one_sided) {
    const double CBRT_EPS = 0x1.965fea53d6e41p-18;       // EPS ** (1 / 3), 6.055454452393343e-06
    double sgn = (x >= 0) ? 1.0 : -1.0;
    double h_def = CBRT_EPS * sgn * np_max(1.0, fabs(x));
    double h = h_def;
    if (rel_step == rel_step) {
        h = rel_step * sgn * fabs(x);
        double dx = (x + h) - x;
        if (dx == 0) h = h_def;
    }
    h = fabs(h);
    double below = x - lb, above = ub - x;
    bool central = (below >= h) && (above >= h);
    double out = h;
    one_sided = false;
    if (!central) {
        if (above >= below) { out = np_min(h, 0.5 * above); one_sided = true; }
        else { out = -np_min(h, 0.5 * below); one_sided = true; }
        double min_dist = np_min(above, below);
        if (fabs(out) <= min_dist) { out = min_dist; one_sided = false; }
    }
    return out;
}

}  // namespace blsq
