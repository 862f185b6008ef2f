// Batched mode, the linearisation kernel (HBM bound): QR of [J | f] per
// problem with the rows in registers.  A header so that a residual model can be
// compiled INTO the kernel (MODE 3, blsq_models.cu: J never touches HBM); the
// library's own instances (blsq_batched_n.cu, one object per N) use modes
// 0 - 2 with NoModel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "blsq_core.cuh"

namespace blsq_lin {
using namespace blsq;

// MODE 3 hook: fills a[0..N-1] (the row of J) and a[N] (the residual) of row
// `row` of problem `pid` (slot `slot` of the active set) in registers.
struct NoModel {
    template <int N>
    __device__ __forceinline__ void row(int64_t, int64_t, int, double (&)[N + 1]) const {}
};

// ---- build knobs (tools/kbench.py explores them) --------------------------
#ifndef BLSQ_LIN_THREADS
#define BLSQ_LIN_THREADS 128
#endif
#ifndef BLSQ_LIN_MINB
#define BLSQ_LIN_MINB 4
#endif

// rows per lane held in registers by lin_kernel, and the register budget:
// N <= 4: 8 rows x 5 columns at 128 registers (4 CTAs / SM); N = 5, 6: 8 rows
// x 7 columns at 168 registers (3 CTAs / SM) -- two problems per warp at
// m = 128 halve the shuffle/sqrt instructions per problem, which is what the
// kernel is bound by (profiles/r1_c3_lin_kernel_ncu.md); N = 7, 8: 4 rows.
#ifndef BLSQ_RPL_SMALL
#define BLSQ_RPL_SMALL 8
#endif
#ifndef BLSQ_RPL_MID
#define BLSQ_RPL_MID 8
#endif
#ifndef BLSQ_LIN_MINB_MID
#define BLSQ_LIN_MINB_MID 3
#endif
template <int N, bool WIDE = (N > 8)> struct LinCfg {
    static constexpr int RPL = (N <= 4) ? BLSQ_RPL_SMALL : (N <= 6 ? BLSQ_RPL_MID : 4);
    static constexpr int MINB = (N <= 4 || RPL <= 4) ? BLSQ_LIN_MINB : BLSQ_LIN_MINB_MID;
};
// N = 9..16 (lane groups of 16 / 32 only): 4 rows per lane up to N = 12,
// then 2, at 2 CTAs / SM (255 registers).  The largest
// budgets without spills in any of the 18 instances of an N: 4 rows at 3 CTAs
// spill 1.3-1.5 KB at N = 12 in MULTI, 4 rows spill at N = 16 even at 2 CTAs
// (profiles/r4_wide_ptxas.md).
#ifndef BLSQ_RPL_WIDE
#define BLSQ_RPL_WIDE 4
#endif
#ifndef BLSQ_RPL_WIDE_TO
#define BLSQ_RPL_WIDE_TO 12
#endif
#ifndef BLSQ_LIN_MINB_WIDE
#define BLSQ_LIN_MINB_WIDE 2
#endif
template <int N> struct LinCfg<N, true> {
    static constexpr int RPL = N <= BLSQ_RPL_WIDE_TO ? BLSQ_RPL_WIDE : 2;
    static constexpr int MINB = BLSQ_LIN_MINB_WIDE;
};

template <int G>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int off = G >> 1; off > 0; off >>= 1)
        v += __shfl_xor_sync(0xffffffffu, v, off, 32);
    return v;
}

// 1/sqrt(d), sqrt(d) and 1/d for the column norms of the Gram-Schmidt sweep
// from ONE reciprocal square root (MUFU.RSQ64H + Newton) instead of a double
// sqrt and a double division; each is within ~1 ulp.  d <= 0 -> zeros.
__device__ __forceinline__ void norm_terms(double d, double& r, double& inv_r, double& inv_d) {
    if (d > 0.0) {
        double y = rsqrt(d);
        double rr = d * y;
        rr = fma(fma(-rr, rr, d), 0.5 * y, rr);        // one Newton step on sqrt
        y = fma(fma(-rr, y, 1.0), y, y);               // and on 1/sqrt
        r = rr; inv_r = y; inv_d = y * y;
    } else {
        r = sqrt(d); inv_r = 0.0; inv_d = 0.0;         // 0 or NaN as before
    }
}

// a / b correctly rounded from y = 1 / b (itself correctly rounded): two
// residual corrections (Markstein).  The finite-difference quotients of scipy's
// _dense_difference are true divisions; with this J_fd is bit for bit NumPy's
// at 5 FMA-pipe instructions instead of a division subroutine per element.
__device__ __forceinline__ double div_rn(double a, double b, double y) {
    double q = a * y;
    q = fma(fma(-b, q, a), y, q);
    q = fma(fma(-b, q, a), y, q);
    return q;
}

// The lane-group class of lin_kernel for m rows: the smallest group whose
// registers hold all m rows, else 32 lanes that fold the rows in chunk by
// chunk (MULTI).  N > 8 has no 8-lane class: lane k stores row k of R.
// Returns launch(std::integral_constant<int, G>(), std::bool_constant<MULTI>()).
// The one place the class is chosen: the library's instances
// (batched_lin) and compiled user models (blsq_user_model.cuh) both use it.
template <int N, class Launch>
int lin_class(int m, Launch&& launch) {
    constexpr int RPL = LinCfg<N>::RPL;
    if constexpr (N <= 8) {
        if (m <= 8 * RPL)
            return launch(std::integral_constant<int, 8>(), std::false_type());
    }
    if (m <= 16 * RPL) return launch(std::integral_constant<int, 16>(), std::false_type());
    if (m <= 32 * RPL) return launch(std::integral_constant<int, 32>(), std::false_type());
    return launch(std::integral_constant<int, 32>(), std::true_type());
}

template <int N> struct PtrList { const double* p[2 * N]; };   // 2 per coordinate (3-point)

// Doubles per vector load of a row of J with n columns at row stride ldj: a
// row starts only as aligned as ldj * 8 bytes allows (J itself aligned to as
// many).  ldj == n gives the dense widths: 4 for n % 4 == 0, 2 for even n.
__host__ __device__ constexpr int lin_ld_width(int n, int ldj) {
    return (n % 4 == 0 && ldj % 4 == 0) ? 4 : ((n % 2 == 0 && ldj % 2 == 0) ? 2 : 1);
}

// One group of G lanes (G = 8, 16 or 32) per problem; row (base + s*G + lane)
// of the current chunk sits in a[s][*] of that lane.
// MODE 0: analytic J (A, m, n).  MODE 1: 2-point differences, Fpert.p[i] is
// F at the i-th perturbed batch, (A, m); dx is (A, n).  MODE 2: 3-point
// differences, Fpert.p[2i], p[2i+1] the two batches of coordinate i, dx is
// (A, 2n): denominators, then the one-sided flags (blsq_fd3_points).
// MULTI: m > G * RPL, the rows are folded in chunk by chunk with the running
// triangle carried in one extra register row; otherwise all rows are resident,
// g / f.f are reduced and written before the sweep and row k of the triangle
// is stored by lane k as soon as it exists (fewer live registers).
// ROWS: ragged batch, problem pid has rows[pid] (clamped to [0, m]) residuals
// and m is only the row stride of F / J / Fpert.  Rows past the count are
// never read and enter the sweep as zeros, exactly like the rows past m of a
// partial last chunk, so a ragged problem gets the record of a dense solve of
// its first rows[pid] residuals with the same lane group.  MULTI folds chunks
// only up to the problem's own count.  The dense path (ROWS = false) is a
// separate instance and compiles to the code it had before.
// LDW > 0 (MODE 0 with ROWS only): J is the (A, m, ldj) output of a batch
// padded to ldj > N parameters (least_squares_batched `cols`); the first N
// columns of each row are read with LDW-double vector loads
// (lin_ld_width(N, ldj)) and the others never are.  rows may be null there
// (every problem has m rows).  Otherwise the same instructions as the
// ROWS instance, so the record is that of a dense (A, m, N) Jacobian.
template <int N, int G, int MODE, bool MULTI, class MODEL = NoModel, bool ROWS = false,
          int LDW = 0>
__global__ void __launch_bounds__(BLSQ_LIN_THREADS, LinCfg<N>::MINB)
lin_kernel(int64_t A, const int32_t* __restrict__ idx, int m,
           const double* __restrict__ F, const double* __restrict__ J,
           PtrList<N> Fpert, const double* __restrict__ dx,
           const int32_t* __restrict__ istate, double* __restrict__ lin,
           MODEL mdl = MODEL(), const int32_t* __restrict__ rows = nullptr, int ldj = 0) {
    static_assert(LDW == 0 || (MODE == 0 && ROWS && N % LDW == 0), "LDW");
    // doubles per vector load of a row of J, and the row stride of J
    constexpr int VW = LDW ? LDW : (N % 4 == 0 ? 4 : (N % 2 == 0 ? 2 : 1));
    const int rs = LDW ? ldj : N;
    constexpr int RPL = LinCfg<N>::RPL;
    constexpr int C = N + 1;                      // columns of [J | f]
    constexpr int AR = MULTI ? RPL + 1 : RPL;     // + carried row of the triangle
    typedef LinRec<N> L;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t slot = tid / G;
    const int lane = (int)(tid % G);
    bool valid = slot < A;
    int64_t pid = 0;
    if (valid) {
        pid = idx ? idx[slot] : slot;
        valid = istate[pid * IS_SIZE + IS_STATUS] == ST_RUNNING;
    }
    if (!__any_sync(0xffffffffu, valid)) return;
    const bool all_valid = __all_sync(0xffffffffu, valid);
    // rows of this problem (ROWS; MULTI: G = 32, so the count is warp-uniform)
    int mp = m;
    if (ROWS && valid) {
        const int r = (LDW && !rows) ? m : rows[pid];
        mp = r < 0 ? 0 : (r > m ? m : r);
    }

    const double* Fp = (MODE == 3) ? nullptr : F + slot * (int64_t)m;
    const double* Jp = (MODE == 0) ? J + slot * (int64_t)m * rs : nullptr;
    double* out = lin + slot * (int64_t)L::SIZE;

    double a[AR][C];
    double myrow[MULTI ? C : 1];  // MULTI: row `lane` (< N) of the triangle, [.. | qtf]
    double gp[N], objp = 0.0;
#pragma unroll
    for (int j = 0; j < N; j++) gp[j] = 0.0;
    if (MULTI) {
#pragma unroll
        for (int j = 0; j < C; j++) { myrow[j] = 0.0; a[AR - 1][j] = 0.0; }
    }

    for (int base = 0; base < (MULTI ? mp : 1); base += G * RPL) {
        // warp-uniform: every group of the warp loads the whole chunk
        const bool full = ROWS ? __all_sync(0xffffffffu, valid && base + G * RPL <= mp)
                               : all_valid && (base + G * RPL <= m);
        // ---- load this chunk ----
        {
            double dxj[N], dxr[N];
            bool onej[N];
            if (MODE == 1) {
#pragma unroll
                for (int j = 0; j < N; j++) {
                    dxr[j] = valid ? dx[slot * N + j] : 1.0;
                    dxj[j] = 1.0 / dxr[j];                           // reciprocal once
                }
            }
            if (MODE == 2) {
#pragma unroll
                for (int j = 0; j < N; j++) {
                    dxr[j] = valid ? dx[slot * 2 * N + j] : 1.0;
                    dxj[j] = 1.0 / dxr[j];
                    onej[j] = valid ? dx[slot * 2 * N + N + j] != 0.0 : false;
                }
            }
#pragma unroll
            for (int s = 0; s < RPL; s++) {
                int row = base + s * G + lane;
                bool ok = full || (valid && row < mp);
                if (ok && MODE == 3) {
                    mdl.template row<N>(slot, pid, row, a[s]);
                } else if (ok) {
                    if (MODE == 0) {
                        const double* rp = Jp + (int64_t)row * rs;
                        if (VW == 4) {
                            // 256-bit streaming loads: a whole 32-byte sector per
                            // instruction and lane (rows of 4 / 8 doubles)
#pragma unroll
                            for (int j = 0; j < N; j += 4)
                                asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];"
                                             : "=d"(a[s][j]), "=d"(a[s][j + 1]),
                                               "=d"(a[s][j + 2]), "=d"(a[s][j + 3])
                                             : "l"(rp + j));
                        } else if (VW == 2) {
#pragma unroll
                            for (int j = 0; j < N; j += 2) {
                                double2 t = __ldcs(reinterpret_cast<const double2*>(rp + j));
                                a[s][j] = t.x;
                                a[s][j + 1] = t.y;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < N; j++) a[s][j] = __ldcs(rp + j);
                        }
                    } else if (MODE == 1) {
#pragma unroll
                        for (int j = 0; j < N; j++)
                            a[s][j] = __ldcs(Fpert.p[j] + slot * (int64_t)m + row);
                    }
                    a[s][N] = __ldcs(Fp + row);
                    if (MODE == 2) {
                        // scipy _dense_difference, '3-point': f2 - f1 (central) or
                        // -3 f0 + 4 f1 - f2 (one sided), in NumPy's evaluation order
                        const double f0 = a[s][N];
#pragma unroll
                        for (int j = 0; j < N; j++) {
                            const double f1 = __ldcs(Fpert.p[2 * j] + slot * (int64_t)m + row);
                            const double f2 = __ldcs(Fpert.p[2 * j + 1] + slot * (int64_t)m + row);
                            a[s][j] = onej[j] ? ((-3.0 * f0 + 4 * f1) - f2) : (f2 - f1);
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < C; j++) a[s][j] = 0.0;
                }
            }
            if (MODE == 1) {
                // scipy _dense_difference: J[:, i] = (f(x + h_i e_i) - f0) / dx_i,
                // the correctly rounded quotient (div_rn); rows that were not
                // loaded hold zeros: (0 - 0) / dx = 0
#pragma unroll
                for (int s = 0; s < RPL; s++) {
#pragma unroll
                    for (int j = 0; j < N; j++)
                        a[s][j] = div_rn(a[s][j] - a[s][N], dxr[j], dxj[j]);
                }
            }
            if (MODE == 2) {
#pragma unroll
                for (int s = 0; s < RPL; s++) {
#pragma unroll
                    for (int j = 0; j < N; j++) a[s][j] = div_rn(a[s][j], dxr[j], dxj[j]);
                }
            }
        }
        // ---- g = J^T f and f.f on the raw rows (trf.py:244, 229) ----
#pragma unroll
        for (int s = 0; s < RPL; s++) {
#pragma unroll
            for (int j = 0; j < N; j++) gp[j] = fma(a[s][j], a[s][N], gp[j]);
            objp = fma(a[s][N], a[s][N], objp);
        }
        if (!MULTI) {
            // all rows are here: finish g and f.f now and free their registers
#pragma unroll
            for (int j = 0; j < N; j++) {
                const double gj = group_sum<G>(gp[j]);
                if (valid && lane == j) out[L::G + j] = gj;
            }
            const double ob = group_sum<G>(objp);
            if (valid && lane == N % G) out[L::OBJ] = ob;
        }
        // ---- carry: row k of the running triangle lives on lane k ----
        if (MULTI) {
#pragma unroll
            for (int j = 0; j < C; j++) a[AR - 1][j] = (lane < N) ? myrow[j] : 0.0;
        }
        // ---- modified Gram-Schmidt on the stacked (carry + chunk) rows ----
#pragma unroll
        for (int k = 0; k < N; k++) {
            double dts[C];
#pragma unroll
            for (int j = k; j < C; j++) {
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < AR; s++) acc = fma(a[s][k], a[s][j], acc);
                dts[j] = group_sum<G>(acc);
            }
            double rkk, inv_rkk, inv_dk;
            norm_terms(dts[k], rkk, inv_rkk, inv_dk);
            // N > 8: with m << N, a column that depends on the ones before it
            // keeps only rounding residue, which shrinks by ~u per projection;
            // after ten of them its squared norm is subnormal and inv_dk = 1/d
            // overflows.  Such a column is treated as dependent, as d <= 0 is
            if (N > 8 && !(dts[k] >= 2.2250738585072014e-308)) {
                inv_rkk = 0.0;
                inv_dk = 0.0;
            }
            if (MULTI) {
                if (lane == k) {
#pragma unroll
                    for (int j = 0; j < C; j++) myrow[j] = 0.0;
                    myrow[k] = rkk;
                }
            } else if (valid && lane == k) {
                out[L::R + tri_index<N>(k, k)] = rkk;
            }
#pragma unroll
            for (int j = k + 1; j < C; j++) {
                const double coef = dts[j] * inv_dk;
                const double rkj = dts[j] * inv_rkk;
                if (MULTI) {
                    if (lane == k) myrow[j] = rkj;
                } else if (valid && lane == k) {
                    if (j < N) out[L::R + tri_index<N>(k, j)] = rkj;
                    else out[L::QTF + k] = rkj;
                }
#pragma unroll
                for (int s = 0; s < AR; s++)
                    a[s][j] = fma(-coef, a[s][k], a[s][j]);
            }
        }
    }
    if (MULTI) {
#pragma unroll
        for (int j = 0; j < N; j++) gp[j] = group_sum<G>(gp[j]);
        objp = group_sum<G>(objp);
        if (valid) {
            // lanes 0..N-1 write one row of the triangle each (+ their g, qtf)
#pragma unroll
            for (int k = 0; k < N; k++) {
                if (lane == k) {
#pragma unroll
                    for (int j = k; j < N; j++) out[L::R + tri_index<N>(k, j)] = myrow[j];
                    out[L::QTF + k] = myrow[N];
                    out[L::G + k] = gp[k];
                }
            }
            if (lane == N % G) out[L::OBJ] = objp;
        }
    }
}

}  // namespace blsq_lin
