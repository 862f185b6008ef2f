// Fused residual/Jacobian kernels for the synthetic workloads (see
// include/blsq_models.h): user-side callbacks, one thread per residual.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/blsq.h"
#include "../../include/blsq_models.h"
#include "blsq_lin.cuh"

namespace {

// ExpDecay2 compiled INTO the linearisation kernel (lin_kernel MODE 3): the
// lanes evaluate their rows of f and J in registers -- same operation order
// as expdecay2_kernel, so the record is bit for bit the one the materialised
// path produces -- and the 2.5 KB of J and f per problem never touch HBM.
struct ExpDecay2Rows {
    const double* t;     // (m)
    const double* X;     // (A, 4) trial points, by slot
    const double* y;     // (B, m) data, by problem id
    int m;
    template <int N>
    __device__ __forceinline__ void row(int64_t slot, int64_t pid, int r, double (&a)[N + 1]) const {
        static_assert(N == 4, "ExpDecay2 has four parameters");
        const double4 x = *reinterpret_cast<const double4*>(X + slot * 4);
        const double tr = t[r];
        const double e1 = exp(-x.y * tr);
        const double e2 = exp(-x.w * tr);
        a[0] = e1;
        a[1] = -x.x * tr * e1;
        a[2] = e2;
        a[3] = -x.z * tr * e2;
        a[4] = x.x * e1 + x.z * e2 - __ldcs(y + pid * m + r);
    }
};

#ifndef BLSQ_EXPDECAY2_QUADS
#define BLSQ_EXPDECAY2_QUADS 1
#endif

// ROWS: ragged batch, problem pid has rows[pid] residuals (clamped to
// [0, m]); rows past the count are neither read nor written
template <bool ROWS>
__device__ __forceinline__ int model_rows(const int32_t* rows, int64_t pid, int m) {
    if (!ROWS) return m;
    const int r = rows[pid];
    return r < 0 ? 0 : (r > m ? m : r);
}

template <bool ROWS>
__global__ void __launch_bounds__(256)
expdecay2_kernel(int64_t A, const int64_t* __restrict__ idx, int m,
                 const double* __restrict__ t, const double* __restrict__ X,
                 const double* __restrict__ y, double* __restrict__ F,
                 double* __restrict__ J, const int32_t* __restrict__ rows) {
    // block = (rows, problems): no 64-bit division per element
    const int64_t s = (int64_t)blockIdx.x * blockDim.y + threadIdx.y;
    const int r = blockIdx.y * blockDim.x + threadIdx.x;
    if (s >= A || r >= m) return;
    const int64_t g = s * m + r;
    int64_t pid = idx ? idx[s] : s;
    if (ROWS && r >= model_rows<ROWS>(rows, pid, m)) return;
    const double4 x = *reinterpret_cast<const double4*>(X + s * 4);
    const double tr = t[r];
    // same operation order as synthetic.ExpDecay2.fun_t / jac_t
    const double e1 = exp(-x.y * tr);
    const double e2 = exp(-x.w * tr);
    F[g] = x.x * e1 + x.z * e2 - __ldcs(y + pid * m + r);
    if (J) {
        // one 256-bit streaming store per Jacobian row: a whole 32-byte sector
        // per thread (two 128-bit stores wrote half sectors at a 32-byte
        // stride, i.e. twice the write transactions)
        const double j1 = -x.x * tr * e1, j3 = -x.z * tr * e2;
        asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(J + g * 4), "d"(e1),
                     "d"(j1), "d"(e2), "d"(j3)
                     : "memory");
    }
}

// m % 4 == 0: one thread per (problem, four consecutive rows): 256-bit loads of
// t and y, one 256-bit store of F and four of J (128 contiguous bytes).  ROWS:
// the quad that straddles the problem's count stores only its rows below it
// (it reads all four: they lie inside the (A, m) buffers)
template <bool ROWS>
__global__ void __launch_bounds__(256)
expdecay2x4_kernel(int64_t A, const int64_t* __restrict__ idx, int m,
                   const double* __restrict__ t, const double* __restrict__ X,
                   const double* __restrict__ y, double* __restrict__ F,
                   double* __restrict__ J, const int32_t* __restrict__ rows) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.y + threadIdx.y;
    const int r = 4 * (blockIdx.y * blockDim.x + threadIdx.x);
    if (s >= A || r >= m) return;
    const int64_t g = s * m + r;
    const int64_t pid = idx ? idx[s] : s;
    const int nk = ROWS ? model_rows<ROWS>(rows, pid, m) - r : 4;   // rows of this quad
    if (ROWS && nk <= 0) return;
    const double4 x = *reinterpret_cast<const double4*>(X + s * 4);
    double tr[4], yv[4], f[4];
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(tr[0]), "=d"(tr[1]), "=d"(tr[2]), "=d"(tr[3])
                 : "l"(t + r));
    asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(yv[0]), "=d"(yv[1]), "=d"(yv[2]), "=d"(yv[3])
                 : "l"(y + pid * m + r));
#pragma unroll
    for (int k = 0; k < 4; k++) {
        // same operation order as synthetic.ExpDecay2.fun_t / jac_t
        const double e1 = exp(-x.y * tr[k]);
        const double e2 = exp(-x.w * tr[k]);
        f[k] = x.x * e1 + x.z * e2 - yv[k];
        if (J && (!ROWS || k < nk)) {
            const double j1 = -x.x * tr[k] * e1, j3 = -x.z * tr[k] * e2;
            asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(J + (g + k) * 4),
                         "d"(e1), "d"(j1), "d"(e2), "d"(j3)
                         : "memory");
        }
    }
    if (ROWS && nk < 4) {
        for (int k = 0; k < nk; k++) F[g + k] = f[k];
        return;
    }
    asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(F + g), "d"(f[0]), "d"(f[1]),
                 "d"(f[2]), "d"(f[3])
                 : "memory");
}

__global__ void __launch_bounds__(256)
gausspeak_kernel(int64_t A, const int64_t* __restrict__ idx, int m,
                 const double* __restrict__ t, const double* __restrict__ X,
                 const double* __restrict__ y, double* __restrict__ F) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.y + threadIdx.y;
    const int r = blockIdx.y * blockDim.x + threadIdx.x;
    if (s >= A || r >= m) return;
    const int64_t g = s * m + r;
    int64_t pid = idx ? idx[s] : s;
    const double* x = X + s * 6;
    const double tr = t[r];
    // same operation order as synthetic.GaussPeak.fun_t
    const double z = (tr - x[1]) / x[2];
    F[g] = x[0] * exp(-0.5 * z * z) + x[3] + x[4] * tr + x[5] * tr * tr -
           __ldcs(y + pid * m + r);
}

// m % 4 == 0: one thread per (problem, four consecutive rows) -- 256-bit
// loads of t and y, one 256-bit streaming store of F, and ONE reciprocal of
// sigma per thread: each quotient (t - mu) / sigma is the correctly rounded
// one from it (blsq_lin::div_rn, Markstein), i.e. the bits of the division
// the one-row kernel and torch perform, at 5 FMA-pipe instructions instead of
// a division subroutine per element.
__global__ void __launch_bounds__(256)
gausspeak4_kernel(int64_t A, const int64_t* __restrict__ idx, int m,
                  const double* __restrict__ t, const double* __restrict__ X,
                  const double* __restrict__ y, double* __restrict__ F) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.y + threadIdx.y;
    const int r = 4 * (blockIdx.y * blockDim.x + threadIdx.x);
    if (s >= A || r >= m) return;
    const int64_t pid = idx ? idx[s] : s;
    const double* x = X + s * 6;
    const double x0 = x[0], x1 = x[1], x2 = x[2], x3 = x[3], x4 = x[4], x5 = x[5];
    const double inv = 1.0 / x2;
    double tr[4], yv[4], f[4];
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(tr[0]), "=d"(tr[1]), "=d"(tr[2]), "=d"(tr[3])
                 : "l"(t + r));
    asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(yv[0]), "=d"(yv[1]), "=d"(yv[2]), "=d"(yv[3])
                 : "l"(y + pid * m + r));
#pragma unroll
    for (int k = 0; k < 4; k++) {
        // same operation order as synthetic.GaussPeak.fun_t
        const double z = blsq_lin::div_rn(tr[k] - x1, x2, inv);
        f[k] = x0 * exp(-0.5 * z * z) + x3 + x4 * tr[k] + x5 * tr[k] * tr[k] - yv[k];
    }
    asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(F + s * m + r), "d"(f[0]),
                 "d"(f[1]), "d"(f[2]), "d"(f[3])
                 : "memory");
}


// ---- tall workload (configs C4/C5): k = n - 4 linear columns + 2 exponentials --
// The Jacobian buffer J (m, n) holds the constant design matrix A in its
// first k columns, so the residual kernel reads A from there:
//   f = J[:, :k] x[:k] + x_k e^{-x_{k+1} t} + x_{k+2} e^{-x_{k+3} t} - y
// A warp takes 32 consecutive rows: each half warp streams 16 of them (16
// lanes per row, 16-byte loads, shuffle reduction, lane i keeps the sum of row
// i), then all 32 lanes evaluate the exponentials of their own row at once.
#ifndef BLSQ_FUN_UNROLL
#define BLSQ_FUN_UNROLL 16
#endif
constexpr int FUN_UNROLL = BLSQ_FUN_UNROLL;
#ifndef BLSQ_FUN_VARIANT
#define BLSQ_FUN_VARIANT 1
#endif
#ifndef BLSQ_FUN_RB
#define BLSQ_FUN_RB 4
#endif

__global__ void __launch_bounds__(256)
linexp_fun_kernel(int64_t m, int n, const double* __restrict__ J,
                  const double* __restrict__ t, const double* __restrict__ y,
                  const double* __restrict__ x, double* __restrict__ F) {
    __shared__ double xs[256];
    for (int i = threadIdx.x; i < n; i += blockDim.x) xs[i] = x[i];
    __syncthreads();
    const int k = n - 4;
    const int lane = threadIdx.x & 31, l16 = lane & 15, half = lane >> 4;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarp = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double xk = xs[k], xk1 = xs[k + 1], xk2 = xs[k + 2], xk3 = xs[k + 3];
    for (int64_t base = warp * 32; base < m; base += nwarp * 32) {
#if BLSQ_FUN_VARIANT == 1
        // RB rows of this half warp per batch: all their loads are issued
        // before the first reduction (rows past m are clamped, their sums are
        // never stored), then one transposing butterfly per batch
        constexpr int RB = BLSQ_FUN_RB;
        double mine = 0.0;
        const int64_t r0 = base + half * 16;
#pragma unroll
        for (int b0 = 0; b0 < 16; b0 += RB) {
            double s[RB];
#pragma unroll
            for (int i = 0; i < RB; i++) s[i] = 0.0;
            for (int c = 2 * l16; c < k; c += 32) {
                const double x0 = xs[c], x1 = xs[c + 1];
                double2 a[RB];
#pragma unroll
                for (int i = 0; i < RB; i++) {
                    int64_t r = r0 + b0 + i;
                    r = r < m ? r : m - 1;
                    a[i] = __ldcs(reinterpret_cast<const double2*>(J + r * n + c));
                }
#pragma unroll
                for (int i = 0; i < RB; i++) {
                    s[i] = fma(a[i].x, x0, s[i]);
                    s[i] = fma(a[i].y, x1, s[i]);
                }
            }
            // butterfly over the 16 lanes: the RB sums end up spread over the
            // lanes (lane j of every group of RB lanes holds row b0 + j)
#pragma unroll
            for (int off = 8; off >= RB; off >>= 1) {
#pragma unroll
                for (int i = 0; i < RB; i++) s[i] += __shfl_xor_sync(0xffffffffu, s[i], off, 16);
            }
#pragma unroll
            for (int off = RB / 2; off > 0; off >>= 1) {
                const bool up = (l16 & off) != 0;
#pragma unroll
                for (int i = 0; i < off; i++) {
                    const double send = up ? s[i] : s[i + off];
                    const double keep = up ? s[i + off] : s[i];
                    s[i] = keep + __shfl_xor_sync(0xffffffffu, send, off, 16);
                }
            }
            // lane l16 holds row b0 + (l16 % RB); lane (b0 + j) needs row b0 + j
            if ((l16 & ~(RB - 1)) == b0) mine = s[0];
        }
#else
        double mine = 0.0;
#pragma unroll FUN_UNROLL
        for (int it = 0; it < 16; it++) {
            const int64_t r = base + half * 16 + it;
            double s = 0.0;
            if (r < m) {
                const double* row = J + r * n;
                for (int c = 2 * l16; c < k; c += 32) {
                    const double2 a = __ldcs(reinterpret_cast<const double2*>(row + c));
                    s = fma(a.x, xs[c], s);
                    s = fma(a.y, xs[c + 1], s);
                }
            }
#pragma unroll
            for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off, 16);
            if (l16 == it) mine = s;
        }
#endif
        const int64_t r = base + lane;
        if (r < m) {
            const double tr = t[r];
            F[r] = mine + xk * exp(-xk1 * tr) + xk2 * exp(-xk3 * tr) - y[r];
        }
    }
}

// J[:, k..k+3] = [e1, -x_k t e1, e2, -x_{k+2} t e2]; the first k columns stay
__global__ void __launch_bounds__(256)
linexp_jac_kernel(int64_t m, int n, double* __restrict__ J, const double* __restrict__ t,
                  const double* __restrict__ x) {
    const int k = n - 4;
    const double xk = x[k], xk1 = x[k + 1], xk2 = x[k + 2], xk3 = x[k + 3];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < m; r += stride) {
        const double tr = t[r];
        const double e1 = exp(-xk1 * tr);
        const double e2 = exp(-xk3 * tr);
        double2* jp = reinterpret_cast<double2*>(J + r * n + k);
        jp[0] = make_double2(e1, -xk * tr * e1);
        jp[1] = make_double2(e2, -xk2 * tr * e2);
    }
}

// 256 threads as (rows of a problem, problems): x covers min(m, 256) rows
// rounded up to a warp, y the problems that fit beside it
bool batched_model_grid(int64_t A, int m, dim3& block, dim3& grid) {
    int bx = m < 256 ? ((m + 31) / 32) * 32 : 256;
    if (m < 32 && 32 % m == 0) bx = m;          // several problems per warp
    int by = 256 / bx;
    if (by < 1) by = 1;
    const int64_t gx = (A + by - 1) / by;
    const int64_t gy = (m + bx - 1) / bx;
    if (gx > 0x7fffffff || gy > 65535) return false;
    block = dim3(bx, by, 1);
    grid = dim3((unsigned)gx, (unsigned)gy, 1);
    return true;
}

}  // namespace

extern "C" {

int blsq_model_expdecay2_linearise(int64_t A, const int32_t* idx, int m, const double* t,
                                   const double* X, const double* y, const int32_t* istate,
                                   double* lin, void* stream) {
    using namespace blsq_lin;
    if (A < 0 || m < 1 || !t || !X || !y || !istate || !lin) return BLSQ_E_BADARG;
    if ((uintptr_t)X % 32) return BLSQ_E_BADARG;                // double4 loads of X
    if (m > 8 * LinCfg<4>::RPL) return BLSQ_E_UNSUPPORTED;      // all rows in one lane group
    if (A == 0) return 0;
    ExpDecay2Rows mdl{t, X, y, m};
    const int64_t blocks = (A * 8 + BLSQ_LIN_THREADS - 1) / BLSQ_LIN_THREADS;
    if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
    lin_kernel<4, 8, 3, false, ExpDecay2Rows><<<(unsigned)blocks, BLSQ_LIN_THREADS, 0,
                                                (cudaStream_t)stream>>>(
        A, idx, m, nullptr, nullptr, PtrList<4>(), nullptr, istate, lin, mdl);
    cudaError_t e_ = cudaGetLastError();
    if (e_ != cudaSuccess) return (int)e_;
    return 0;
}

int blsq_model_expdecay2_rows(int64_t A, const int64_t* idx, int m, const double* t,
                              const double* X, const double* y, const int32_t* rows,
                              double* F, double* J, void* stream) {
    if (A < 0 || m < 1 || !t || !X || !y || !F) return BLSQ_E_BADARG;
    // double4 loads of X and 256-bit stores of the rows of J in every variant
    if ((uintptr_t)X % 32 || (uintptr_t)J % 32) return BLSQ_E_BADARG;
    if (A == 0) return 0;
    dim3 block, grid;
    const bool quads = BLSQ_EXPDECAY2_QUADS && m % 4 == 0 && ((uintptr_t)t % 32 == 0) &&
                       ((uintptr_t)y % 32 == 0) && ((uintptr_t)F % 32 == 0);
    if (!batched_model_grid(A, quads ? m / 4 : m, block, grid)) return BLSQ_E_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    if (quads && rows)
        expdecay2x4_kernel<true><<<grid, block, 0, s>>>(A, idx, m, t, X, y, F, J, rows);
    else if (quads)
        expdecay2x4_kernel<false><<<grid, block, 0, s>>>(A, idx, m, t, X, y, F, J, nullptr);
    else if (rows)
        expdecay2_kernel<true><<<grid, block, 0, s>>>(A, idx, m, t, X, y, F, J, rows);
    else
        expdecay2_kernel<false><<<grid, block, 0, s>>>(A, idx, m, t, X, y, F, J, nullptr);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

int blsq_model_expdecay2(int64_t A, const int64_t* idx, int m, const double* t,
                         const double* X, const double* y, double* F, double* J,
                         void* stream) {
    return blsq_model_expdecay2_rows(A, idx, m, t, X, y, nullptr, F, J, stream);
}

int blsq_model_gausspeak(int64_t A, const int64_t* idx, int m, const double* t,
                         const double* X, const double* y, double* F,
                         void* stream) {
    if (A < 0 || m < 1 || !t || !X || !y || !F) return BLSQ_E_BADARG;
    if (A == 0) return 0;
    dim3 block, grid;
    // rows in fours when the row pointers stay 32-byte aligned
    const bool quads = m % 4 == 0 && ((uintptr_t)t % 32 == 0) && ((uintptr_t)y % 32 == 0) &&
                       ((uintptr_t)F % 32 == 0);
    if (!batched_model_grid(A, quads ? m / 4 : m, block, grid)) return BLSQ_E_UNSUPPORTED;
    if (quads)
        gausspeak4_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(A, idx, m, t, X, y, F);
    else
        gausspeak_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(A, idx, m, t, X, y, F);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}


int blsq_model_linexp_fun(int64_t m, int n, const double* J, const double* t,
                          const double* y, const double* x, double* F, void* stream) {
    if (m < 0 || n < 6 || n > 256 || (n & 1) || !J || !t || !y || !x || !F) return BLSQ_E_BADARG;
    if ((uintptr_t)J % 16) return BLSQ_E_BADARG;               // 128-bit loads of J
    if (m == 0) return 0;
    int64_t blocks = (m + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    linexp_fun_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(m, n, J, t, y, x, F);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

int blsq_model_linexp_jac(int64_t m, int n, double* J, const double* t, const double* x,
                          void* stream) {
    if (m < 0 || n < 6 || n > 256 || (n & 1) || !J || !t || !x) return BLSQ_E_BADARG;
    if ((uintptr_t)J % 16) return BLSQ_E_BADARG;               // 128-bit stores into J
    if (m == 0) return 0;
    int64_t blocks = (m + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    linexp_jac_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(m, n, J, t, x);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

}  // extern "C"
