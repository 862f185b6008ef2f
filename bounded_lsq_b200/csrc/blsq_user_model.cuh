// Residual models written by the user and compiled into the batched
// linearisation kernel (bounded_lsq_b200.models.compile_model).
//
// CONTRACT (version BLSQ_USER_MODEL_VERSION)
//
//   struct Model {                       // any name, given to compile_model
//       static constexpr int N = 6;      // parameters per problem, 1 .. 16
//       // residual r (0 <= r < c.m) of problem pid at the point x
//       __device__ double residual(const double (&x)[N], int64_t pid, int r,
//                                  const blsq_model_ctx& c) const;
//       // optional, enables the analytic kinds ('exact', 'inlined'):
//       // row r of the Jacobian, j[k] = d residual_r / d x_k
//       __device__ void jacobian_row(const double (&x)[N], int64_t pid, int r,
//                                    const blsq_model_ctx& c, double (&j)[N]) const;
//   };
//
// The residual may instead be a template on its scalar type,
//
//       template <class T>
//       __device__ T residual(const T (&x)[N], int64_t pid, int r,
//                             const blsq_model_ctx& c) const;
//
// written with the operations and functions blsq_dual.cuh lists.  Without a
// jacobian_row, the analytic kinds then derive the Jacobian row from it by
// forward-mode dual numbers (T = blsq_dual::Dual<N>); with T = double it is
// the residual.  An explicit jacobian_row always wins.
//
// The struct is default-constructed on the device and its functions must be
// pure: the same (x, pid, r, data) gives the same bits wherever it is
// evaluated.  c.data[k] is the k-th data tensor of the callbacks' `args`
// (float64, contiguous): a PerProblem tensor is indexed by the problem id pid
// (row pid of the whole batch, whatever the active set), a shared one is the
// same for every problem.  c.m is the number of residuals per problem.
//
// One source gives two routes to the same record (LinRec, blsq_lin.cuh):
//   materialised  fun writes F (A, m) = residual, jac writes J (A, m, N) =
//                 jacobian_row; blsq_linearise_batched then reads them (MODE 0
//                 with J, MODE 1 with the 2-point batches F(Xp[j])).
//   inlined       lin_kernel MODE 3 calls an adapter below for each of its
//                 rows: the row of [J | f] is formed in registers, J, F and the
//                 finite-difference batches never reach HBM.
// The file is compiled with the library's flags (-fmad=false, sm_100a): no
// operation is contracted differently where the functions are inlined, so
// both routes evaluate the same IEEE operations on the same inputs and the
// records agree bit for bit.  The 2-point adapter forms each quotient as
// MODE 1 does, div_rn(f(Xp[j]) - f, dx[j], 1.0 / dx[j]).  A derived
// Jacobian's dual evaluation gives f as its value channel, the bits of the
// double residual (blsq_dual.cuh), so a TRF row takes [J | f] from one
// evaluation.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>
#include <utility>

#include "../../include/blsq.h"
#include "blsq_dual.cuh"
#include "blsq_lin.cuh"

#define BLSQ_USER_MODEL_VERSION 1
#define BLSQ_MODEL_MAX_DATA 8

struct blsq_model_ctx {
    int m;                                     // residuals per problem
    const double* data[BLSQ_MODEL_MAX_DATA];   // the callbacks' data tensors, in args order
};

namespace blsq_um {
using blsq_lin::lin_kernel;
using blsq_lin::PtrList;

template <class M, class = void>
struct has_jacobian_row : std::false_type {};
template <class M>
struct has_jacobian_row<
    M, std::void_t<decltype(std::declval<const M&>().jacobian_row(
           std::declval<const double (&)[M::N]>(), int64_t(), int(),
           std::declval<const blsq_model_ctx&>(), std::declval<double (&)[M::N]>()))>>
    : std::true_type {};

template <class M, class = void>
struct has_dual_residual : std::false_type {};
template <class M>
struct has_dual_residual<
    M, std::enable_if_t<std::is_same<
           blsq_dual::Dual<M::N>,
           decltype(std::declval<const M&>().residual(
               std::declval<const blsq_dual::Dual<M::N> (&)[M::N]>(), int64_t(), int(),
               std::declval<const blsq_model_ctx&>()))>::value>> : std::true_type {};

// where a model's Jacobian comes from: 0 none, 1 jacobian_row, 2 derived from
// the templated residual (blsq_um_info's out[1])
template <class M>
constexpr int jac_source = has_jacobian_row<M>::value ? 1 : has_dual_residual<M>::value ? 2 : 0;

template <int N>
__device__ __forceinline__ void load_x(const double* __restrict__ p, double (&x)[N]) {
#pragma unroll
    for (int k = 0; k < N; k++) x[k] = p[k];
}

// Row r of the Jacobian at x into j, from jacobian_row or from one dual
// evaluation of the residual with x[k].d = e_k.  Returns the residual at x:
// the dual's value channel, or the double residual after jacobian_row (left
// unevaluated where the caller drops it).
template <class M>
__device__ __forceinline__ double jac_row(const M& mdl, const double (&x)[M::N], int64_t pid,
                                          int r, const blsq_model_ctx& c, double (&j)[M::N]) {
    constexpr int N = M::N;
    if constexpr (jac_source<M> == 1) {
        mdl.jacobian_row(x, pid, r, c, j);
        return mdl.residual(x, pid, r, c);
    } else {
        static_assert(jac_source<M> == 2, "the model has no Jacobian");
        blsq_dual::Dual<N> xd[N];
#pragma unroll
        for (int k = 0; k < N; k++) {
            xd[k].v = x[k];
            xd[k].d[k] = 1.0;
        }
        const blsq_dual::Dual<N> f = mdl.residual(xd, pid, r, c);
#pragma unroll
        for (int k = 0; k < N; k++) j[k] = f.d[k];
        return f.v;
    }
}

// MODE 3 analytic row: J at Xj (SPLIT, dogbox's bound-snapped point) or at X
// (TRF, one load of the point for both), f at X
template <class M, bool SPLIT>
struct AnalyticRows {
    blsq_model_ctx c;
    const double* X;    // (A, N) by slot
    const double* Xj;   // (A, N) by slot, SPLIT only
    template <int N>
    __device__ __forceinline__ void row(int64_t slot, int64_t pid, int r, double (&a)[N + 1]) const {
        static_assert(N == M::N, "N");
        const M mdl{};
        double x[N], j[N];
        load_x(X + slot * N, x);
        if (SPLIT) {
            double xj[N];
            load_x(Xj + slot * N, xj);
            jac_row(mdl, xj, pid, r, c, j);
            a[N] = mdl.residual(x, pid, r, c);
        } else {
            a[N] = jac_row(mdl, x, pid, r, c, j);
        }
#pragma unroll
        for (int k = 0; k < N; k++) a[k] = j[k];
    }
};

// MODE 3 2-point row: f at X, column k from f at Xp[k] (the (N, A, N) points
// of blsq_fd2_points) and the step dx[slot, k], as MODE 1 forms it
template <class M>
struct Fd2Rows {
    blsq_model_ctx c;
    const double* X;    // (A, N) by slot
    const double* Xp;   // (N, A, N)
    const double* dx;   // (A, N)
    int64_t A;
    template <int N>
    __device__ __forceinline__ void row(int64_t slot, int64_t pid, int r, double (&a)[N + 1]) const {
        static_assert(N == M::N, "N");
        const M mdl{};
        double x[N];
        load_x(X + slot * N, x);
        const double f0 = mdl.residual(x, pid, r, c);
#pragma unroll
        for (int k = 0; k < N; k++) {
            double xp[N];
            load_x(Xp + (k * A + slot) * N, xp);
            const double d = dx[slot * N + k];
            a[k] = blsq_lin::div_rn(mdl.residual(xp, pid, r, c) - f0, d, 1.0 / d);
        }
        a[N] = f0;
    }
};

template <class M>
__global__ void __launch_bounds__(256)
fun_kernel(int64_t A, const int64_t* __restrict__ idx, int m, const double* __restrict__ X,
           double* __restrict__ F, blsq_model_ctx c) {
    constexpr int N = M::N;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= A * m) return;
    const int64_t s = t / m;
    const int r = (int)(t - s * m);
    const int64_t pid = idx ? idx[s] : s;
    double x[N];
    load_x(X + s * N, x);
    F[t] = M{}.residual(x, pid, r, c);
}

template <class M>
__global__ void __launch_bounds__(256)
jac_kernel(int64_t A, const int64_t* __restrict__ idx, int m, const double* __restrict__ X,
           double* __restrict__ J, blsq_model_ctx c) {
    constexpr int N = M::N;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= A * m) return;
    const int64_t s = t / m;
    const int r = (int)(t - s * m);
    const int64_t pid = idx ? idx[s] : s;
    double x[N], j[N];
    load_x(X + s * N, x);
    jac_row(M{}, x, pid, r, c, j);
#pragma unroll
    for (int k = 0; k < N; k++) J[t * N + k] = j[k];
}

inline int launch_check() {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

inline int make_ctx(int m, const double* const* data, int ndata, blsq_model_ctx& c) {
    if (ndata < 0 || ndata > BLSQ_MODEL_MAX_DATA || (ndata && !data)) return BLSQ_E_BADARG;
    c.m = m;
    for (int k = 0; k < BLSQ_MODEL_MAX_DATA; k++) c.data[k] = k < ndata ? data[k] : nullptr;
    return 0;
}

// lin_kernel MODE 3 with the adapter `rows`, in the lane-group class that
// batched_lin<N> picks for m (blsq_lin.cuh lin_class)
template <int N, class Rows>
int launch_lin(int64_t A, const int32_t* idx, int m, const Rows& rows, const int32_t* istate,
               double* lin, cudaStream_t s) {
    return blsq_lin::lin_class<N>(m, [&](auto g, auto multi) -> int {
        constexpr int G = decltype(g)::value;
        const int64_t blocks = (A * G + BLSQ_LIN_THREADS - 1) / BLSQ_LIN_THREADS;
        if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
        lin_kernel<N, G, 3, decltype(multi)::value, Rows>
            <<<(unsigned)blocks, BLSQ_LIN_THREADS, 0, s>>>(
                A, idx, m, nullptr, nullptr, PtrList<N>(), nullptr, istate, lin, rows);
        return launch_check();
    });
}

// the entry points behind BLSQ_USER_MODEL_ENTRY_POINTS
template <class M>
int info(int* out) {
    out[0] = M::N;
    out[1] = jac_source<M>;
    out[2] = BLSQ_USER_MODEL_VERSION;
    return 0;
}

template <class M>
int linearise(int64_t A, const int32_t* idx, int m, const double* X, const double* Xj,
              const double* const* data, int ndata, const int32_t* istate, double* lin,
              void* stream) {
    if constexpr (jac_source<M> == 0) {
        return BLSQ_E_UNSUPPORTED;
    } else {
        blsq_model_ctx c;
        if (A < 0 || m < 1 || !X || !istate || !lin || make_ctx(m, data, ndata, c))
            return BLSQ_E_BADARG;
        if (A == 0) return 0;
        const cudaStream_t s = (cudaStream_t)stream;
        if (Xj && Xj != X)
            return launch_lin<M::N>(A, idx, m, AnalyticRows<M, true>{c, X, Xj}, istate, lin, s);
        return launch_lin<M::N>(A, idx, m, AnalyticRows<M, false>{c, X, nullptr}, istate, lin, s);
    }
}

template <class M>
int linearise_fd2(int64_t A, const int32_t* idx, int m, const double* X, const double* Xp,
                  const double* dx, const double* const* data, int ndata,
                  const int32_t* istate, double* lin, void* stream) {
    blsq_model_ctx c;
    if (A < 0 || m < 1 || !X || !Xp || !dx || !istate || !lin || make_ctx(m, data, ndata, c))
        return BLSQ_E_BADARG;
    if (A == 0) return 0;
    return launch_lin<M::N>(A, idx, m, Fd2Rows<M>{c, X, Xp, dx, A}, istate, lin,
                            (cudaStream_t)stream);
}

template <class M>
int fun(int64_t A, const int64_t* idx, int m, const double* X, const double* const* data,
        int ndata, double* F, void* stream) {
    blsq_model_ctx c;
    if (A < 0 || m < 1 || !X || !F || make_ctx(m, data, ndata, c)) return BLSQ_E_BADARG;
    if (A == 0) return 0;
    const int64_t blocks = (A * m + 255) / 256;
    if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
    fun_kernel<M><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(A, idx, m, X, F, c);
    return launch_check();
}

template <class M>
int jac(int64_t A, const int64_t* idx, int m, const double* X, const double* const* data,
        int ndata, double* J, void* stream) {
    if constexpr (jac_source<M> == 0) {
        return BLSQ_E_UNSUPPORTED;
    } else {
        blsq_model_ctx c;
        if (A < 0 || m < 1 || !X || !J || make_ctx(m, data, ndata, c)) return BLSQ_E_BADARG;
        if (A == 0) return 0;
        const int64_t blocks = (A * m + 255) / 256;
        if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
        jac_kernel<M><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(A, idx, m, X, J, c);
        return launch_check();
    }
}

}  // namespace blsq_um

// The C entry points of one compiled model (the generated source ends with
// this line).  Return codes as in include/blsq.h: 0, BLSQ_E_* (< 0) or a
// CUDA error (> 0).
#define BLSQ_USER_MODEL_ENTRY_POINTS(MODEL)                                                 \
    static_assert(MODEL::N >= 1 && MODEL::N <= BLSQ_MAX_BATCHED_N,                          \
                  "a compiled model has 1 .. 16 parameters (static constexpr int N)");      \
    extern "C" {                                                                            \
    int blsq_um_info(int* out) { return blsq_um::info<MODEL>(out); }                        \
    int blsq_um_linearise(int64_t A, const int32_t* idx, int m, const double* X,            \
                          const double* Xj, const double* const* data, int ndata,           \
                          const int32_t* istate, double* lin, void* stream) {               \
        return blsq_um::linearise<MODEL>(A, idx, m, X, Xj, data, ndata, istate, lin,        \
                                         stream);                                           \
    }                                                                                       \
    int blsq_um_linearise_fd2(int64_t A, const int32_t* idx, int m, const double* X,        \
                              const double* Xp, const double* dx,                           \
                              const double* const* data, int ndata,                         \
                              const int32_t* istate, double* lin, void* stream) {           \
        return blsq_um::linearise_fd2<MODEL>(A, idx, m, X, Xp, dx, data, ndata, istate,     \
                                             lin, stream);                                  \
    }                                                                                       \
    int blsq_um_fun(int64_t A, const int64_t* idx, int m, const double* X,                  \
                    const double* const* data, int ndata, double* F, void* stream) {        \
        return blsq_um::fun<MODEL>(A, idx, m, X, data, ndata, F, stream);                   \
    }                                                                                       \
    int blsq_um_jac(int64_t A, const int64_t* idx, int m, const double* X,                  \
                    const double* const* data, int ndata, double* J, void* stream) {        \
        return blsq_um::jac<MODEL>(A, idx, m, X, data, ndata, J, stream);                   \
    }                                                                                       \
    const char* blsq_um_error_string(int code) {                                            \
        return code > 0 ? cudaGetErrorString((cudaError_t)code)                             \
                        : (code == BLSQ_E_BADARG ? "invalid argument" : "unsupported");     \
    }                                                                                       \
    }
