// Batched mode for 9..16 parameters per problem: the lin_kernel and
// round_kernel instances of one N, chosen by -DBLSQ_WIDE_N=<N> (the Makefile
// builds this file once per N, so the eight objects compile in parallel and
// blsq_batched.o keeps the code it had for N <= 8).  blsq_batched.cu
// dispatches to them from the C ABI entry points.
//
// lin_kernel: lane groups of 16 or 32 only.  The all-rows-resident path stores
// row k of R, Q^T f[k] and g[k] from lane k, so a group needs at least N
// lanes; LinCfg<N, true> (blsq_lin.cuh) sets the rows per lane and registers.
// round_kernel: the per-thread code of N <= 8 (blsq_core.cuh), unchanged.
#include "blsq_batched_kernels.cuh"

#ifndef BLSQ_WIDE_N
#error "compile with -DBLSQ_WIDE_N=<9..16>"
#endif
static_assert(BLSQ_WIDE_N >= 9 && BLSQ_WIDE_N <= BLSQ_MAX_BATCHED_N, "BLSQ_WIDE_N");

template <int N>
int wide_launch_lin(int64_t A, const int32_t* idx, int m, const double* F,
                    const double* J, const double* const* Fp_host, const double* dx,
                    int jac_mode, const int32_t* istate, double* lin,
                    const int32_t* rows, cudaStream_t s) {
    static_assert(N > 8 && N <= 16, "lane groups of 16 or 32 hold N <= 16 rows of R");
    return launch_lin<N>(A, idx, m, F, J, Fp_host, dx, jac_mode, istate, lin, rows, s);
}

template <int N>
int wide_launch_round(int method, int64_t A, const int32_t* idx, const double* lin,
                      const double* x0, const double* lb, const double* ub,
                      int bstride, const double* scaling, SolveParams P, int first,
                      double* state, int32_t* istate, double* Xnew, double* Xjac,
                      int32_t* work, int32_t* count, const int32_t* rows, cudaStream_t s) {
    return launch_round<N>(method, A, idx, lin, x0, lb, ub, bstride, scaling, P, first,
                           state, istate, Xnew, Xjac, work, count, rows, s);
}

template int wide_launch_lin<BLSQ_WIDE_N>(int64_t, const int32_t*, int, const double*,
                                          const double*, const double* const*,
                                          const double*, int, const int32_t*, double*,
                                          const int32_t*, cudaStream_t);
template int wide_launch_round<BLSQ_WIDE_N>(int, int64_t, const int32_t*, const double*,
                                            const double*, const double*, const double*,
                                            int, const double*, SolveParams, int, double*,
                                            int32_t*, double*, double*, int32_t*, int32_t*,
                                            const int32_t*, cudaStream_t);
