// Batched mode: every lin_kernel and round_kernel instance of one parameter
// count N, chosen by -DBLSQ_N=<N>.  The Makefile builds this file once per
// N = 1..16, so make -j compiles the objects in parallel; the C ABI
// (blsq_batched.cu) reaches them through batched_lin<N> and batched_round<N>.
//
// lin_kernel for N > 8: lane groups of 16 or 32 only.  The all-rows-resident
// path stores row k of R, Q^T f[k] and g[k] from lane k, so a group needs at
// least N lanes; LinCfg<N, true> (blsq_lin.cuh) sets the rows per lane and
// registers.  round_kernel: the same per-thread code (blsq_core.cuh) for every N.
#include "blsq_batched_kernels.cuh"

#ifndef BLSQ_N
#error "compile with -DBLSQ_N=<1..16>"
#endif
static_assert(BLSQ_N >= 1 && BLSQ_N <= BLSQ_MAX_BATCHED_N, "BLSQ_N");

template <int N>
int batched_lin(int64_t A, const int32_t* idx, int m, int ldj, const double* F,
                const double* J, const double* const* Fp_host, const double* dx,
                int jac_mode, const int32_t* istate, double* lin,
                const int32_t* rows, cudaStream_t s) {
    PtrList<N> pl;
    const int np = jac_mode == 2 ? 2 * N : (jac_mode == 1 ? N : 0);
    for (int j = 0; j < 2 * N; j++) pl.p[j] = (j < np) ? Fp_host[j] : nullptr;
    // a ragged batch is classed by its width m, not by its counts
    return lin_class<N>(m, [&](auto g, auto multi) {
        return launch_lin_g<N, decltype(g)::value, decltype(multi)::value>(
            A, idx, m, ldj, F, J, pl, dx, jac_mode, istate, lin, rows, s);
    });
}

// rows == null: the dense instances; else the ragged ones (round_slot ROWS)
template <int N>
int batched_round(int method, int64_t A, const int32_t* idx, const double* lin,
                  const double* x0, const double* lb, const double* ub,
                  int bstride, const double* scaling, SolveParams P, int first,
                  double* state, int32_t* istate, double* Xnew, double* Xjac,
                  int32_t* work, int32_t* count, const int32_t* rows, cudaStream_t s) {
    if (rows)
        return launch_round_r<N, true>(method, A, idx, lin, x0, lb, ub, bstride, scaling, P,
                                       first, state, istate, Xnew, Xjac, work, count, rows, s);
    return launch_round_r<N, false>(method, A, idx, lin, x0, lb, ub, bstride, scaling, P,
                                    first, state, istate, Xnew, Xjac, work, count, nullptr, s);
}

template int batched_lin<BLSQ_N>(int64_t, const int32_t*, int, int, const double*,
                                 const double*, const double* const*, const double*, int,
                                 const int32_t*, double*, const int32_t*, cudaStream_t);
template int batched_round<BLSQ_N>(int, int64_t, const int32_t*, const double*,
                                   const double*, const double*, const double*, int,
                                   const double*, SolveParams, int, double*, int32_t*,
                                   double*, double*, int32_t*, int32_t*, const int32_t*,
                                   cudaStream_t);

#if defined(BLSQ_PHASE_CLOCKS) && BLSQ_N == 4
// tools/phase_probe.py only (it solves N = 4 problems): cycles [0..15] and
// visits [16..31] per phase of trf_round_impl since the last reset.  The
// counters are per object, so this reads the ones of the N = 4 round kernels.
extern "C" int blsq_debug_phase_read(unsigned long long* out, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out, blsq_phase_acc, sizeof(blsq_phase_acc));
    if (e == cudaSuccess && reset) {
        unsigned long long z[32] = {0};
        e = cudaMemcpyToSymbol(blsq_phase_acc, z, sizeof(z));
    }
    return (int)e;
}
#endif
