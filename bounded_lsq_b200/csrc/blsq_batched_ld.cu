// Batched mode, ragged parameter counts: the lin_kernel instances that read the
// first N columns of a Jacobian padded to ldj > N columns (the (A, m, n)
// callback output of a least_squares_batched `cols` batch, read in place by
// each segment of N-parameter problems).  One object per N, chosen by
// -DBLSQ_LD_N=<N>, so that make -j compiles them in parallel and the objects
// of the dense instances keep their code.  Analytic Jacobians only: the
// finite-difference modes never read J.
#include "blsq_batched_kernels.cuh"

#ifndef BLSQ_LD_N
#error "compile with -DBLSQ_LD_N=<1..16>"
#endif
static_assert(BLSQ_LD_N >= 1 && BLSQ_LD_N <= BLSQ_MAX_BATCHED_N, "BLSQ_LD_N");

namespace {

template <int N, int G, bool MULTI, int W>
int launch_ld_w(unsigned blocks, int64_t A, const int32_t* idx, int m, int ldj,
                const double* F, const double* J, const int32_t* istate, double* lin,
                const int32_t* rows, cudaStream_t s) {
    lin_kernel<N, G, 0, MULTI, NoModel, true, W><<<blocks, BLSQ_LIN_THREADS, 0, s>>>(
        A, idx, m, F, J, PtrList<N>{}, nullptr, istate, lin, NoModel(), rows, ldj);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

// the vector width follows from N and ldj (lin_ld_width): an instance per width
template <int N, int G, bool MULTI>
int launch_ld_g(int64_t A, const int32_t* idx, int m, int ldj, const double* F,
                const double* J, const int32_t* istate, double* lin, const int32_t* rows,
                cudaStream_t s) {
    const int64_t blocks = (A * G + BLSQ_LIN_THREADS - 1) / BLSQ_LIN_THREADS;
    if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
    const int w = lin_ld_width(N, ldj);
    if constexpr (N % 4 == 0) {
        if (w == 4)
            return launch_ld_w<N, G, MULTI, 4>((unsigned)blocks, A, idx, m, ldj, F, J, istate,
                                               lin, rows, s);
    }
    if constexpr (N % 2 == 0) {
        if (w == 2)
            return launch_ld_w<N, G, MULTI, 2>((unsigned)blocks, A, idx, m, ldj, F, J, istate,
                                               lin, rows, s);
    }
    return launch_ld_w<N, G, MULTI, 1>((unsigned)blocks, A, idx, m, ldj, F, J, istate, lin,
                                       rows, s);
}

}  // namespace

// the lane-group class of launch_lin (from the width m)
template <int N>
int ld_launch_lin(int64_t A, const int32_t* idx, int m, int ldj, const double* F,
                  const double* J, const int32_t* istate, double* lin,
                  const int32_t* rows, cudaStream_t s) {
    constexpr int RPL = LinCfg<N>::RPL;
    if constexpr (N <= 8) {
        if (m <= 8 * RPL)
            return launch_ld_g<N, 8, false>(A, idx, m, ldj, F, J, istate, lin, rows, s);
    }
    if (m <= 16 * RPL)
        return launch_ld_g<N, 16, false>(A, idx, m, ldj, F, J, istate, lin, rows, s);
    if (m <= 32 * RPL)
        return launch_ld_g<N, 32, false>(A, idx, m, ldj, F, J, istate, lin, rows, s);
    return launch_ld_g<N, 32, true>(A, idx, m, ldj, F, J, istate, lin, rows, s);
}

template int ld_launch_lin<BLSQ_LD_N>(int64_t, const int32_t*, int, int, const double*,
                                      const double*, const int32_t*, double*,
                                      const int32_t*, cudaStream_t);
