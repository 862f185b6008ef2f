// Batched mode: the templated round kernel and the launchers of lin_kernel and
// round_kernel, shared by blsq_batched.cu (N = 1..8, and the C ABI) and
// blsq_batched_wide.cu (N = 9..16, one object per N so that make -j compiles
// them in parallel).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/blsq.h"
#include "blsq_core.cuh"
#include "blsq_lin.cuh"

using namespace blsq;
using namespace blsq_lin;

#define BLSQ_LAUNCH_CHECK()                                  \
    do {                                                     \
        cudaError_t e_ = cudaGetLastError();                 \
        if (e_ != cudaSuccess) return (int)e_;               \
    } while (0)

namespace {

#ifndef BLSQ_ROUND_THREADS
#define BLSQ_ROUND_THREADS 128
#endif
#ifndef BLSQ_ROUND_MINB
#define BLSQ_ROUND_MINB 4
#endif

// MODE 0: the whole round in one kernel.  TRF with a worklist (work != null):
// MODE 1 runs the round with the Gauss-Newton shortcut and appends the slots
// that need the SVD route to work[1..] (work[0] = their number); MODE 2 then
// finishes exactly those slots with dense warps (blsq_core.cuh trf_round_impl).
// 1: L2 prefetch of the TRF records at the top of the round (C2 full-batch
// round 0.248 -> 0.215 ms per 1e6 problems, profiles/r2_kbench_prefetch.jsonl).
// Measured against it and dropped: the same prefetch into L1 (no different), a
// one-wave grid striding over the slots and prefetching one slot ahead
// (0.313 ms), and staging both records through shared memory with 16-byte
// cp.async copies (0.266 ms).
#ifndef BLSQ_ROUND_PREFETCH
#define BLSQ_ROUND_PREFETCH 1
#endif
#if BLSQ_ROUND_PREFETCH == 2
#define BLSQ_PREFETCH(p) asm volatile("prefetch.global.L1 [%0];" ::"l"(p))
#else
#define BLSQ_PREFETCH(p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p))
#endif

template <int N, int METHOD, int MODE, bool ROWS>
__device__ __forceinline__ bool
round_slot(int64_t slot, int64_t A, const int32_t* __restrict__ idx,
           const double* __restrict__ lin, const double* __restrict__ x0,
           const double* __restrict__ lb, const double* __restrict__ ub,
           int bstride, const double* __restrict__ scaling, const SolveParams& P,
           int first, double* __restrict__ state,
           int32_t* __restrict__ istate, double* __restrict__ Xnew,
           double* __restrict__ Xjac, int32_t* __restrict__ work,
           const int32_t* __restrict__ rows) {
    typedef LinRec<N> L;
    constexpr int SS = (METHOD == BLSQ_METHOD_TRF) ? TrfState<N>::SIZE
                                                   : DogState<N>::SIZE;
    if (slot >= A) return false;
    const int64_t pid = idx ? idx[slot] : slot;
    int32_t* ip = istate + pid * IS_SIZE;
    // ROWS, a ragged batch: the decisions that use m (full_rank, the
    // Gauss-Newton certificate, dogbox's rcond) see this problem's own number
    // of rows.  A separate instance: a runtime test here costs the dense
    // TRF rounds spill traffic.
    SolveParams Pp = P;
    if (ROWS) {
        const int r = rows[pid];
        Pp.m = r < 0 ? 0 : (r > P.m ? P.m : r);
    }
    double sc[N];
#pragma unroll
    for (int i = 0; i < N; i++) sc[i] = scaling ? scaling[i] : 1.0;
    if (METHOD == BLSQ_METHOD_TRF) {
#if BLSQ_ROUND_PREFETCH
        // every line of the two records is requested NOW: the round reads them
        // block by block behind data-dependent branches, and at 16 warps per
        // SM one DRAM round trip per block is what the kernel waits for
        {
            const char* s0 = reinterpret_cast<const char*>(state + pid * (int64_t)SS);
            const char* l0 = reinterpret_cast<const char*>(lin + slot * (int64_t)L::SIZE);
#pragma unroll
            for (int o = 0; o < SS * 8; o += 128) BLSQ_PREFETCH(s0 + o);
#pragma unroll
            for (int o = 0; o < L::SIZE * 8; o += 128) BLSQ_PREFETCH(l0 + o);
            if (bstride) {
                BLSQ_PREFETCH(lb + pid * bstride);
                BLSQ_PREFETCH(ub + pid * bstride);
            }
        }
#endif
        // the records stay in memory: trf_round_impl fetches the blocks it
        // needs when it needs them (256-bit loads) and stores what changed
        int ist[4];
        {
            int4 t0 = *reinterpret_cast<const int4*>(ip);
            ist[0] = t0.x; ist[1] = t0.y; ist[2] = t0.z; ist[3] = t0.w;
        }
        if (ist[IS_STATUS] != ST_RUNNING) return false;
        const int rc = trf_round_impl<N, MODE>(
            state + pid * (int64_t)SS, ist, lin + slot * (int64_t)L::SIZE, x0 + pid * N,
            lb + pid * bstride, ub + pid * bstride, sc, Pp, first, Xnew + slot * N);
        *reinterpret_cast<int4*>(ip) = make_int4(ist[0], ist[1], ist[2], ist[3]);
        if (MODE == 1 && rc == TRF_DEFER)
            work[1 + atomicAdd(work, 1)] = (int32_t)slot;
        return ist[IS_STATUS] == ST_RUNNING;
    }
    constexpr int XNEW = N;
    int ist[IS_SIZE];
    {
        int4 t0 = *reinterpret_cast<const int4*>(ip);
        int4 t1 = *reinterpret_cast<const int4*>(ip + 4);
        ist[0] = t0.x; ist[1] = t0.y; ist[2] = t0.z; ist[3] = t0.w;
        ist[4] = t1.x; ist[5] = t1.y; ist[6] = t1.z; ist[7] = t1.w;
    }
    if (ist[IS_STATUS] != ST_RUNNING) return false;
    double st[SS];
    double* sp = state + pid * (int64_t)SS;
    if (SS % 2 == 0) {
#pragma unroll
        for (int i = 0; i < SS; i += 2) {
            double2 t = *reinterpret_cast<const double2*>(sp + i);
            st[i] = t.x;
            st[i + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < SS; i++) st[i] = sp[i];
    }
    double ln[L::SIZE];
    {
        const double* lp = lin + slot * (int64_t)L::SIZE;
#pragma unroll
        for (int i = 0; i < L::SIZE; i += 2) {
            double2 t = *reinterpret_cast<const double2*>(lp + i);
            ln[i] = t.x;
            ln[i + 1] = t.y;
        }
    }
    const bool go = dogbox_round<N>(st, ist, ln, x0 + pid * N, lb + pid * bstride,
                                    ub + pid * bstride, sc, Pp, first);
    if (SS % 2 == 0) {
#pragma unroll
        for (int i = 0; i < SS; i += 2)
            *reinterpret_cast<double2*>(sp + i) = make_double2(st[i], st[i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < SS; i++) sp[i] = st[i];
    }
    *reinterpret_cast<int4*>(ip) = make_int4(ist[0], ist[1], ist[2], ist[3]);
    *reinterpret_cast<int4*>(ip + 4) = make_int4(ist[4], ist[5], ist[6], ist[7]);
    if (go) {
#pragma unroll
        for (int i = 0; i < N; i++) Xnew[slot * N + i] = st[XNEW + i];
        if (Xjac) {
#pragma unroll
            for (int i = 0; i < N; i++) {
                double xj = st[XNEW + i];
                // the point dogbox.py:256-261 would evaluate J at
                int ob = ((ist[IS_FREE] >> i) & 1) ? get2(ist[IS_MARKS], i)
                                                   : get2(ist[IS_ONB], i);
                if (ob == -1) xj = lb[pid * bstride + i];
                if (ob == 1) xj = ub[pid * bstride + i];
                Xjac[slot * N + i] = xj;
            }
        }
    }
    return ist[IS_STATUS] == ST_RUNNING;
}

// CTAs per SM of the round kernel: TRF N <= 4 runs best at 4 x 128 threads
// (128 registers; 3 x 164 without spills measured 5 % slower), dogbox and the
// larger N at 2 (255 registers: C3, N = 6 dogbox, 0.60 ms per 10^6 problems at
// 4 CTAs, 0.50 at 3, 0.44 at 2 where it no longer spills).
template <int N, int METHOD> struct RoundCfg {
    static constexpr int MINB =
        (METHOD == BLSQ_METHOD_DOGBOX || N > 4) ? (BLSQ_ROUND_MINB > 2 ? 2 : BLSQ_ROUND_MINB)
                                                : BLSQ_ROUND_MINB;
};

template <int N, int METHOD, int MODE, bool ROWS>
__global__ void __launch_bounds__(BLSQ_ROUND_THREADS, (RoundCfg<N, METHOD>::MINB))
round_kernel(int64_t A, const int32_t* __restrict__ idx,
             const double* __restrict__ lin, const double* __restrict__ x0,
             const double* __restrict__ lb, const double* __restrict__ ub,
             int bstride, const double* __restrict__ scaling, SolveParams P,
             int first, double* __restrict__ state,
             int32_t* __restrict__ istate, double* __restrict__ Xnew,
             double* __restrict__ Xjac, int32_t* __restrict__ work,
             int32_t* __restrict__ count, const int32_t* __restrict__ rows) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (MODE == 2) {
        // the worklist length is only known on the device: a small grid
        // strides over it
        const int64_t cnt = work[0];
        for (int64_t w = tid; w < cnt; w += (int64_t)gridDim.x * blockDim.x)
            round_slot<N, METHOD, MODE, ROWS>(work[1 + w], A, idx, lin, x0, lb, ub, bstride, scaling,
                                        P, first, state, istate, Xnew, Xjac, work, rows);
        return;
    }
    const bool run = round_slot<N, METHOD, MODE, ROWS>(tid, A, idx, lin, x0, lb, ub, bstride, scaling,
                                                 P, first, state, istate, Xnew, Xjac, work, rows);
    if (!count) return;
    // running problems after this round: one atomic per CTA; the last CTA to
    // arrive publishes the total in count[2] and re-arms the two counters, so
    // the host needs no memset and no separate counting launch per round
    __shared__ int block_run;
    if (threadIdx.x == 0) block_run = 0;
    __syncthreads();
    const unsigned bal = __ballot_sync(0xffffffffu, run);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&block_run, __popc(bal));
    __syncthreads();
    if (threadIdx.x == 0) {
        if (block_run) atomicAdd(count, block_run);
        __threadfence();
        const int ticket = atomicAdd(count + 1, 1);
        if (ticket == (int)gridDim.x - 1) {
            __threadfence();
            count[2] = atomicExch(count, 0);
            count[1] = 0;
        }
    }
}

template <int N, int G, bool MULTI, bool ROWS>
int launch_lin_r(unsigned blocks, int64_t A, const int32_t* idx, int m, const double* F,
                 const double* J, const PtrList<N>& pl, const double* dx,
                 int jac_mode, const int32_t* istate, double* lin,
                 const int32_t* rows, cudaStream_t s) {
    if (jac_mode == 0)
        lin_kernel<N, G, 0, MULTI, NoModel, ROWS><<<blocks, BLSQ_LIN_THREADS, 0, s>>>(
            A, idx, m, F, J, pl, dx, istate, lin, NoModel(), rows);
    else if (jac_mode == 1)
        lin_kernel<N, G, 1, MULTI, NoModel, ROWS><<<blocks, BLSQ_LIN_THREADS, 0, s>>>(
            A, idx, m, F, J, pl, dx, istate, lin, NoModel(), rows);
    else
        lin_kernel<N, G, 2, MULTI, NoModel, ROWS><<<blocks, BLSQ_LIN_THREADS, 0, s>>>(
            A, idx, m, F, J, pl, dx, istate, lin, NoModel(), rows);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

// rows == null: the dense instances; else the ragged ones (lin_kernel ROWS)
template <int N, int G, bool MULTI>
int launch_lin_g(int64_t A, const int32_t* idx, int m, const double* F,
                 const double* J, const PtrList<N>& pl, const double* dx,
                 int jac_mode, const int32_t* istate, double* lin,
                 const int32_t* rows, cudaStream_t s) {
    int64_t threads = A * G;
    int64_t blocks = (threads + BLSQ_LIN_THREADS - 1) / BLSQ_LIN_THREADS;
    if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
    if (rows)
        return launch_lin_r<N, G, MULTI, true>((unsigned)blocks, A, idx, m, F, J, pl, dx,
                                               jac_mode, istate, lin, rows, s);
    return launch_lin_r<N, G, MULTI, false>((unsigned)blocks, A, idx, m, F, J, pl, dx,
                                            jac_mode, istate, lin, nullptr, s);
}

template <int N>
int launch_lin(int64_t A, const int32_t* idx, int m, const double* F,
               const double* J, const double* const* Fp_host, const double* dx,
               int jac_mode, const int32_t* istate, double* lin,
               const int32_t* rows, cudaStream_t s) {
    constexpr int RPL = LinCfg<N>::RPL;
    PtrList<N> pl;
    const int np = jac_mode == 2 ? 2 * N : (jac_mode == 1 ? N : 0);
    for (int j = 0; j < 2 * N; j++) pl.p[j] = (j < np) ? Fp_host[j] : nullptr;
    // smallest lane group whose registers hold all m rows (else 32 + chunks);
    // a ragged batch is classed by its width m, not by its counts.  N > 8
    // has no 8-lane class: lane k stores row k of R (lin_kernel)
    if constexpr (N <= 8) {
        if (m <= 8 * RPL)
            return launch_lin_g<N, 8, false>(A, idx, m, F, J, pl, dx, jac_mode, istate, lin,
                                             rows, s);
    }
    if (m <= 16 * RPL)
        return launch_lin_g<N, 16, false>(A, idx, m, F, J, pl, dx, jac_mode, istate, lin, rows, s);
    if (m <= 32 * RPL)
        return launch_lin_g<N, 32, false>(A, idx, m, F, J, pl, dx, jac_mode, istate, lin, rows, s);
    return launch_lin_g<N, 32, true>(A, idx, m, F, J, pl, dx, jac_mode, istate, lin, rows, s);
}

template <int N, bool ROWS>
int launch_round_r(int method, int64_t A, const int32_t* idx, const double* lin,
                 const double* x0, const double* lb, const double* ub,
                 int bstride, const double* scaling, SolveParams P, int first,
                 double* state, int32_t* istate, double* Xnew, double* Xjac,
                 int32_t* work, int32_t* count, const int32_t* rows, cudaStream_t s) {
    int64_t blocks = (A + BLSQ_ROUND_THREADS - 1) / BLSQ_ROUND_THREADS;
    if (blocks > 0x7fffffff) return BLSQ_E_UNSUPPORTED;
    const unsigned gb = (unsigned)blocks;
    if (method == BLSQ_METHOD_TRF && work) {
        cudaError_t e = cudaMemsetAsync(work, 0, sizeof(int32_t), s);
        if (e != cudaSuccess) return (int)e;
        round_kernel<N, BLSQ_METHOD_TRF, 1, ROWS><<<gb, BLSQ_ROUND_THREADS, 0, s>>>(
            A, idx, lin, x0, lb, ub, bstride, scaling, P, first, state, istate, Xnew, Xjac, work,
            count, rows);
        BLSQ_LAUNCH_CHECK();
        // ~5 % of the problems land on the worklist: an eighth of the grid
        // (at least 4 CTAs per SM) strides over it
        unsigned g2 = gb / 8 > 592u ? gb / 8 : (gb < 592u ? gb : 592u);
        round_kernel<N, BLSQ_METHOD_TRF, 2, ROWS><<<g2, BLSQ_ROUND_THREADS, 0, s>>>(
            A, idx, lin, x0, lb, ub, bstride, scaling, P, first, state, istate, Xnew, Xjac, work,
            nullptr, rows);
    } else if (method == BLSQ_METHOD_TRF) {
        round_kernel<N, BLSQ_METHOD_TRF, 0, ROWS><<<gb, BLSQ_ROUND_THREADS, 0, s>>>(
            A, idx, lin, x0, lb, ub, bstride, scaling, P, first, state, istate, Xnew, Xjac, work,
            count, rows);
    } else {
        round_kernel<N, BLSQ_METHOD_DOGBOX, 0, ROWS><<<gb, BLSQ_ROUND_THREADS, 0, s>>>(
            A, idx, lin, x0, lb, ub, bstride, scaling, P, first, state, istate, Xnew, Xjac, work,
            count, rows);
    }
    BLSQ_LAUNCH_CHECK();
    return 0;
}

// rows == null: the dense instances; else the ragged ones (round_slot ROWS)
template <int N>
int launch_round(int method, int64_t A, const int32_t* idx, const double* lin,
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

}  // namespace

// lin_kernel for a Jacobian padded to ldj > N columns (blsq_linearise_batched_ld),
// defined in blsq_batched_ld.cu, one object per N
template <int N>
int ld_launch_lin(int64_t A, const int32_t* idx, int m, int ldj, const double* F,
                  const double* J, const int32_t* istate, double* lin,
                  const int32_t* rows, cudaStream_t s);

// the instances for N = 9..16, defined in blsq_batched_wide.cu
template <int N>
int wide_launch_lin(int64_t A, const int32_t* idx, int m, const double* F,
                    const double* J, const double* const* Fp_host, const double* dx,
                    int jac_mode, const int32_t* istate, double* lin,
                    const int32_t* rows, cudaStream_t s);
template <int N>
int wide_launch_round(int method, int64_t A, const int32_t* idx, const double* lin,
                      const double* x0, const double* lb, const double* ub,
                      int bstride, const double* scaling, SolveParams P, int first,
                      double* state, int32_t* istate, double* Xnew, double* Xjac,
                      int32_t* work, int32_t* count, const int32_t* rows, cudaStream_t s);
