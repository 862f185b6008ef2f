// Batched mode kernels + C ABI (include/blsq.h) for sm_100a.
//
// Two kernels per round of the lock-step solve:
//
//   lin_kernel    HBM-bound.  A group of 8/16/32 lanes owns one problem; the
//                 lanes stream the rows of [J | f] with coalesced vector loads
//                 straight into registers and run a modified Gram-Schmidt QR
//                 with f as the last column, dot products reduced by warp
//                 shuffles inside the group.  Output per problem: packed R,
//                 Q^T f, g = J^T f, f.f  (a few hundred bytes).
//   round_kernel  FP64-bound.  One thread owns one problem and runs the whole
//                 n x n tail in registers (blsq_core.cuh): ratio test, accept,
//                 Coleman-Li scaling, SVD, LM parameter, candidates, select.
//
// Reference lines each stage stands in for are cited in blsq_core.cuh and
// include/blsq.h.
#include "blsq_batched_kernels.cuh"

namespace {

__global__ void init_kernel(int method, int64_t B, int n, int SS, int XNEW,
                            const double* __restrict__ x0,
                            const double* __restrict__ lb,
                            const double* __restrict__ ub, int bstride,
                            double* __restrict__ state,
                            int32_t* __restrict__ istate,
                            double* __restrict__ Xnew) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * n) return;
    int64_t b = t / n;
    int i = (int)(t % n);
    double x = x0[t];
    if (method == BLSQ_METHOD_TRF)
        x = strictly_feasible(x, lb[b * bstride + i], ub[b * bstride + i], 1e-10);
    state[b * SS + XNEW + i] = x;
    state[b * SS + i] = x;              // X
    Xnew[t] = x;
    if (i == 0) {
        int32_t* ip = istate + b * IS_SIZE;
        ip[IS_STATUS] = ST_RUNNING;
#pragma unroll
        for (int k = 1; k < IS_SIZE; k++) ip[k] = 0;
    }
}

__global__ void on_bound_kernel(int64_t B, int n,
                                const int32_t* __restrict__ istate,
                                int64_t* __restrict__ mask) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * n) return;
    int64_t b = t / n;
    int i = (int)(t % n);
    mask[t] = get2(istate[b * IS_SIZE + IS_ONB], i);
}

__global__ void count_running_kernel(int64_t B,
                                     const int32_t* __restrict__ idx,
                                     const int32_t* __restrict__ istate,
                                     int32_t* __restrict__ count) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool run = false;
    if (t < B) {
        int64_t pid = idx ? idx[t] : t;
        run = istate[pid * IS_SIZE + IS_STATUS] == ST_RUNNING;
    }
    unsigned bal = __ballot_sync(0xffffffffu, run);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(count, __popc(bal));
}


// ---- ordered compaction of the active set (three small launches) ------------
// Slot s (problem idx[s], or s) survives when its problem is still running;
// survivors keep their order.  Each block owns CMP_SLOTS consecutive slots.
constexpr int CMP_THREADS = 256;
constexpr int CMP_PER = 4;
constexpr int CMP_SLOTS = CMP_THREADS * CMP_PER;

__device__ __forceinline__ int compact_local(int64_t A, const int32_t* __restrict__ idx,
                                             const int32_t* __restrict__ istate,
                                             int64_t base, bool (&keep)[CMP_PER],
                                             int64_t (&pid)[CMP_PER], int& block_total) {
    __shared__ int wsum[CMP_THREADS / 32];
    int c = 0;
#pragma unroll
    for (int j = 0; j < CMP_PER; j++) {
        const int64_t s = base + (int64_t)threadIdx.x * CMP_PER + j;
        keep[j] = false;
        pid[j] = 0;
        if (s < A) {
            pid[j] = idx ? idx[s] : s;
            keep[j] = istate[pid[j] * IS_SIZE + IS_STATUS] == ST_RUNNING;
        }
        c += keep[j];
    }
    // exclusive scan of c over the block
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = c;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < CMP_THREADS / 32; w++) {
        const int v = wsum[w];
        if (w < warp) before += v;
        total += v;
    }
    block_total = total;
    return before + inc - c;
}

__global__ void __launch_bounds__(CMP_THREADS)
compact_count_kernel(int64_t A, const int32_t* __restrict__ idx,
                     const int32_t* __restrict__ istate, int32_t* __restrict__ bsum) {
    bool keep[CMP_PER];
    int64_t pid[CMP_PER];
    int total;
    compact_local(A, idx, istate, (int64_t)blockIdx.x * CMP_SLOTS, keep, pid, total);
    if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// exclusive scan of the block totals by one block (serial chunks per thread)
__global__ void __launch_bounds__(1024)
compact_scan_kernel(int nblocks, int32_t* __restrict__ bsum) {
    __shared__ int part[1024];
    const int per = (nblocks + 1023) / 1024;
    const int b0 = threadIdx.x * per;
    int s = 0;
    for (int k = 0; k < per; k++)
        if (b0 + k < nblocks) s += bsum[b0 + k];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int t = 0; t < 1024; t++) { const int v = part[t]; part[t] = run; run += v; }
        bsum[nblocks] = run;            // the number of survivors, for the host
    }
    __syncthreads();
    int run = part[threadIdx.x];
    for (int k = 0; k < per; k++)
        if (b0 + k < nblocks) { const int v = bsum[b0 + k]; bsum[b0 + k] = run; run += v; }
}

__global__ void __launch_bounds__(CMP_THREADS)
compact_scatter_kernel(int64_t A, const int32_t* __restrict__ idx,
                       const int32_t* __restrict__ istate, int n,
                       const int32_t* __restrict__ boff,
                       const double* __restrict__ Xnew, const double* __restrict__ Xjac,
                       int32_t* __restrict__ idx_out, int64_t* __restrict__ idx64_out,
                       double* __restrict__ Xnew_out, double* __restrict__ Xjac_out) {
    bool keep[CMP_PER];
    int64_t pid[CMP_PER];
    int total;
    const int64_t base = (int64_t)blockIdx.x * CMP_SLOTS;
    int pos = boff[blockIdx.x] + compact_local(A, idx, istate, base, keep, pid, total);
#pragma unroll
    for (int j = 0; j < CMP_PER; j++) {
        if (!keep[j]) continue;
        const int64_t s = base + (int64_t)threadIdx.x * CMP_PER + j;
        idx_out[pos] = (int32_t)pid[j];
        if (idx64_out) idx64_out[pos] = pid[j];
        for (int i = 0; i < n; i++) {
            Xnew_out[(int64_t)pos * n + i] = Xnew[s * n + i];
            if (Xjac) Xjac_out[(int64_t)pos * n + i] = Xjac[s * n + i];
        }
        pos++;
    }
}

// ---- padded trial batches of a ragged-parameter batch (blsq_pad_points) ------
struct PadTable {
    blsq_pad_segment seg[BLSQ_MAX_BATCHED_N];
    int nseg;
};

// one thread per (batch p, slot, coordinate k) of out (P, A, n)
__global__ void pad_points_kernel(PadTable tab, int64_t A, int n, int fd,
                                  double* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t P = fd ? (int64_t)fd * n : 1;
    if (t >= P * A * n) return;
    const int k = (int)(t % n);
    const int64_t slot = (t / n) % A;
    const int p = (int)(t / ((int64_t)n * A));
    int j = 0;
    while (j + 1 < tab.nseg && slot >= tab.seg[j + 1].off) j++;
    const blsq_pad_segment& g = tab.seg[j];
    const int64_t s = slot - g.off;
    double v;
    if (k >= g.n)
        v = g.x0[(g.idx ? (int64_t)g.idx[s] : s) * n + k];      // held fixed
    else if (fd && p < fd * g.n)
        v = g.Xp[((int64_t)p * g.A + s) * g.n + k];             // its own FD point
    else
        v = g.X[s * g.n + k];
    out[t] = v;
}

}  // namespace

#ifdef BLSQ_ONLY_N46      /* quick builds for tools/build_variants.sh */
#define BLSQ_DISPATCH_N(n, CALL)          \
    switch (n) {                          \
        case 4: { constexpr int N_ = 4; CALL; } break; \
        case 6: { constexpr int N_ = 6; CALL; } break; \
        default: return BLSQ_E_UNSUPPORTED; \
    }
#else
#define BLSQ_DISPATCH_N(n, CALL)          \
    switch (n) {                          \
        case 1: { constexpr int N_ = 1; CALL; } break; \
        case 2: { constexpr int N_ = 2; CALL; } break; \
        case 3: { constexpr int N_ = 3; CALL; } break; \
        case 4: { constexpr int N_ = 4; CALL; } break; \
        case 5: { constexpr int N_ = 5; CALL; } break; \
        case 6: { constexpr int N_ = 6; CALL; } break; \
        case 7: { constexpr int N_ = 7; CALL; } break; \
        case 8: { constexpr int N_ = 8; CALL; } break; \
        case 9: { constexpr int N_ = 9; CALL; } break; \
        case 10: { constexpr int N_ = 10; CALL; } break; \
        case 11: { constexpr int N_ = 11; CALL; } break; \
        case 12: { constexpr int N_ = 12; CALL; } break; \
        case 13: { constexpr int N_ = 13; CALL; } break; \
        case 14: { constexpr int N_ = 14; CALL; } break; \
        case 15: { constexpr int N_ = 15; CALL; } break; \
        case 16: { constexpr int N_ = 16; CALL; } break; \
        default: return BLSQ_E_UNSUPPORTED; \
    }
#endif

namespace {

// N = 9..16 are compiled in blsq_batched_wide.cu (one object per N)
template <int N>
int dispatch_lin(int64_t A, const int32_t* idx, int m, const double* F,
                 const double* J, const double* const* Fp_host, const double* dx,
                 int jac_mode, const int32_t* istate, double* lin,
                 const int32_t* rows, cudaStream_t s) {
    if constexpr (N <= 8)
        return launch_lin<N>(A, idx, m, F, J, Fp_host, dx, jac_mode, istate, lin, rows, s);
    else
        return wide_launch_lin<N>(A, idx, m, F, J, Fp_host, dx, jac_mode, istate, lin, rows, s);
}

template <int N>
int dispatch_round(int method, int64_t A, const int32_t* idx, const double* lin,
                   const double* x0, const double* lb, const double* ub,
                   int bstride, const double* scaling, SolveParams P, int first,
                   double* state, int32_t* istate, double* Xnew, double* Xjac,
                   int32_t* work, int32_t* count, const int32_t* rows, cudaStream_t s) {
    if constexpr (N <= 8)
        return launch_round<N>(method, A, idx, lin, x0, lb, ub, bstride, scaling, P, first,
                               state, istate, Xnew, Xjac, work, count, rows, s);
    else
        return wide_launch_round<N>(method, A, idx, lin, x0, lb, ub, bstride, scaling, P,
                                    first, state, istate, Xnew, Xjac, work, count, rows, s);
}

}  // namespace

extern "C" {

int blsq_state_layout(int method, int n, int* out) {
    if (!out) return BLSQ_E_BADARG;
    if (method != BLSQ_METHOD_TRF && method != BLSQ_METHOD_DOGBOX) return BLSQ_E_BADARG;
    BLSQ_DISPATCH_N(n, {
        if (method == BLSQ_METHOD_TRF) {
            typedef TrfState<N_> S;
            out[0] = S::SIZE; out[1] = S::X; out[2] = S::XNEW; out[3] = S::SCALE;
            out[4] = S::OBJ; out[5] = S::DELTA; out[6] = S::GNORM; out[7] = S::G;
            out[8] = S::ALPHA;
        } else {
            typedef DogState<N_> S;
            out[0] = S::SIZE; out[1] = S::X; out[2] = S::XNEW; out[3] = S::SCALE;
            out[4] = S::OBJ; out[5] = S::DELTA; out[6] = S::GNORM; out[7] = S::G;
            out[8] = -1;
        }
    });
    return 0;
}

int blsq_lin_record_size(int n) {
    BLSQ_DISPATCH_N(n, { return LinRec<N_>::SIZE; });
    return BLSQ_E_UNSUPPORTED;
}

int blsq_init_batched(int method, int64_t B, int n, const double* x0,
                      const double* lb, const double* ub, int bstride,
                      double* state, int32_t* istate, double* Xnew,
                      void* stream) {
    if (B < 0 || !x0 || !lb || !ub || !state || !istate || !Xnew) return BLSQ_E_BADARG;
    if (bstride != 0 && bstride != n) return BLSQ_E_BADARG;
    int lay[9];
    int rc = blsq_state_layout(method, n, lay);
    if (rc) return rc;
    if (B == 0) return 0;
    int64_t blocks = (B * n + 255) / 256;
    init_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        method, B, n, lay[0], lay[2], x0, lb, ub, bstride, state, istate, Xnew);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

int blsq_linearise_batched_rows(int64_t A, const int32_t* idx, int m, int n,
                                const double* F, const double* J,
                                const double* const* Fp_host, const double* dx,
                                int jac_mode, const int32_t* istate, double* lin,
                                const int32_t* rows, void* stream) {
    if (A < 0 || m < 1 || !F || !istate || !lin) return BLSQ_E_BADARG;
    if (jac_mode < 0 || jac_mode > 2) return BLSQ_E_BADARG;
    if (jac_mode == 0 && !J) return BLSQ_E_BADARG;
    // lin_kernel loads the rows of J with 256-bit (n % 4 == 0) or 128-bit
    // (n = 2, 6, 10, 14) vector loads: a misaligned J would fault the device
    if (jac_mode == 0 && (uintptr_t)J % (8 * lin_ld_width(n, n))) return BLSQ_E_BADARG;
    if (jac_mode != 0 && (!dx || !Fp_host)) return BLSQ_E_BADARG;
    if (jac_mode != 0 && n >= 1 && n <= BLSQ_MAX_BATCHED_N)
        for (int j = 0; j < jac_mode * n; j++)
            if (!Fp_host[j]) return BLSQ_E_BADARG;
    if (A == 0) return 0;
    BLSQ_DISPATCH_N(n, {
        return dispatch_lin<N_>(A, idx, m, F, J, Fp_host, dx, jac_mode, istate,
                                lin, rows, (cudaStream_t)stream);
    });
    return 0;
}

int blsq_linearise_batched(int64_t A, const int32_t* idx, int m, int n,
                           const double* F, const double* J,
                           const double* const* Fp_host, const double* dx,
                           int jac_mode, const int32_t* istate, double* lin,
                           void* stream) {
    return blsq_linearise_batched_rows(A, idx, m, n, F, J, Fp_host, dx, jac_mode, istate,
                                       lin, nullptr, stream);
}

int blsq_linearise_batched_ld(int64_t A, const int32_t* idx, int m, int n, int ldj,
                              const double* F, const double* J,
                              const double* const* Fp_host, const double* dx,
                              int jac_mode, const int32_t* istate, double* lin,
                              const int32_t* rows, void* stream) {
    if (ldj < n) return BLSQ_E_BADARG;
    if (ldj == n || jac_mode != 0)
        return blsq_linearise_batched_rows(A, idx, m, n, F, J, Fp_host, dx, jac_mode, istate,
                                           lin, rows, stream);
    if (A < 0 || m < 1 || !F || !J || !istate || !lin) return BLSQ_E_BADARG;
    // a row of J starts only as aligned as ldj * 8 bytes allows: the vector
    // width follows from both n and ldj, and J must be aligned to it
    if ((uintptr_t)J % (8 * lin_ld_width(n, ldj))) return BLSQ_E_BADARG;
    if (A == 0) return 0;
#ifdef BLSQ_ONLY_N46
    return BLSQ_E_UNSUPPORTED;
#else
    BLSQ_DISPATCH_N(n, {
        return ld_launch_lin<N_>(A, idx, m, ldj, F, J, istate, lin, rows, (cudaStream_t)stream);
    });
    return 0;
#endif
}

int blsq_pad_points(int nseg, const blsq_pad_segment* seg_host, int64_t A, int n, int fd,
                    double* out, void* stream) {
    if (nseg < 1 || nseg > BLSQ_MAX_BATCHED_N || !seg_host || !out || A < 0) return BLSQ_E_BADARG;
    if (n < 1 || n > BLSQ_MAX_BATCHED_N || fd < 0 || fd > 2) return BLSQ_E_BADARG;
    PadTable tab;
    tab.nseg = nseg;
    int64_t off = 0;
    for (int j = 0; j < nseg; j++) {
        const blsq_pad_segment& g = seg_host[j];
        if (g.off != off || g.A < 0 || g.n < 1 || g.n > n) return BLSQ_E_BADARG;
        if (g.A > 0 && (!g.x0 || !g.X || (fd && !g.Xp))) return BLSQ_E_BADARG;
        tab.seg[j] = g;
        off += g.A;
    }
    if (off != A) return BLSQ_E_BADARG;
    if (A == 0) return 0;
    const int64_t total = (fd ? (int64_t)fd * n : 1) * A * n;
    pad_points_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        tab, A, n, fd, out);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

int blsq_round_batched_rows(int method, int64_t A, const int32_t* idx, int m, int n,
                            const double* lin, const double* x0, const double* lb,
                            const double* ub, int bstride, const double* scaling,
                            double ftol, double xtol, double gtol, int max_nfev,
                            int first, double* state, int32_t* istate, double* Xnew,
                            double* Xjac, int32_t* work, int32_t* count,
                            const int32_t* rows, void* stream) {
    if (A < 0 || !lin || !x0 || !lb || !ub || !state || !istate || !Xnew) return BLSQ_E_BADARG;
    if (method != BLSQ_METHOD_TRF && method != BLSQ_METHOD_DOGBOX) return BLSQ_E_BADARG;
    if (bstride != 0 && bstride != n) return BLSQ_E_BADARG;
    if (A == 0) {
        if (count) {
            cudaError_t e = cudaMemsetAsync(count, 0, 3 * sizeof(int32_t), (cudaStream_t)stream);
            if (e != cudaSuccess) return (int)e;
        }
        return 0;
    }
    SolveParams P;
    P.ftol = ftol; P.xtol = xtol; P.gtol = gtol;
    P.max_nfev = max_nfev; P.m = m; P.jac_scaling = scaling ? 0 : 1;
    BLSQ_DISPATCH_N(n, {
        return dispatch_round<N_>(method, A, idx, lin, x0, lb, ub, bstride,
                                  scaling, P, first, state, istate, Xnew, Xjac,
                                  work, count, rows, (cudaStream_t)stream);
    });
    return 0;
}

int blsq_round_batched(int method, int64_t A, const int32_t* idx, int m, int n,
                       const double* lin, const double* x0, const double* lb,
                       const double* ub, int bstride, const double* scaling,
                       double ftol, double xtol, double gtol, int max_nfev,
                       int first, double* state, int32_t* istate, double* Xnew,
                       double* Xjac, int32_t* work, int32_t* count, void* stream) {
    return blsq_round_batched_rows(method, A, idx, m, n, lin, x0, lb, ub, bstride, scaling,
                                   ftol, xtol, gtol, max_nfev, first, state, istate, Xnew,
                                   Xjac, work, count, nullptr, stream);
}

int blsq_dogbox_on_bound(int64_t B, int n, const int32_t* istate,
                         int64_t* mask, void* stream) {
    if (B < 0 || n < 1 || n > BLSQ_MAX_BATCHED_N || !istate || !mask) return BLSQ_E_BADARG;
    if (B == 0) return 0;
    int64_t blocks = (B * n + 255) / 256;
    on_bound_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(B, n, istate, mask);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

int blsq_count_running(int64_t B, const int32_t* idx, const int32_t* istate,
                       int32_t* count, void* stream) {
    if (B < 0 || !istate || !count) return BLSQ_E_BADARG;
    cudaError_t e = cudaMemsetAsync(count, 0, sizeof(int32_t), (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
    if (B == 0) return 0;
    int64_t blocks = (B + 255) / 256;
    count_running_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(B, idx, istate, count);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

int64_t blsq_compact_work_size(int64_t A) {
    if (A < 0) return BLSQ_E_BADARG;
    return (A + CMP_SLOTS - 1) / CMP_SLOTS + 1;
}

int blsq_compact_batched(int64_t A, const int32_t* idx, const int32_t* istate, int n,
                         const double* Xnew, const double* Xjac, int32_t* idx_out,
                         int64_t* idx64_out, double* Xnew_out, double* Xjac_out,
                         int32_t* work, void* stream) {
    if (A < 0 || n < 1 || !istate || !Xnew || !idx_out || !Xnew_out || !work) return BLSQ_E_BADARG;
    if (Xjac && !Xjac_out) return BLSQ_E_BADARG;
    if (A >= ((int64_t)1 << 31)) return BLSQ_E_UNSUPPORTED;      /* problem ids are int32 */
    if (A == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const int nblocks = (int)((A + CMP_SLOTS - 1) / CMP_SLOTS);
    compact_count_kernel<<<nblocks, CMP_THREADS, 0, s>>>(A, idx, istate, work);
    BLSQ_LAUNCH_CHECK();
    compact_scan_kernel<<<1, 1024, 0, s>>>(nblocks, work);
    BLSQ_LAUNCH_CHECK();
    compact_scatter_kernel<<<nblocks, CMP_THREADS, 0, s>>>(A, idx, istate, n, work, Xnew, Xjac,
                                                          idx_out, idx64_out, Xnew_out, Xjac_out);
    BLSQ_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"

#ifdef BLSQ_PHASE_CLOCKS
// tools/phase_probe.py only: cycles [0..15] and visits [16..31] per phase of
// trf_round_impl since the last reset
extern "C" int blsq_debug_phase_read(unsigned long long* out, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out, blsq_phase_acc, sizeof(blsq_phase_acc));
    if (e == cudaSuccess && reset) {
        unsigned long long z[32] = {0};
        e = cudaMemcpyToSymbol(blsq_phase_acc, z, sizeof(z));
    }
    return (int)e;
}
#endif
