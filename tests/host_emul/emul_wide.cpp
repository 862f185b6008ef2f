// TEST INFRASTRUCTURE ONLY -- never loaded by the bounded_lsq_b200 package.
//
// The host emulation of emul.cpp with the batched entry points for
// n = 1..16 (include/blsq.h, version 102) instead of 1..8, plus the ragged
// entry points of emul_rows.cpp.  emul.cpp is included with its four
// n-dispatching entry points renamed (*_upto8); the public ones below hand
// n <= 8 to them and run n = 9..16 through the same templates (lin_host,
// trf_round, dogbox_round).  blsq_init_batched is renamed too (it reads the
// layout through blsq_state_layout) and restated below.  The libraries built from emul.cpp and
// emul_rows.cpp are unchanged.  Built by tests/test_batched_wide.py.
#define blsq_state_layout blsq_state_layout_upto8
#define blsq_lin_record_size blsq_lin_record_size_upto8
#define blsq_linearise_batched blsq_linearise_batched_upto8
#define blsq_round_batched blsq_round_batched_upto8
#define blsq_init_batched blsq_init_batched_upto8
#include "emul.cpp"
#undef blsq_init_batched
#undef blsq_state_layout
#undef blsq_lin_record_size
#undef blsq_linearise_batched
#undef blsq_round_batched

#define DISPATCH_WIDE_N(n, CALL)                          \
    switch (n) {                                          \
        case 9: { constexpr int N_ = 9; CALL; } break;    \
        case 10: { constexpr int N_ = 10; CALL; } break;  \
        case 11: { constexpr int N_ = 11; CALL; } break;  \
        case 12: { constexpr int N_ = 12; CALL; } break;  \
        case 13: { constexpr int N_ = 13; CALL; } break;  \
        case 14: { constexpr int N_ = 14; CALL; } break;  \
        case 15: { constexpr int N_ = 15; CALL; } break;  \
        case 16: { constexpr int N_ = 16; CALL; } break;  \
        default: return BLSQ_E_UNSUPPORTED;               \
    }

namespace {

// blsq_round_batched of emul.cpp for one N
template <int N>
void round_host(int method, int64_t A, const int32_t* idx, const double* lin,
                const double* x0, const double* lb, const double* ub, int bs,
                const double* scaling, const SolveParams& P, int first, double* state,
                int32_t* istate, double* Xnew, double* Xjac) {
    double sc[N];
    for (int i = 0; i < N; i++) sc[i] = scaling ? scaling[i] : 1.0;
    for (int64_t s = 0; s < A; s++) {
        int64_t pid = idx ? idx[s] : s;
        int32_t* ist = istate + pid * IS_SIZE;
        if (ist[IS_STATUS] != ST_RUNNING) continue;
        const double* ln = lin + s * LinRec<N>::SIZE;
        bool go;
        double* st;
        int xnew_off = N;
        if (method == BLSQ_METHOD_TRF) {
            xnew_off = TrfState<N>::XNEW;
            st = state + pid * TrfState<N>::SIZE;
            go = trf_round<N>(st, ist, ln, x0 + pid * N, lb + pid * bs, ub + pid * bs, sc, P,
                              first);
        } else {
            st = state + pid * DogState<N>::SIZE;
            go = dogbox_round<N>(st, ist, ln, x0 + pid * N, lb + pid * bs, ub + pid * bs, sc,
                                 P, first);
        }
        if (!go) continue;
        for (int i = 0; i < N; i++) {
            double xn = st[xnew_off + i];
            Xnew[s * N + i] = xn;
            if (Xjac) {
                double xj = xn;
                if (method == BLSQ_METHOD_DOGBOX) {
                    int ob = ((ist[IS_FREE] >> i) & 1) ? get2(ist[IS_MARKS], i)
                                                       : get2(ist[IS_ONB], i);
                    if (ob == -1) xj = lb[pid * bs + i];
                    if (ob == 1) xj = ub[pid * bs + i];
                }
                Xjac[s * N + i] = xj;
            }
        }
    }
}

int clamp_rows(const int32_t* rows, int64_t pid, int m) {
    const int r = rows[pid];
    return r < 0 ? 0 : (r > m ? m : r);
}

}  // namespace

extern "C" {

int blsq_state_layout(int method, int n, int* out) {
    if (n <= 8) return blsq_state_layout_upto8(method, n, out);
    DISPATCH_WIDE_N(n, {
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

int blsq_init_batched(int method, int64_t B, int n, const double* x0,
                      const double* lb, const double* ub, int bs,
                      double* state, int32_t* istate, double* Xnew, void*) {
    int lay[9];
    int rc = blsq_state_layout(method, n, lay);
    if (rc) return rc;
    int SS = lay[0];
    for (int64_t b = 0; b < B; b++) {
        for (int i = 0; i < n; i++) {
            double x = x0[b * n + i];
            if (method == BLSQ_METHOD_TRF)
                x = strictly_feasible(x, lb[b * bs + i], ub[b * bs + i], 1e-10);
            state[b * SS + lay[2] + i] = x;
            state[b * SS + i] = x;
            Xnew[b * n + i] = x;
        }
        int32_t* ip = istate + b * IS_SIZE;
        for (int k = 0; k < IS_SIZE; k++) ip[k] = 0;
        ip[IS_STATUS] = ST_RUNNING;
    }
    return 0;
}

int blsq_lin_record_size(int n) {
    if (n <= 8) return blsq_lin_record_size_upto8(n);
    DISPATCH_WIDE_N(n, { return LinRec<N_>::SIZE; });
    return BLSQ_E_UNSUPPORTED;
}

int blsq_linearise_batched(int64_t A, const int32_t* idx, int m, int n,
                           const double* F, const double* J,
                           const double* const* Fp, const double* dx, int mode,
                           const int32_t* istate, double* lin, void* stream) {
    if (n <= 8)
        return blsq_linearise_batched_upto8(A, idx, m, n, F, J, Fp, dx, mode, istate, lin,
                                            stream);
    DISPATCH_WIDE_N(n, {
        for (int64_t s = 0; s < A; s++) {
            int64_t pid = idx ? idx[s] : s;
            if (istate[pid * IS_SIZE + IS_STATUS] != ST_RUNNING) continue;
            lin_host<N_>(m, F, J, Fp, s, dx, mode, lin + s * LinRec<N_>::SIZE);
        }
    });
    return 0;
}

int blsq_round_batched(int method, int64_t A, const int32_t* idx, int m, int n,
                       const double* lin, const double* x0, const double* lb,
                       const double* ub, int bs, const double* scaling,
                       double ftol, double xtol, double gtol, int max_nfev,
                       int first, double* state, int32_t* istate, double* Xnew,
                       double* Xjac, int32_t* work, int32_t* count, void* stream) {
    if (n <= 8)
        return blsq_round_batched_upto8(method, A, idx, m, n, lin, x0, lb, ub, bs, scaling,
                                        ftol, xtol, gtol, max_nfev, first, state, istate,
                                        Xnew, Xjac, work, count, stream);
    SolveParams P;
    P.ftol = ftol; P.xtol = xtol; P.gtol = gtol;
    P.max_nfev = max_nfev; P.m = m; P.jac_scaling = scaling ? 0 : 1;
    DISPATCH_WIDE_N(n, {
        round_host<N_>(method, A, idx, lin, x0, lb, ub, bs, scaling, P, first, state, istate,
                       Xnew, Xjac);
    });
    if (count) {
        int c = 0;
        for (int64_t s = 0; s < A; s++)
            c += istate[(idx ? idx[s] : s) * IS_SIZE + IS_STATUS] == ST_RUNNING;
        count[2] = c;
    }
    return 0;
}

// Ragged batches, as emul_rows.cpp: each running slot is handed to the dense
// entry point above as a batch of one problem with m = rows[pid].
int blsq_linearise_batched_rows(int64_t A, const int32_t* idx, int m, int n,
                                const double* F, const double* J,
                                const double* const* Fp, const double* dx, int mode,
                                const int32_t* istate, double* lin, const int32_t* rows,
                                void* stream) {
    if (!rows) return blsq_linearise_batched(A, idx, m, n, F, J, Fp, dx, mode, istate, lin, stream);
    const int LS = blsq_lin_record_size(n);
    if (LS < 0) return LS;
    const int np = mode == 2 ? 2 * n : (mode == 1 ? n : 0);
    std::vector<const double*> fp(np > 0 ? np : 1);
    for (int64_t s = 0; s < A; s++) {
        const int32_t pid = (int32_t)(idx ? idx[s] : s);
        if (istate[(int64_t)pid * IS_SIZE + IS_STATUS] != ST_RUNNING) continue;
        for (int j = 0; j < np; j++) fp[j] = Fp[j] + s * m;
        const int rc = blsq_linearise_batched(
            1, &pid, clamp_rows(rows, pid, m), n, F + s * m, J ? J + s * m * n : nullptr,
            np ? fp.data() : nullptr, dx ? dx + s * (mode == 2 ? 2 * n : n) : nullptr, mode,
            istate, lin + s * LS, stream);
        if (rc) return rc;
    }
    return 0;
}

int blsq_round_batched_rows(int method, int64_t A, const int32_t* idx, int m, int n,
                            const double* lin, const double* x0, const double* lb,
                            const double* ub, int bs, const double* scaling,
                            double ftol, double xtol, double gtol, int max_nfev,
                            int first, double* state, int32_t* istate, double* Xnew,
                            double* Xjac, int32_t* work, int32_t* count,
                            const int32_t* rows, void* stream) {
    if (!rows)
        return blsq_round_batched(method, A, idx, m, n, lin, x0, lb, ub, bs, scaling, ftol,
                                  xtol, gtol, max_nfev, first, state, istate, Xnew, Xjac,
                                  work, count, stream);
    const int LS = blsq_lin_record_size(n);
    if (LS < 0) return LS;
    for (int64_t s = 0; s < A; s++) {
        const int32_t pid = (int32_t)(idx ? idx[s] : s);
        const int rc = blsq_round_batched(
            method, 1, &pid, clamp_rows(rows, pid, m), n, lin + s * LS, x0, lb, ub, bs,
            scaling, ftol, xtol, gtol, max_nfev, first, state, istate, Xnew + s * n,
            Xjac ? Xjac + s * n : nullptr, nullptr, nullptr, stream);
        if (rc) return rc;
    }
    if (count) {
        int c = 0;
        for (int64_t s = 0; s < A; s++)
            c += istate[(idx ? idx[s] : s) * IS_SIZE + IS_STATUS] == ST_RUNNING;
        count[2] = c;
    }
    return 0;
}

}  // extern "C"
