// TEST INFRASTRUCTURE ONLY -- never loaded by the bounded_lsq_b200 package.
//
// The host emulation of emul.cpp plus the two entry points of ragged batches
// (include/blsq.h, version 101): blsq_linearise_batched_rows and
// blsq_round_batched_rows.  Each running slot is handed to the dense host
// entry point as a batch of one problem with m = rows[pid] and its base
// pointers shifted to that slot, so a ragged problem runs exactly the code a
// dense problem of rows[pid] residuals runs.  Built by
// tests/test_ragged_batches.py.
#include "emul.cpp"

namespace {
int clamp_rows(const int32_t* rows, int64_t pid, int m) {
    const int r = rows[pid];
    return r < 0 ? 0 : (r > m ? m : r);
}
}  // namespace

extern "C" {

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
        // one problem: its rows are the first rows[pid] of slot s
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
