// TEST INFRASTRUCTURE ONLY -- never loaded by the bounded_lsq_b200 package.
//
// The host emulation of emul_wide.cpp (n = 1..16, ragged rows) plus the two
// entry points of ragged parameter counts (include/blsq.h, version 103):
// blsq_linearise_batched_ld gathers the first n columns of each running
// slot's rows of the padded Jacobian and hands them to the dense host entry
// point, and blsq_pad_points assembles the padded callback batches.  The
// libraries built from emul.cpp, emul_rows.cpp and emul_wide.cpp are
// unchanged.  Built by tests/test_ragged_cols.py.
#include "emul_wide.cpp"

extern "C" {

int blsq_linearise_batched_ld(int64_t A, const int32_t* idx, int m, int n, int ldj,
                              const double* F, const double* J,
                              const double* const* Fp, const double* dx, int mode,
                              const int32_t* istate, double* lin, const int32_t* rows,
                              void* stream) {
    if (ldj < n) return BLSQ_E_BADARG;
    if (ldj == n || mode != 0)
        return blsq_linearise_batched_rows(A, idx, m, n, F, J, Fp, dx, mode, istate, lin, rows,
                                           stream);
    std::vector<double> Jn((size_t)(A > 0 ? A : 0) * m * n);
    for (int64_t s = 0; s < A; s++) {
        const int64_t pid = idx ? idx[s] : s;
        if (istate[pid * IS_SIZE + IS_STATUS] != ST_RUNNING) continue;
        for (int r = 0; r < m; r++)
            for (int j = 0; j < n; j++)
                Jn[((size_t)s * m + r) * n + j] = J[((int64_t)s * m + r) * ldj + j];
    }
    return blsq_linearise_batched_rows(A, idx, m, n, F, Jn.data(), Fp, dx, mode, istate, lin,
                                       rows, stream);
}

int blsq_pad_points(int nseg, const blsq_pad_segment* seg, int64_t A, int n, int fd,
                    double* out, void*) {
    if (nseg < 1 || nseg > BLSQ_MAX_BATCHED_N || !seg || !out || A < 0) return BLSQ_E_BADARG;
    if (n < 1 || n > BLSQ_MAX_BATCHED_N || fd < 0 || fd > 2) return BLSQ_E_BADARG;
    int64_t off = 0;
    for (int j = 0; j < nseg; j++) {
        if (seg[j].off != off || seg[j].A < 0 || seg[j].n < 1 || seg[j].n > n)
            return BLSQ_E_BADARG;
        off += seg[j].A;
    }
    if (off != A) return BLSQ_E_BADARG;
    const int P = fd ? fd * n : 1;
    for (int j = 0; j < nseg; j++) {
        const blsq_pad_segment& g = seg[j];
        for (int p = 0; p < P; p++)
            for (int64_t s = 0; s < g.A; s++) {
                const int64_t row = g.idx ? g.idx[s] : s;
                double* o = out + ((int64_t)p * A + g.off + s) * n;
                for (int k = 0; k < n; k++)
                    o[k] = k >= g.n ? g.x0[row * n + k]
                         : (fd && p < fd * g.n) ? g.Xp[((int64_t)p * g.A + s) * g.n + k]
                                                : g.X[s * g.n + k];
            }
    }
    return 0;
}

}  // extern "C"
