/* blsq.h -- C ABI of the B200-native bounded least-squares hot path.
 *
 * The reference (nmayorov/bounded-lsq) is pure Python and has no FFI; the seam
 * this library replaces is the Python call
 *     least_squares.py:373-379   trf(fun, jac, x0, lb, ub, ftol, xtol, gtol,
 *                                    max_nfev, scaling) / dogbox(...)
 * and the helpers those two call (bounds.py, trust_region.py).  Each entry
 * point cites the reference lines it stands in for.  INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - arrays are dense row-major float64 / int32 / int64 / uint8;
 *   - `stream` is a cudaStream_t passed as void*; nothing synchronises;
 *   - no allocation, no global state; the caller owns every buffer;
 *   - return 0 on success, <0 for an invalid argument (BLSQ_E_*), >0 for a
 *     cudaError_t raised by the launch;
 *   - bounds are either shared by all problems (bstride = 0, arrays of n) or
 *     per problem (bstride = n, arrays of B*n).
 */
#ifndef BLSQ_H_
#define BLSQ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLSQ_VERSION 103

#define BLSQ_E_BADARG (-1)      /* null pointer / negative size */
#define BLSQ_E_UNSUPPORTED (-2) /* n outside 1..BLSQ_MAX_BATCHED_N, ... */

/* batched mode takes 1 <= n <= 16 (version 102; 8 before): istate packs two
 * bits per coordinate in one int32 (dogbox's on_bound and bound marks) */
#define BLSQ_MAX_BATCHED_N 16

#define BLSQ_METHOD_TRF 0
#define BLSQ_METHOD_DOGBOX 1

/* per-problem status while a batched solve is in flight; values >= 0 are the
 * reference's termination codes (least_squares.py:30-37) */
#define BLSQ_STATUS_RUNNING (-1)
#define BLSQ_STATUS_ERR_TR_ZERO (-101)    /* trust_region.py:28-29 ValueError */
#define BLSQ_STATUS_ERR_TR_OUTSIDE (-102) /* trust_region.py:34-35 ValueError */

#define BLSQ_ISTATE_SIZE 8 /* int32 per problem: status, nfev, njev, ... */

int blsq_version(void);
const char* blsq_error_string(int code);

/* ---- layout queries (host) ------------------------------------------- */

/* Offsets (in doubles) of the fields of one problem's state record:
 * out[0]=record size, [1]=x, [2]=x_new, [3]=scale, [4]=obj, [5]=Delta,
 * [6]=optimality (g_norm), [7]=g, [8]=alpha (TRF only, else -1). */
int blsq_state_layout(int method, int n, int* out_host);
/* Size in doubles of one linearisation record (packed R, Q^T f, J^T f, f.f) */
int blsq_lin_record_size(int n);

/* ---- elementwise bound geometry: bit-exact with bounds.py ------------- */

/* bounds.py:24-48 step_size_to_bound, one row of n per problem */
int blsq_step_size_to_bound(int64_t B, int n, const double* x, const double* d,
                            const double* lb, const double* ub, int bstride,
                            double* step, int64_t* hits, void* stream);
/* bounds.py:51-76 find_active_constraints */
int blsq_find_active_constraints(int64_t B, int n, const double* x,
                                 const double* lb, const double* ub,
                                 int bstride, double rtol, int64_t* mask,
                                 void* stream);
/* bounds.py:79-103 make_strictly_feasible */
int blsq_make_strictly_feasible(int64_t B, int n, const double* x,
                                const double* lb, const double* ub, int bstride,
                                double rstep, double* out, void* stream);
/* bounds.py:106-149 scaling_vector (Coleman-Li v and dv/dx) */
int blsq_scaling_vector(int64_t B, int n, const double* x, const double* g,
                        const double* lb, const double* ub, int bstride,
                        double* v, double* jv, void* stream);
/* bounds.py:19-21 in_bounds; ok[b] = 1/0 */
int blsq_in_bounds(int64_t B, int n, const double* x, const double* lb,
                   const double* ub, int bstride, uint8_t* ok, void* stream);
/* least_squares.py:248-252 x_covariance = (J^T J)^-1, from the triangular
 * factor of J kept by the solve: R packed upper (packed = 1; batched state
 * records: rec = state, stride = record size, r_off = layout R) or dense
 * row-major n x n (packed = 0; tall mode: rec = fac + R).  cov (B, n, n);
 * NaN where R is singular ("the inverse doesn't exist"). */
int blsq_covariance(int64_t B, int n, const double* rec, int64_t stride, int r_off,
                    int packed, double* cov, void* stream);
/* dogbox.py:9-35 find_intersection; flags bit0 orig_l, bit1 orig_u,
 * bit2 tr_l, bit3 tr_u */
int blsq_find_intersection(int64_t B, int n, const double* x, const double* tr,
                           const double* lb, const double* ub, int bstride,
                           double* lo, double* hi, uint8_t* flags,
                           void* stream);

/* ---- 2-point finite differences (least_squares.py:357-365; scipy
 *      _numdiff._compute_absolute_step/_adjust_scheme_to_bounds) ---------- */

/* For each of A active problems (slot s, problem idx[s] or s when idx is
 * null): h_i with the bound adjustment, the n perturbed points
 * Xp[i,s,:] = x + h_i e_i (layout (n, A, n): one (A, n) batch per coordinate,
 * i.e. one callback call per coordinate like scipy's loop) and
 * dx[s,i] = (x_i + h_i) - x_i.  rel_step = NaN means diff_step=None. */
int blsq_fd2_points(int64_t A, const int32_t* idx, int n, const double* x,
                    const double* lb, const double* ub, int bstride,
                    double rel_step, double* Xp, double* dx, void* stream);

/* 3-point scheme (jac='3-point', scipy '2-sided' with the one-sided fallback
 * near a bound).  Xp has layout (2n, A, n): batches 2i, 2i+1 are the two
 * evaluation points of coordinate i -- (x - h, x + h) for a central
 * difference, (x + h, x + 2h) for the one-sided 3-point stencil.  dxo is
 * (A, 2n): dxo[s, i] = the denominator, dxo[s, n + i] = 1.0 if one sided. */
int blsq_fd3_points(int64_t A, const int32_t* idx, int n, const double* x,
                    const double* lb, const double* ub, int bstride,
                    double rel_step, double* Xp, double* dxo, void* stream);

/* ---- batched solve: init -> [callbacks -> linearise -> round]* -------- */

/* trf.py:201 (x = make_strictly_feasible(x0, rstep=1e-10)) / dogbox.py:131
 * (x = x0): marks every problem running and writes the first evaluation
 * point to the state record and to Xnew (B x n). */
int blsq_init_batched(int method, int64_t B, int n, const double* x0,
                      const double* lb, const double* ub, int bstride,
                      double* state, int32_t* istate, double* Xnew,
                      void* stream);

/* Linearisation at the trial points (trf.py:244,264-274; dogbox.py:170,197):
 * one QR of [J | f] per problem -> packed R, Q^T f, g = J^T f, f.f.
 *   jac_mode 0: J is (A, m, n) row-major (analytic Jacobian callback)
 *   jac_mode 1: Fp_host is a HOST array of n device pointers, Fp_host[i] =
 *               residuals (A, m) at the i-th perturbed batch of
 *               blsq_fd2_points, dx (A, n) its denominators;
 *               J[:, i] = (Fp_i - f) / dx_i is formed in registers (scipy
 *               _dense_difference) and never materialised.
 *   jac_mode 2: 3-point: Fp_host holds 2n device pointers in the batch order
 *               of blsq_fd3_points, dx is its (A, 2n) dxo array;
 *               J[:, i] = (f2 - f1) / dx_i or (-3 f + 4 f1 - f2) / dx_i.
 * Slots whose problem is no longer running are skipped.
 * Alignment (jac_mode 0): the rows of J are read with vector loads, so J must
 * be 32-byte aligned for n = 4, 8, 12, 16 and 16-byte aligned for n = 2, 6, 10,
 * 14; otherwise BLSQ_E_BADARG before any launch.
 * Valid range: sums of squares are formed in double, so every squared column
 * norm of [J | f] must be a normal double (entries between about 2^-500 and
 * 2^500 at m <= 1100); outside it the record is inaccurate or not finite. */
int blsq_linearise_batched(int64_t A, const int32_t* idx, int m, int n,
                           const double* F, const double* J,
                           const double* const* Fp_host, const double* dx,
                           int jac_mode, const int32_t* istate, double* lin,
                           void* stream);

/* One round of the outer/inner loops for every running problem
 * (trf.py:238-352 or dogbox.py:164-267): ratio test of the trial in flight,
 * Delta/alpha update, termination tests, accept, Coleman-Li scaling + SVD of
 * the hat-space triangle + LM parameter + reflective/gradient candidates
 * (TRF) or active set + Gauss-Newton/Cauchy + box dogleg (dogbox), and the
 * next trial point into the state record and Xnew[slot].
 * Xjac (nullable) receives the point the Jacobian of an accepted step is
 * evaluated at: for dogbox that is the trial with the coordinates that hit a
 * bound snapped onto it (dogbox.py:256-261 -- f is taken at x_new, J at the
 * snapped x); for TRF it equals Xnew.
 * scaling: n doubles (shared) or null for scaling='jac'.
 * work (nullable, A + 1 int32): with it the TRF round runs as two kernels --
 * every problem takes the Gauss-Newton shortcut of solve_lsq_trust_region
 * (trust_region.py:108-117: full rank certified, |p| <= Delta; ~95 % of the
 * solves) and the rest are collected in `work` and finished through the SVD
 * route with dense warps.  Without it (or for dogbox): one kernel.
 * count (nullable, 4 int32, zero before the first use): count[2] receives the
 * number of slots still running after this round (what blsq_count_running
 * would return) at no extra launch: one atomic per CTA into count[0], the
 * last CTA to finish publishes the total and re-arms count[0..1]. */
int blsq_round_batched(int method, int64_t A, const int32_t* idx, int m, int n,
                       const double* lin, const double* x0, const double* lb,
                       const double* ub, int bstride, const double* scaling,
                       double ftol, double xtol, double gtol, int max_nfev,
                       int first, double* state, int32_t* istate, double* Xnew,
                       double* Xjac, int32_t* work, int32_t* count, void* stream);

/* Ragged batches (version 101): the two calls above with a per-problem number
 * of residuals.  rows (nullable, int32) is indexed by problem id like istate
 * (idx[slot], or the slot when idx is null); problem pid has residuals
 * 0 .. rows[pid]-1.  m stays the row stride of F, J and Fp_host[*]; rows past
 * rows[pid] are never read and may hold anything (NaN included).  Each problem
 * is solved as the reference solves the problem made of its first rows[pid]
 * residuals: the cost, full_rank = m >= n and the smin > eps*m*smax test
 * (trust_region.py:108-112), the Gauss-Newton certificate and dogbox's
 * rcond = eps*max(m, n_free) use rows[pid].  The kernels clamp rows[pid] to
 * [0, m] for memory safety; callers reject counts outside 1 .. m.  With
 * rows = null both are the calls above, bit for bit. */
int blsq_linearise_batched_rows(int64_t A, const int32_t* idx, int m, int n,
                                const double* F, const double* J,
                                const double* const* Fp_host, const double* dx,
                                int jac_mode, const int32_t* istate, double* lin,
                                const int32_t* rows, void* stream);
int blsq_round_batched_rows(int method, int64_t A, const int32_t* idx, int m, int n,
                            const double* lin, const double* x0, const double* lb,
                            const double* ub, int bstride, const double* scaling,
                            double ftol, double xtol, double gtol, int max_nfev,
                            int first, double* state, int32_t* istate, double* Xnew,
                            double* Xjac, int32_t* work, int32_t* count,
                            const int32_t* rows, void* stream);

/* Ragged parameter counts (version 103): a batch whose problems have their
 * own number of parameters is solved as segments, one per count N, each a
 * dense lock-step solve of N-parameter problems whose trial points share one
 * padded (A, ldj) callback batch (least_squares_batched `cols`).
 *
 * blsq_linearise_batched_rows for the segment's slots of an (A, m, ldj)
 * Jacobian: row r of slot s starts at J + (s * m + r) * ldj, and only its
 * first n columns are read (the others may hold anything, NaN included).
 * F, Fp_host, dx, lin, istate and rows are those of the n-parameter
 * segment, as for blsq_linearise_batched_rows; the finite-difference modes
 * do not read J, so ldj only matters for jac_mode 0.  With ldj == n (or
 * jac_mode != 0) this is exactly blsq_linearise_batched_rows.  ldj < n is
 * BLSQ_E_BADARG.  The record is bit for bit the one of a dense (A, m, n) J
 * with the same columns.
 * Alignment (jac_mode 0, ldj > n): a row start is only as aligned as ldj * 8
 * bytes allows, so the rows are read with 4-double loads when 4 divides both
 * n and ldj, 2-double loads when 2 does, else one double at a time; J must be
 * aligned to that width (32 or 16 bytes), otherwise BLSQ_E_BADARG before any
 * launch.  J aligned for the padded width ldj (blsq_linearise_batched) always
 * is. */
int blsq_linearise_batched_ld(int64_t A, const int32_t* idx, int m, int n, int ldj,
                              const double* F, const double* J,
                              const double* const* Fp_host, const double* dx,
                              int jac_mode, const int32_t* istate, double* lin,
                              const int32_t* rows, void* stream);

/* One segment of a padded callback batch (blsq_pad_points): slots
 * off .. off+A-1 of the batch hold its A active problems, in order. */
typedef struct {
    int64_t off;          /* first slot; segments tile 0 .. A-1 in order */
    int64_t A;            /* its slots (0: an empty segment) */
    int n;                /* its parameters, 1 <= n <= the padded width */
    const int32_t* idx;   /* slot -> row of x0 (nullable: the slot itself) */
    const double* x0;     /* its problems' x0, rows of the padded width */
    const double* X;      /* (A, n) its points (Xnew / Xjac of its solve) */
    const double* Xp;     /* (fd * n, A, n) its blsq_fd2_points / blsq_fd3_points
                             batches; read only when fd != 0 */
} blsq_pad_segment;

/* The trial points of a ragged-parameter batch in the padded layout the
 * callbacks take (no reference counterpart: the reference solves one problem
 * of its own size per call).  nseg (1 .. BLSQ_MAX_BATCHED_N) segments from
 * the HOST array seg_host; n is the padded width.  Coordinates k >= seg.n of
 * every point are the problem's x0[k], unchanged (padded parameters are held
 * fixed).
 *   fd 0: out (A, n), slot s = X[s] padded.
 *   fd 1: out (n, A, n), the 2-point batches: batch i of a segment with
 *         seg.n > i is its Xp[i], of the others X (not perturbed: their
 *         residuals at that batch are never read).
 *   fd 2: out (2n, A, n), the 3-point batches 2i, 2i+1 likewise.
 * The segments' offsets must tile 0 .. A-1; otherwise BLSQ_E_BADARG. */
int blsq_pad_points(int nseg, const blsq_pad_segment* seg_host, int64_t A, int n, int fd,
                    double* out, void* stream);

/* dogbox.py:152-154,254: on_bound as the reference's int array (B x n) */
int blsq_dogbox_on_bound(int64_t B, int n, const int32_t* istate,
                         int64_t* mask, void* stream);

/* count[0] = number of slots 0..A-1 (problem idx[s], or s when idx is null)
 * still running (device int32) */
int blsq_count_running(int64_t A, const int32_t* idx, const int32_t* istate,
                       int32_t* count, void* stream);

/* Ordered compaction of the active set (host logic of the lock-step driver;
 * no reference counterpart: the reference solves one problem per call).  Slots
 * whose problem is still running keep their order: idx_out[k] (int32) and
 * idx64_out[k] (nullable, for torch gathers) = problem id of the k-th
 * survivor, Xnew_out / Xjac_out (k, n) its trial points (Xjac nullable).  The
 * outputs must not alias the inputs.  work: blsq_compact_work_size(A) int32;
 * its LAST element receives the number of survivors. */
int64_t blsq_compact_work_size(int64_t A);
int blsq_compact_batched(int64_t A, const int32_t* idx, const int32_t* istate, int n,
                         const double* Xnew, const double* Xjac, int32_t* idx_out,
                         int64_t* idx64_out, double* Xnew_out, double* Xjac_out,
                         int32_t* work, void* stream);


/* ---- tall mode: one problem, m_local rows on this rank, 2 <= n <= 256 -----
 *
 * Per Jacobian evaluation (trf.py:244,264-274; dogbox.py:170,197-199) the
 * rank runs a preconditioned Cholesky QR on [J | f]:
 *   blsq_tall_gram(1)   -> record {J_s^T J_s} over this rank's rows, or over
 *                          one row tile out of `sstride` (sketch: pass 1 only
 *                          has to deliver a preconditioner)
 *   (all-gather the records over the ranks)
 *   blsq_tall_factor(1) -> R1 = chol(sum of records), R1^-1
 *   blsq_tall_gram(2)   -> record {Y^T Y, Y^T f, f.f, J^T f}, Y = J R1^-1,
 *                          every row
 *   (all-gather)
 *   blsq_tall_factor(2) -> R = chol(.) R1 (J = Q R), Q^T f, g = J^T f, f.f,
 *                          and fac.refine = 1 when Y^T Y is too far from the
 *                          identity for one Cholesky pass to be accurate; then
 *   blsq_tall_factor(3) -> R1 <- R, R1^-1; repeat gram(2), factor(2)
 * With sstride = 1 this is CholeskyQR2.  A record is
 * blsq_tall_record_size(n) doubles: G row-major (upper triangle valid) |
 * Y^T f (n) | f.f | J^T f (n).  `fac` holds blsq_tall_fac_size(n) doubles
 * (offsets: blsq_tall_layout).  fac.info != 0: NaN/zero Jacobian.  Rank
 * deficient Jacobians are handled by a diagonal shift of ~16 n eps |G|. */
#define BLSQ_MAX_TALL_N 256
int64_t blsq_tall_gram_work_size(int n);   /* doubles of `work` for blsq_tall_gram */
int64_t blsq_tall_fac_size(int n);
int64_t blsq_tall_record_size(int n);
int blsq_tall_sample_stride(int64_t m_local, int n);   /* recommended sstride */
int blsq_tall_gram(int pass, int64_t m, int n, const double* J, const double* f,
                   const double* Rinv, int sstride, double* work, double* out,
                   void* stream);
int blsq_tall_factor(int pass, int n, int nranks, int64_t gstride,
                     const double* grams, double* fac, void* stream);
/* out[0] = sum f_i^2 over this rank's rows (trf.py:311, dogbox.py:224);
 * work: 4 * (number of SMs) doubles */
int blsq_tall_sumsq(int64_t m, const double* f, double* work, double* out,
                    void* stream);


/* The n x n tail of one round for the tall problem (one CTA).  `state`
 * (blsq_tall_layout out[0] doubles) and `istate` (out[1] int32) persist
 * between the calls; x, bounds and every n-sized quantity are replicated on
 * all ranks and every rank runs the same calls on the same inputs.
 *   phase 0  init: trf.py:201 / dogbox.py:131 -> state.x_new = start point
 *   phase 1  judge: ||f(x_new)||^2 = sum of ssq_parts[0..nranks) (rank order);
 *            ratio test, Delta/alpha update, termination tests, accept
 *            (trf.py:310-352, dogbox.py:222-267).  istate[3] = accepted.
 *   phase 2  propose: `fac` is the factor record of the Jacobian at state.x;
 *            new_lin != 0 when it changed since the last call.  Coleman-Li
 *            scaling, SVD of the hat-space triangle, LM parameter, candidates
 *            (trf.py:238-308) or active set, Gauss-Newton/Cauchy, box dogleg
 *            (dogbox.py:164-220) -> state.x_new, or a final istate[0] status.
 * work: n*n doubles (used when n > 128).  scaling: n doubles or null ('jac').
 * blsq_tall_layout: out[0..15] = state size, istate size, offsets of x,
 * x_new, obj, Delta, optimality, on_bound (istate), fac size, offsets of R,
 * Q^T f, g, f.f, info, packed R1^-1 inside fac, offset of scale (state),
 * offset of refine (fac): 17 values. */
int blsq_tall_layout(int n, int64_t* out_host);
int blsq_tall_round(int method, int phase, int n, int64_t m_total, int nranks,
                    const double* ssq_parts, const double* fac,
                    const double* x0, const double* lb, const double* ub,
                    const double* scaling, double ftol, double xtol,
                    double gtol, int max_nfev, int first, int new_lin,
                    double* state, int32_t* istate, double* work, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BLSQ_H_ */
