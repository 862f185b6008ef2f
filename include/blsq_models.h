/* blsq_models.h -- residual/Jacobian callbacks of the synthetic workloads
 * named in BASELINE.json (configs C2, C3) as single fused CUDA kernels.
 *
 * These are USER-SIDE code: what a caller of least_squares would otherwise
 * write as a chain of PyTorch elementwise ops (bounded_lsq_b200/synthetic.py
 * fun_t / jac_t).  They are not part of the reference boundary in blsq.h; they
 * exist so bench.py can show the solver with callbacks that do not dominate
 * the run.  Same operation order as the torch forms, so results are bit
 * identical to them.
 *
 * idx (nullable) maps row s of X/F/J to the problem whose data row y[idx[s]]
 * it uses -- the active-set gather is fused into the load.
 */
#ifndef BLSQ_MODELS_H_
#define BLSQ_MODELS_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* y = a e^{-b t} + c e^{-d t}: F (A, m) = model - y[idx]; J (A, m, 4) or null.
 * X and J must be 32-byte aligned (double4 loads, 256-bit stores), else
 * BLSQ_E_BADARG; so must X of blsq_model_expdecay2_linearise. */
int blsq_model_expdecay2(int64_t A, const int64_t* idx, int m, const double* t,
                         const double* X, const double* y, double* F, double* J,
                         void* stream);
/* Ragged batches: rows (nullable, int32, indexed by problem id like y) gives
 * problem pid rows[pid] residuals; only rows r < rows[pid] of F and J are
 * written (the rest of each (m) / (m, 4) block is left as it was) and only
 * those rows of y are used.  rows = null: blsq_model_expdecay2. */
int blsq_model_expdecay2_rows(int64_t A, const int64_t* idx, int m, const double* t,
                              const double* X, const double* y, const int32_t* rows,
                              double* F, double* J, void* stream);
/* The same model compiled INTO the linearisation kernel: the lin records of
 * blsq_linearise_batched (include/blsq.h) for the A trial points X, without
 * F and J ever being written to memory.  idx: int32 problem ids of the slots
 * (nullable), as for blsq_linearise_batched.  m <= 64. */
int blsq_model_expdecay2_linearise(int64_t A, const int32_t* idx, int m, const double* t,
                                   const double* X, const double* y, const int32_t* istate,
                                   double* lin, void* stream);
/* y = A e^{-((t-mu)/sigma)^2/2} + c0 + c1 t + c2 t^2: F (A, m) */
int blsq_model_gausspeak(int64_t A, const int64_t* idx, int m, const double* t,
                         const double* X, const double* y, double* F,
                         void* stream);
/* tall workload (C4/C5): J (m, n) keeps the constant design matrix in its
 * first n-4 columns; x is a DEVICE pointer to n doubles.
 *   fun: F = J[:, :n-4] x[:n-4] + x_k e^{-x_{k+1} t} + x_{k+2} e^{-x_{k+3} t} - y
 *   jac: rewrites columns n-4..n-1 of J for the point x
 * J must be 16-byte aligned (128-bit loads and stores), else BLSQ_E_BADARG. */
int blsq_model_linexp_fun(int64_t m, int n, const double* J, const double* t,
                          const double* y, const double* x, double* F,
                          void* stream);
int blsq_model_linexp_jac(int64_t m, int n, double* J, const double* t,
                          const double* x, void* stream);
#ifdef __cplusplus
}
#endif
#endif
