"""Fused CUDA residual/Jacobian callbacks for the synthetic workloads.

User-side code (include/blsq_models.h): the same functions as
``synthetic.ExpDecay2.fun_t/jac_t`` and ``synthetic.GaussPeak.fun_t`` as one
kernel each, with the active-set gather of the per-problem data fused into
the load.  They use the *indexed* callback protocol of the batched driver:
``fun(X, idx, *args)`` with ``fun.blsq_indexed = True`` receives the raw
per-problem tensors plus the active problem ids instead of gathered copies.
"""
from __future__ import annotations

import torch

from . import _lib as L
from . import synthetic


def _t_on(model, dev, cache):
    t = cache.get(dev)
    if t is None:
        t = torch.as_tensor(model.t, dtype=torch.float64, device=dev)
        cache[dev] = t
    return t


def callbacks(model_name, jac_kind="exact", lib=None, rows=False):
    """(fun, jac) for ``least_squares_batched(..., args=(PerProblem(y),))``.

    ``rows=True`` (ExpDecay2, ragged batches): the callbacks take the
    per-problem residual counts as a second argument,
    ``args=(PerProblem(y), PerProblem(rows))`` with ``options={'rows': rows}``,
    and write f and J only for the rows r < rows[b]; the padding of the (A, m)
    and (A, m, 4) outputs is left unwritten (the solver never reads it)."""
    lib = lib or L.get_lib()
    if not lib.has("blsq_model_expdecay2"):
        raise L.BlsqError("library built without blsq_models.cu")
    model = getattr(synthetic, model_name)()
    tcache = {}
    last = {}
    inlined = jac_kind == "inlined"
    if rows and (model_name != "ExpDecay2" or inlined):
        raise ValueError("rows-aware callbacks exist for ExpDecay2 with "
                         "jac_kind 'exact' or a finite-difference scheme")

    if model_name == "ExpDecay2":
        def run(X, idx, y, want_j, nrows=None):
            A = X.shape[0]
            t = _t_on(model, X.device, tcache)
            F = torch.empty((A, model.m), dtype=torch.float64, device=X.device)
            J = torch.empty((A, model.m, 4), dtype=torch.float64,
                            device=X.device) if want_j else None
            ip = None if idx is None else idx.data_ptr()
            jp = None if J is None else J.data_ptr()
            X = L.aligned(X.contiguous(), 32)       # the kernels load X with double4
            if nrows is None:
                lib.call("blsq_model_expdecay2", A, ip, model.m, t.data_ptr(),
                         X.data_ptr(), y.data_ptr(), F.data_ptr(), jp, lib.stream(X))
            else:
                if nrows.dtype != torch.int32:
                    raise ValueError("rows-aware callbacks take int32 `rows`")
                lib.call("blsq_model_expdecay2_rows", A, ip, model.m, t.data_ptr(),
                         X.data_ptr(), y.data_ptr(), nrows.data_ptr(), F.data_ptr(), jp,
                         lib.stream(X))
            return F, J

        def fun(X, idx, y, nrows=None):
            # F and J come out of one kernel; J is handed to the `jac` call
            # that follows for the same X and dropped otherwise (the cache
            # never outlives the next callback: 2 GB at the C2 batch size)
            F, J = run(X, idx, y, jac_kind == "exact" and not inlined, nrows)
            last.clear()
            if J is not None:
                last[(X.data_ptr(), X.shape[0])] = J
            return F

        def jac(X, idx, y, nrows=None):
            J = last.pop((X.data_ptr(), X.shape[0]), None)
            last.clear()
            if J is None:
                _, J = run(X, idx, y, True, nrows)
            return J

    elif model_name == "GaussPeak":
        def fun(X, idx, y):
            A = X.shape[0]
            t = _t_on(model, X.device, tcache)
            F = torch.empty((A, model.m), dtype=torch.float64, device=X.device)
            lib.call("blsq_model_gausspeak", A,
                     None if idx is None else idx.data_ptr(), model.m,
                     t.data_ptr(), X.data_ptr(), y.data_ptr(), F.data_ptr(),
                     lib.stream(X))
            return F
        jac = None
    else:
        raise ValueError(model_name)

    if model_name == "ExpDecay2" and jac_kind == "inlined":
        if not lib.has("blsq_model_expdecay2_linearise"):
            raise L.BlsqError("library built without the inlined ExpDecay2 linearisation")

        def linearise(X, idx32, p_istate, p_lin, stream, y):
            """The lin records of the trial points X straight from (X, t, y): the
            model is compiled into the linearisation kernel, J and f never
            touch HBM.  Same bits as fun + jac + blsq_linearise_batched."""
            t = _t_on(model, X.device, tcache)
            lib.call("blsq_model_expdecay2_linearise", X.shape[0],
                     None if idx32 is None else idx32.data_ptr(), model.m,
                     t.data_ptr(), X.data_ptr(), y.data_ptr(), p_istate, p_lin, stream)
            return model.m
        fun.blsq_linearise = linearise
        jac_kind = "exact"
    fun.blsq_indexed = True
    fun.blsq_release = last.clear          # called by the front end when a solve ends
    if jac is not None:
        jac.blsq_indexed = True
    if jac_kind != "exact":
        return fun, jac_kind
    return fun, jac


def tall_callbacks(wl, lib=None):
    """(fun, jac) for the tall workload ``synthetic.TallLinExp[Device]`` as two
    fused kernels: the residual reads the design matrix from the first n-4
    columns of the Jacobian buffer ``wl.J_t``; the Jacobian callback rewrites
    the four exponential columns in place and returns the buffer."""
    lib = lib or L.get_lib()
    if not lib.has("blsq_model_linexp_fun"):
        raise L.BlsqError("library built without blsq_models.cu")

    def fun(x):
        x = x.contiguous()
        F = torch.empty(wl.m, dtype=torch.float64, device=x.device)
        lib.call("blsq_model_linexp_fun", wl.m, wl.n, wl.J_t.data_ptr(),
                 wl.t_t.data_ptr(), wl.y_t.data_ptr(), x.data_ptr(),
                 F.data_ptr(), lib.stream(x))
        return F

    def jac(x):
        x = x.contiguous()
        lib.call("blsq_model_linexp_jac", wl.m, wl.n, wl.J_t.data_ptr(),
                 wl.t_t.data_ptr(), x.data_ptr(), lib.stream(x))
        return wl.J_t

    return fun, jac
