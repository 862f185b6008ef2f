"""Fused CUDA residual/Jacobian callbacks for the synthetic workloads.

``compile_model`` compiles a residual model written by the user as a small
CUDA C++ struct (contract: ``csrc/blsq_user_model.cuh``) into callbacks of the
same protocol, whose inlined kinds run the model inside the linearisation
kernel.

User-side code (include/blsq_models.h): the same functions as
``synthetic.ExpDecay2.fun_t/jac_t`` and ``synthetic.GaussPeak.fun_t`` as one
kernel each, with the active-set gather of the per-problem data fused into
the load.  They use the *indexed* callback protocol of the batched driver:
``fun(X, idx, *args)`` with ``fun.blsq_indexed = True`` receives the raw
per-problem tensors plus the active problem ids instead of gathered copies.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

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

        def linearise(X, Xjac, Xp, dx, idx32, p_istate, p_lin, stream, y):
            """The lin records of the trial points X straight from (X, t, y): the
            model is compiled into the linearisation kernel, J and f never
            touch HBM.  Same bits as fun + jac + blsq_linearise_batched.  TRF
            rounds only: dogbox's Jacobian points and finite differences are
            declined (None), those rounds call fun and jac."""
            if Xjac is not None or Xp is not None:
                return None
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


# ---- residual models compiled from user source ------------------------------

_PKG = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG, "csrc")
# what a compiled model is built from besides its source: part of the cache key
_HEADERS = [os.path.join(_CSRC, f) for f in ("blsq_user_model.cuh", "blsq_dual.cuh",
                                             "blsq_lin.cuh", "blsq_core.cuh", "Makefile")] + \
           [os.path.join(_PKG, "..", "include", "blsq.h")]
MAX_DATA = 8                              # BLSQ_MODEL_MAX_DATA
KINDS = ("exact", "2-point", "3-point", "inlined", "inlined-2-point")
_JACOBIAN = {0: None, 1: "analytic", 2: "autodiff"}     # blsq_um_info out[1]
_NVCC_VERSION = {}
_LOADED = {}


def _nvcc():
    """The nvcc that `make` in csrc/ runs for the library: $NVCC, else PATH."""
    exe = shutil.which(os.environ.get("NVCC", "nvcc"))
    if exe is None:
        raise L.BlsqError("nvcc not found: compile_model needs the CUDA toolkit "
                          "that builds the library (nvcc on PATH or $NVCC)")
    if exe not in _NVCC_VERSION:
        _NVCC_VERSION[exe] = subprocess.run([exe, "--version"], capture_output=True,
                                            text=True, check=True).stdout
    return exe, _NVCC_VERSION[exe]


def _default_cache_dir():
    base = os.environ.get("XDG_CACHE_HOME") or os.path.join(os.path.expanduser("~"), ".cache")
    return os.path.join(base, "bounded_lsq_b200", "models")


def generated_source(source, name="Model"):
    """The .cu that compile_model builds: the contract header, the user's
    source (diagnostics point at its own lines) and the entry points."""
    if not name.isidentifier():
        raise ValueError(f"model name {name!r} is not a C++ identifier")
    return ('#include "blsq_user_model.cuh"\n'
            '#line 1 "model.cu"\n'
            f"{source}\n"
            f"BLSQ_USER_MODEL_ENTRY_POINTS({name})\n")


def compile_model(source, name="Model", cache_dir=None):
    """Compile the residual model ``name`` defined in ``source`` (CUDA C++,
    contract in ``csrc/blsq_user_model.cuh``) for sm_100a with the library's
    own flags and return a :class:`CompiledModel`.

    The shared object is cached under ``cache_dir`` (default: a per-user cache
    directory) by a hash of the generated source, the headers it includes, the
    Makefile (the flags) and ``nvcc --version``; a cached object is loaded
    without running nvcc.  It is written under a temporary name and renamed,
    so concurrent processes compiling the same model do not collide.  A
    compile error raises BlsqError with nvcc's diagnostics."""
    cu = generated_source(source, name)
    nvcc, version = _nvcc()
    h = hashlib.sha256()
    for part in [cu.encode(), version.encode()] + [open(p, "rb").read() for p in _HEADERS]:
        h.update(hashlib.sha256(part).digest())
    key = h.hexdigest()[:32]
    cache_dir = os.path.abspath(cache_dir or _default_cache_dir())
    path = os.path.join(cache_dir, f"blsq_model_{key}.so")
    log = path[:-3] + ".ptxas.log"
    built = False
    if not os.path.exists(path):
        os.makedirs(cache_dir, exist_ok=True)
        with tempfile.TemporaryDirectory(dir=cache_dir, prefix=".build-") as tmp:
            src = os.path.join(tmp, "model.cu")
            with open(src, "w") as f:
                f.write(cu)
            out = os.path.join(tmp, "model.so")
            r = subprocess.run(["make", "-s", "-C", _CSRC, "user-model", f"NVCC={nvcc}",
                                f"SRC={src}", f"OUT={out}"], capture_output=True, text=True)
            if r.returncode != 0 or not os.path.exists(out):
                raise L.BlsqError(f"compile_model({name!r}): nvcc failed\n{r.stderr}{r.stdout}")
            with open(os.path.join(tmp, "ptxas.log"), "w") as f:
                f.write(r.stderr)
            os.replace(os.path.join(tmp, "ptxas.log"), log)
            os.replace(out, path)
        built = True
    if path not in _LOADED:
        _LOADED[path] = C.CDLL(path)
    return CompiledModel(_LOADED[path], path, name, built)


_p, _i, _l = C.c_void_p, C.c_int, C.c_int64
_UM_SIGNATURES = {
    "blsq_um_info": [_p],
    "blsq_um_linearise": [_l, _p, _i, _p, _p, _p, _i, _p, _p, _p],
    "blsq_um_linearise_fd2": [_l, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p],
    "blsq_um_fun": [_l, _p, _i, _p, _p, _i, _p, _p],
    "blsq_um_jac": [_l, _p, _i, _p, _p, _i, _p, _p],
}


class CompiledModel:
    """A residual model compiled by :func:`compile_model`.

    ``n``: its number of parameters; ``jacobian``: where its Jacobian rows
    come from, ``'analytic'`` (its ``jacobian_row``), ``'autodiff'`` (derived
    from a residual templated on the scalar type by forward-mode dual
    numbers) or None; ``has_jacobian``: ``jacobian is not None``; ``path``:
    the shared object; ``built``: whether this call ran nvcc (False: loaded
    from the cache)."""

    def __init__(self, dll, path, name, built):
        self._dll, self.path, self.name, self.built = dll, path, name, built
        for fn, args in _UM_SIGNATURES.items():
            getattr(dll, fn).argtypes = args
            getattr(dll, fn).restype = _i
        dll.blsq_um_error_string.argtypes = [_i]
        dll.blsq_um_error_string.restype = C.c_char_p
        info = (C.c_int * 3)()
        dll.blsq_um_info(info)
        self.n, self.jacobian, self.version = info[0], _JACOBIAN[info[1]], info[2]
        self.has_jacobian = self.jacobian is not None

    def _call(self, fn, *args):
        rc = getattr(self._dll, fn)(*args)
        if rc != 0:
            msg = self._dll.blsq_um_error_string(rc).decode()
            raise L.BlsqError(f"{self.name}: {fn} failed: {msg} (code {rc})")

    def _data(self, X, data):
        if len(data) > MAX_DATA:
            raise ValueError(f"a compiled model takes at most {MAX_DATA} data tensors, "
                             f"got {len(data)}")
        for k, d in enumerate(data):
            if not isinstance(d, torch.Tensor) or d.dtype != torch.float64 \
                    or not d.is_contiguous() or not d.is_cuda or d.device != X.device:
                raise ValueError(
                    f"data argument {k} of a compiled model must be a contiguous float64 "
                    f"tensor on the solve's CUDA device {X.device} (a PerProblem or shared "
                    "argument), got "
                    + (f"{d.dtype} on {d.device}" if isinstance(d, torch.Tensor)
                       else type(d).__name__))
        return (C.c_void_p * MAX_DATA)(*[d.data_ptr() for d in data]), len(data)

    def callbacks(self, jac_kind, m, lib=None):
        """(fun, jac) for ``least_squares_batched(fun, x0, jac=jac, args=data)``
        with m residuals per problem, as ``models.callbacks`` returns them:

        * ``'exact'``: materialised F and J kernels (needs a Jacobian:
          ``jacobian_row`` or a templated residual);
        * ``'2-point'``, ``'3-point'``: the materialised F kernel and the
          scheme's name; the solver forms the differences;
        * ``'inlined'``: the model compiled into the linearisation kernel,
          J and f never reach HBM (needs a Jacobian, as ``'exact'``);
        * ``'inlined-2-point'``: 2-point differences formed in registers in
          the linearisation kernel, f and the perturbed batches never reach HBM.

        The data (the callbacks' ``args``: at most 8 contiguous float64 tensors
        on the solve's device, ``PerProblem`` or shared) reach the model as
        ``blsq_model_ctx::data`` in order.  The inlined kinds serve every
        round of a dense TRF or dogbox solve; they do not take ``rows`` or
        ``cols``.

        A derived Jacobian (``jacobian == 'autodiff'``) is exact up to
        rounding; TRF rows take J and f from one dual evaluation, dogbox rows
        J from the dual at the Jacobian point and f from the double residual.
        Both routes give the same bits, as they do with ``jacobian_row``."""
        if jac_kind not in KINDS:
            raise ValueError(f"jac_kind must be one of {KINDS}, got {jac_kind!r}")
        if jac_kind in ("exact", "inlined") and not self.has_jacobian:
            raise ValueError(f"{self.name} defines no jacobian_row and its residual is not a "
                             f"template on the scalar type: jac_kind {jac_kind!r} needs one "
                             "of them (or use '2-point' or 'inlined-2-point')")
        m = int(m)
        if m < 1:
            raise ValueError("m must be >= 1")
        lib = lib or L.get_lib()
        if not lib.requires_cuda:
            raise L.BlsqError("compiled models run on CUDA devices only; the "
                              "host-emulation library cannot run them")
        n = self.n

        def run(entry, X, idx, data, shape):
            ptrs, nd = self._data(X, data)
            X = X.contiguous()
            out = torch.empty(shape, dtype=torch.float64, device=X.device)
            self._call(entry, X.shape[0], None if idx is None else idx.data_ptr(), m,
                       X.data_ptr(), ptrs, nd, out.data_ptr(), lib.stream(X))
            return out

        def fun(X, idx, *data):
            return run("blsq_um_fun", X, idx, data, (X.shape[0], m))

        def jac(X, idx, *data):
            return run("blsq_um_jac", X, idx, data, (X.shape[0], m, n))

        fun.blsq_indexed = True
        jac.blsq_indexed = True
        if jac_kind == "inlined":
            def linearise(X, Xjac, Xp, dx, idx32, p_istate, p_lin, stream, *data):
                """lin records of the trial points X, J at Xjac (dogbox) or X."""
                if Xp is not None:
                    return None
                ptrs, nd = self._data(X, data)
                self._call("blsq_um_linearise", X.shape[0],
                           None if idx32 is None else idx32.data_ptr(), m, X.data_ptr(),
                           None if Xjac is None else Xjac.data_ptr(), ptrs, nd,
                           p_istate, p_lin, stream)
                return m
            fun.blsq_linearise = linearise
        elif jac_kind == "inlined-2-point":
            def linearise(X, Xjac, Xp, dx, idx32, p_istate, p_lin, stream, *data):
                """lin records from f at X and at the 2-point batches Xp."""
                if Xp is None:
                    return None
                ptrs, nd = self._data(X, data)
                self._call("blsq_um_linearise_fd2", X.shape[0],
                           None if idx32 is None else idx32.data_ptr(), m, X.data_ptr(),
                           Xp.data_ptr(), dx.data_ptr(), ptrs, nd, p_istate, p_lin, stream)
                return m
            fun.blsq_linearise = linearise
            return fun, "2-point"
        if jac_kind in ("2-point", "3-point"):
            return fun, jac_kind
        return fun, jac
