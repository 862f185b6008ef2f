"""ctypes binding of the C ABI declared in ``include/blsq.h``.

The shared library is built in-tree (``bounded_lsq_b200/libblsq_b200.so``, see
``__graft_entry__.build``).  There is no fallback: if the library is missing
or a tensor is not on a CUDA device the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# BLSQ_B200_LIB: tuning builds (tools/build_variants.sh); default = in-tree
LIB_PATH = os.environ.get("BLSQ_B200_LIB") or os.path.join(_HERE, "libblsq_b200.so")

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_d = C.c_double

# name -> argtypes; mirrors include/blsq.h one to one
SIGNATURES = {
    "blsq_version": [],
    "blsq_state_layout": [_i, _i, _p],
    "blsq_lin_record_size": [_i],
    "blsq_step_size_to_bound": [_l, _i, _p, _p, _p, _p, _i, _p, _p, _p],
    "blsq_find_active_constraints": [_l, _i, _p, _p, _p, _i, _d, _p, _p],
    "blsq_make_strictly_feasible": [_l, _i, _p, _p, _p, _i, _d, _p, _p],
    "blsq_scaling_vector": [_l, _i, _p, _p, _p, _p, _i, _p, _p, _p],
    "blsq_in_bounds": [_l, _i, _p, _p, _p, _i, _p, _p],
    "blsq_find_intersection": [_l, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p],
    "blsq_covariance": [_l, _i, _p, _l, _i, _i, _p, _p],
    "blsq_fd2_points": [_l, _p, _i, _p, _p, _p, _i, _d, _p, _p, _p],
    "blsq_fd3_points": [_l, _p, _i, _p, _p, _p, _i, _d, _p, _p, _p],
    "blsq_compact_batched": [_l, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "blsq_init_batched": [_i, _l, _i, _p, _p, _p, _i, _p, _p, _p, _p],
    "blsq_linearise_batched": [_l, _p, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p],
    "blsq_round_batched": [_i, _l, _p, _i, _i, _p, _p, _p, _p, _i, _p,
                           _d, _d, _d, _i, _i, _p, _p, _p, _p, _p, _p, _p],
    "blsq_linearise_batched_rows": [_l, _p, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p],
    "blsq_round_batched_rows": [_i, _l, _p, _i, _i, _p, _p, _p, _p, _i, _p,
                                _d, _d, _d, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "blsq_linearise_batched_ld": [_l, _p, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p],
    "blsq_pad_points": [_i, _p, _l, _i, _i, _p, _p],
    "blsq_dogbox_on_bound": [_l, _i, _p, _p, _p],
    "blsq_count_running": [_l, _p, _p, _p, _p],
    "blsq_model_expdecay2": [_l, _p, _i, _p, _p, _p, _p, _p, _p],
    "blsq_model_expdecay2_rows": [_l, _p, _i, _p, _p, _p, _p, _p, _p, _p],
    "blsq_model_gausspeak": [_l, _p, _i, _p, _p, _p, _p, _p],
    "blsq_model_expdecay2_linearise": [_l, _p, _i, _p, _p, _p, _p, _p, _p],
    "blsq_model_linexp_fun": [_l, _i, _p, _p, _p, _p, _p, _p],
    "blsq_model_linexp_jac": [_l, _i, _p, _p, _p, _p],
    "blsq_tall_gram": [_i, _l, _i, _p, _p, _p, _i, _p, _p, _p],
    "blsq_tall_sample_stride": [_l, _i],
    "blsq_tall_factor": [_i, _i, _i, _l, _p, _p, _p],
    "blsq_tall_sumsq": [_l, _p, _p, _p, _p],
    "blsq_tall_layout": [_i, _p],
    "blsq_tall_round": [_i, _i, _i, _l, _i, _p, _p, _p, _p, _p, _p, _d, _d, _d,
                        _i, _i, _i, _p, _p, _p, _p],
}


class PadSegment(C.Structure):
    """blsq_pad_segment (include/blsq.h)."""
    _fields_ = [("off", C.c_int64), ("A", C.c_int64), ("n", C.c_int), ("idx", _p),
                ("x0", _p), ("X", _p), ("Xp", _p)]


METHOD_TRF = 0
METHOD_DOGBOX = 1
ISTATE_SIZE = 8
MAX_BATCHED_N = 16                 # BLSQ_MAX_BATCHED_N
STATUS_RUNNING = -1
STATUS_ERR_TR_ZERO = -101
STATUS_ERR_TR_OUTSIDE = -102


class BlsqError(RuntimeError):
    pass


def _ptr(t):
    if t is None:
        return None
    return t.data_ptr()


def aligned(t, nbytes):
    """``t``, or a copy in a fresh allocation when its address is not a
    multiple of ``nbytes``: the kernels move rows with 128- and 256-bit loads,
    and a contiguous view (e.g. J carved out of one buffer with F) can start
    anywhere."""
    return t if t.data_ptr() % nbytes == 0 else t.clone()


class Lib:
    """Thin checked wrapper: tensors in, raw pointers out."""

    requires_cuda = True

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise BlsqError(
                f"{path} not found: build the CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'). "
                "bounded_lsq_b200 has no CPU fallback.")
        self.path = path
        self._dll = C.CDLL(path)
        self._dll.blsq_error_string.restype = C.c_char_p
        self._dll.blsq_error_string.argtypes = [_i]
        if hasattr(self._dll, "blsq_compact_work_size"):
            self._dll.blsq_compact_work_size.argtypes = [_l]
            self._dll.blsq_compact_work_size.restype = _l
        for name in ("blsq_tall_gram_work_size", "blsq_tall_fac_size",
                     "blsq_tall_record_size"):
            if hasattr(self._dll, name):
                f = getattr(self._dll, name)
                f.argtypes = [_i]
                f.restype = _l
        self._fn = {}
        for name, args in SIGNATURES.items():
            try:
                f = getattr(self._dll, name)
            except AttributeError:
                continue
            f.argtypes = args
            f.restype = _i
            self._fn[name] = f

    # -- plumbing ----------------------------------------------------------
    def device_guard(self, ref):
        """Context manager that makes ``ref``'s device the CUDA current device:
        the kernels are launched on the current device, so it must be the one
        that owns the pointers and the stream (a solve on cuda:1 while cuda:0
        is current would otherwise launch on GPU 0 with GPU 1's memory)."""
        if isinstance(ref, torch.Tensor) and ref.is_cuda:
            return torch.cuda.device(ref.device)
        import contextlib
        return contextlib.nullcontext()

    def same_device(self, ref, **tensors):
        for name, t in tensors.items():
            if isinstance(t, torch.Tensor) and t.device != ref.device:
                raise BlsqError(f"`{name}` is on {t.device} but `x0` is on "
                                f"{ref.device}: all tensors of a solve must "
                                "live on one device")

    def stream(self, ref):
        if ref.is_cuda:
            return torch.cuda.current_stream(ref.device).cuda_stream
        return None

    def check_tensor(self, t, dtype, name):
        if t is None:
            return
        if self.requires_cuda and not t.is_cuda:
            raise BlsqError(f"`{name}` must live on a CUDA device "
                            "(bounded_lsq_b200 has no CPU path)")
        if t.dtype != dtype:
            raise BlsqError(f"`{name}` must be {dtype}, got {t.dtype}")
        if not t.is_contiguous():
            raise BlsqError(f"`{name}` must be contiguous")

    def call(self, name, *args):
        rc = self._fn[name](*args)
        if rc != 0:
            msg = self._dll.blsq_error_string(rc).decode()
            raise BlsqError(f"{name} failed: {msg} (code {rc})")

    def has(self, name):
        return name in self._fn

    # -- layout queries ----------------------------------------------------
    def version(self):
        return self._fn["blsq_version"]()

    def state_layout(self, method, n):
        out = (C.c_int * 9)()
        rc = self._fn["blsq_state_layout"](method, n, C.cast(out, _p))
        if rc != 0:
            raise BlsqError(f"blsq_state_layout({method}, {n}) failed: {rc}")
        keys = ("size", "x", "x_new", "scale", "obj", "delta", "gnorm", "g",
                "alpha")
        d = dict(zip(keys, list(out)))
        d["R"] = d["g"] - n - n * (n + 1) // 2          # R | Q^T f | g are contiguous
        return d

    def tall_layout(self, n):
        out = (C.c_int64 * 17)()
        rc = self._fn["blsq_tall_layout"](n, C.cast(out, _p))
        if rc != 0:
            raise BlsqError(f"blsq_tall_layout({n}) failed: {rc}")
        keys = ("state_size", "istate_size", "x", "x_new", "obj", "delta",
                "gnorm", "on_bound", "fac_size", "R", "qtf", "g", "fobj",
                "info", "rinvp", "scale", "refine")
        d = dict(zip(keys, list(out)))
        d["gram_work"] = int(self._dll.blsq_tall_gram_work_size(n))
        d["record"] = int(self._dll.blsq_tall_record_size(n))
        return d

    def lin_record_size(self, n):
        rc = self._fn["blsq_lin_record_size"](n)
        if rc <= 0:
            raise BlsqError(f"blsq_lin_record_size({n}) failed: {rc}")
        return rc

    # -- elementwise (bounds.py) -------------------------------------------
    def _bounds_args(self, x, lb, ub):
        f64 = torch.float64
        self.check_tensor(x, f64, "x")
        self.check_tensor(lb, f64, "lb")
        self.check_tensor(ub, f64, "ub")
        if x.dim() != 2:
            raise BlsqError("`x` must be (B, n)")
        B, n = x.shape
        if lb.shape == (n,) and ub.shape == (n,):
            bstride = 0
        elif lb.shape == (B, n) and ub.shape == (B, n):
            bstride = n
        else:
            raise BlsqError("bounds must be (n,) or (B, n)")
        return B, n, bstride

    def step_size_to_bound(self, x, d, lb, ub):
        B, n, bs = self._bounds_args(x, lb, ub)
        self.check_tensor(d, torch.float64, "d")
        step = torch.empty(B, dtype=torch.float64, device=x.device)
        hits = torch.empty((B, n), dtype=torch.int64, device=x.device)
        self.call("blsq_step_size_to_bound", B, n, _ptr(x), _ptr(d), _ptr(lb),
                  _ptr(ub), bs, _ptr(step), _ptr(hits), self.stream(x))
        return step, hits

    def find_active_constraints(self, x, lb, ub, rtol):
        B, n, bs = self._bounds_args(x, lb, ub)
        mask = torch.empty((B, n), dtype=torch.int64, device=x.device)
        self.call("blsq_find_active_constraints", B, n, _ptr(x), _ptr(lb),
                  _ptr(ub), bs, float(rtol), _ptr(mask), self.stream(x))
        return mask

    def make_strictly_feasible(self, x, lb, ub, rstep=0.0):
        B, n, bs = self._bounds_args(x, lb, ub)
        out = torch.empty_like(x)
        self.call("blsq_make_strictly_feasible", B, n, _ptr(x), _ptr(lb),
                  _ptr(ub), bs, float(rstep), _ptr(out), self.stream(x))
        return out

    def scaling_vector(self, x, g, lb, ub):
        B, n, bs = self._bounds_args(x, lb, ub)
        self.check_tensor(g, torch.float64, "g")
        v = torch.empty_like(x)
        jv = torch.empty_like(x)
        self.call("blsq_scaling_vector", B, n, _ptr(x), _ptr(g), _ptr(lb),
                  _ptr(ub), bs, _ptr(v), _ptr(jv), self.stream(x))
        return v, jv

    def in_bounds(self, x, lb, ub):
        B, n, bs = self._bounds_args(x, lb, ub)
        ok = torch.empty(B, dtype=torch.uint8, device=x.device)
        self.call("blsq_in_bounds", B, n, _ptr(x), _ptr(lb), _ptr(ub), bs,
                  _ptr(ok), self.stream(x))
        return ok

    def find_intersection(self, x, tr, lb, ub):
        B, n, bs = self._bounds_args(x, lb, ub)
        self.check_tensor(tr, torch.float64, "tr")
        lo = torch.empty_like(x)
        hi = torch.empty_like(x)
        flags = torch.empty((B, n), dtype=torch.uint8, device=x.device)
        self.call("blsq_find_intersection", B, n, _ptr(x), _ptr(tr), _ptr(lb),
                  _ptr(ub), bs, _ptr(lo), _ptr(hi), _ptr(flags),
                  self.stream(x))
        return lo, hi, flags


_LIB = None


def get_lib():
    """The process-wide CUDA library handle (raises if it was not built)."""
    global _LIB
    if _LIB is None:
        _LIB = Lib()
    return _LIB
