"""``least_squares`` front end with the reference's surface.

Mirrors ``bounded_lsq/least_squares.py:120-383`` (argument validation,
callback wrapping, method dispatch, messages) for ``method='trf'|'dogbox'``;
the iterations run in the sm_100a kernels behind ``include/blsq.h``.

Two entry points:

``least_squares``          one problem, exactly the reference's semantics
                           (``x0`` at most 1-D).  Callbacks receive / return
                           torch CUDA float64 tensors.
``least_squares_batched``  B independent problems in lock step: ``x0`` is
                           (B, n), ``fun(X, ...) -> (A, m)``,
                           ``jac(X, ...) -> (A, m, n)``; per-problem callback
                           data is passed as ``PerProblem(tensor)`` in ``args``.

No CPU path: tensors must be CUDA tensors and the CUDA library must be built.
"""
from __future__ import annotations

from warnings import warn

import torch

from . import _lib as L
from .batched import PerProblem, BatchedCallbacks, solve_batched

EPS = 2.220446049250313e-16
SQRT_EPS = EPS ** 0.5

# least_squares.py:30-37
TERMINATION_MESSAGES = {
    0: "The maximum number of function evaluations is exceeded.",
    1: "`gtol` termination condition is satisfied.",
    2: "`ftol` termination condition is satisfied.",
    3: "`xtol` termination condition is satisfied.",
    4: "Both `ftol` and `xtol` termination conditions are satisfied.",
}


class OptimizeResult(dict):
    """Attribute-access dict with the fields of scipy's OptimizeResult
    (least_squares.py:206-252)."""

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:
            raise AttributeError(name) from e

    __setattr__ = dict.__setitem__
    __delattr__ = dict.__delitem__

    def __dir__(self):
        return list(self.keys())


def check_tolerance(ftol, xtol, gtol):
    """least_squares.py:15-27."""
    message = "{} is too low, setting to machine epsilon {}."
    if ftol < EPS:
        warn(message.format("`ftol`", EPS))
        ftol = EPS
    if xtol < EPS:
        warn(message.format("`xtol`", EPS))
        xtol = EPS
    if gtol < EPS:
        warn(message.format("`gtol`", EPS))
        gtol = EPS
    return ftol, xtol, gtol


def _default_device():
    if not torch.cuda.is_available():
        raise L.BlsqError("bounded_lsq_b200 needs a CUDA device (sm_100a); "
                          "there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def _to_f64(a, device):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64)
    return torch.as_tensor(a, dtype=torch.float64, device=device)


def prepare_bounds(bounds, x0):
    """bounds.py:7-16 -- scalar bounds are expanded to x0's last dimension."""
    lb, ub = (_to_f64(b, x0.device) for b in bounds)
    n = x0.shape[-1]
    if lb.dim() == 0:
        lb = lb.expand(n).contiguous()
    if ub.dim() == 0:
        ub = ub.expand(n).contiguous()
    return lb.contiguous(), ub.contiguous()


def check_scaling(scaling, x0, used=None):
    """least_squares.py:100-117 (shared across the batch: shape (n,)).  used:
    only the first `used` entries must be positive (ragged `cols`: the
    entries past the largest count are never read)."""
    if isinstance(scaling, str) and scaling == 'jac':
        return scaling
    try:
        scaling = _to_f64(scaling, x0.device)
    except (ValueError, TypeError, RuntimeError):
        raise ValueError("`scaling` must be 'jac' or array-like with numbers.")
    n = x0.shape[-1]
    if scaling.dim() == 0:
        scaling = scaling.expand(n)
    if used is None:
        if bool(torch.any(scaling <= 0).item()):
            raise ValueError("`scaling` must contain only positive values.")
    if scaling.shape != (n,):
        raise ValueError("Inconsistent shapes between `scaling` and `x0`.")
    if used is not None and bool(torch.any(scaling[:used] <= 0).item()):
        raise ValueError("`scaling` must contain only positive values.")
    return scaling.contiguous()


def _validate_common(method, bounds, jac):
    if method == 'lm':
        raise ValueError("`method='lm'` (MINPACK wrapper, least_squares.py:"
                         "52-97) is outside the B200 hot path; use 'trf' or "
                         "'dogbox'.")
    if method not in ('trf', 'dogbox'):
        raise ValueError("`method` must be 'dogbox', 'trf' or 'lm'.")
    if len(bounds) != 2:
        raise ValueError("`bounds` must contain 2 elements.")
    if jac not in ('2-point', '3-point') and not callable(jac):
        raise ValueError("`jac` must be '2-point', '3-point' or callable.")


def least_squares_batched(fun, x0, jac='2-point', bounds=(-float('inf'), float('inf')),
                          method='trf', ftol=SQRT_EPS, xtol=SQRT_EPS,
                          gtol=SQRT_EPS, max_nfev=None, scaling=1.0,
                          diff_step=None, args=(), kwargs={}, options={},
                          _lib=None):
    """Solve B independent bounded problems (same n, m, method, tolerances).

    x0 : (B, n) with 1 <= n <= 16 (ValueError beyond).  bounds : scalars, (n,)
    or (B, n) tensors.
    fun(X, *args, **kwargs) -> (A, m) and jac(X, *args, **kwargs) -> (A, m, n)
    are called on the A <= B problems still running (rows in problem order);
    wrap per-problem tensors in ``PerProblem`` so they are gathered alike.
    Every field of the result has a leading B dimension.

    ``options``: ``chunk`` (solve the batch that many problems at a time),
    ``x_covariance``, ``h2d_chunks`` / ``device`` (host inputs), ``rows``
    and ``cols`` (ragged batches, below), and the driver knobs of
    ``batched.solve_batched``.

    Ragged batches, ``options={'rows': rows}``: ``rows`` is an integer tensor of
    shape (B,), on the CPU or on the solve's device.  The callbacks keep
    returning dense (A, m) / (A, m, n) tensors, m being the padded width, but
    problem b only has residuals 0 .. rows[b]-1: the rows past it are never
    read and may hold anything, NaN included.  Each problem is solved as the
    reference solves the problem made of its first rows[b] residuals (cost,
    full-rank test, Gauss-Newton certificate, dogbox's rcond).  ``res.fun`` is
    zero past rows[b].  A callback that wants the counts takes them as one more
    argument, ``args=(..., PerProblem(rows))``: they are gathered and chunked
    like the other per-problem data.  Not available with models compiled into
    the linearisation (``models.callbacks(..., 'inlined')``).  Without
    ``rows`` the solve is exactly the dense one.

    Ragged parameter counts, ``options={'cols': cols}``: ``cols`` is an
    integer tensor of shape (B,), on the CPU or on the solve's device, with
    1 <= cols[b] <= n.  Problem b is solved as the reference solves the
    problem made of its first cols[b] parameters: x0, bounds and scaling cut
    to cols[b] entries, ``max_nfev=None`` meaning 100 * cols[b], and every
    n-dependent decision (full-rank test, dogbox's rcond, the norms) taking
    cols[b].  Its other coordinates are held fixed: in every X handed to
    ``fun`` / ``jac`` (trial and finite-difference points) they are x0[b]
    unchanged, so a callback may read them as fixed model parameters, and
    ``res.x`` returns them unchanged.  Jacobian columns past cols[b] are never
    read (they may hold anything, NaN included); bounds and scaling past
    cols[b] are not checked.  ``active_mask`` is 0 and ``x_covariance`` has
    zero rows and columns past cols[b].  The batch runs as one segment per
    distinct count (at most 16), in lock step with one callback call per
    round: the callbacks see the running problems segment by segment (the
    stable sort of the problems by cols[b]), so per-problem data must be
    passed as ``PerProblem`` (or read through the ids of the indexed
    protocol).  ``cols`` works with ``rows``, ``chunk``, per-problem bounds,
    the analytic and finite-difference Jacobians and ``x_covariance``.  Host
    inputs are staged as without it, but the first round waits for every
    copy: the streaming prologue runs the problems in their original order,
    not segment by segment.  Not available with models compiled into the
    linearisation.  Without ``cols`` the solve is exactly the dense one.
    """
    lib = _lib if _lib is not None else L.get_lib()
    _validate_common(method, bounds, jac)
    options = dict(options)
    # the target device: x0's, or options['device'] for host inputs
    if isinstance(x0, torch.Tensor) and x0.is_cuda:
        target = x0.device
    elif lib.requires_cuda:
        target = torch.device(options.get("device") or _default_device())
    else:
        target = None
    guard = torch.cuda.device(target) if target is not None else \
        lib.device_guard(None)
    chunk = options.pop("chunk", None)
    for key in ("rows", "cols"):
        if options.get(key) is not None and getattr(fun, "blsq_linearise", None) is not None:
            raise ValueError(f"`{key}` is not supported with a model compiled into the "
                             "linearisation (models.callbacks(..., 'inlined')).")
    with guard:
        if chunk is not None and isinstance(x0, torch.Tensor) and x0.dim() == 2 \
                and x0.shape[0] > int(chunk) > 0:
            return _least_squares_chunked(lib, int(chunk), fun, x0, jac, bounds, method,
                                          ftol, xtol, gtol, max_nfev, scaling, diff_step,
                                          args, kwargs, options)
        return _least_squares_batched(lib, fun, x0, jac, bounds, method, ftol, xtol,
                                      gtol, max_nfev, scaling, diff_step, args,
                                      kwargs, options)


def _least_squares_chunked(lib, chunk, fun, x0, jac, bounds, method, ftol, xtol, gtol,
                           max_nfev, scaling, diff_step, args, kwargs, options):
    """``options={'chunk': K}``: the batch is solved K problems at a time and the
    results are concatenated -- the working set of a round (callback outputs,
    records) is that of K problems whatever B is (config C3: 10M problems in 1M
    chunks).  Host inputs are staged once for the whole batch; a chunk starts
    when its own copies have landed."""
    B = x0.shape[0]
    plan = None
    rows = options.pop("rows", None)
    cols = options.pop("cols", None)
    if lib.requires_cuda and not x0.is_cuda:
        x0, args, kwargs, plan = _stage_host_inputs(x0, args, kwargs, options)
    else:
        options.pop("h2d_chunks", None)
        options.pop("device", None)
    if rows is not None:
        rows = _check_rows(rows, B, x0.device)         # copied once, sliced per chunk
    if cols is not None:
        cols = _check_cols(cols, B, x0.shape[-1], x0.device)

    def part(v, c0, c1):
        if isinstance(v, PerProblem):
            return PerProblem(v.tensor[c0:c1])
        return v

    def bound(b, c0, c1):
        shape = getattr(b, "shape", ())
        if len(shape) == 2 and shape[0] == B:
            return b[c0:c1]
        return b
    outs = []
    for c0 in range(0, B, chunk):
        c1 = min(B, c0 + chunk)
        if plan is not None:
            cur = torch.cuda.current_stream(x0.device)
            if plan.x0_event is not None:
                cur.wait_event(plan.x0_event)
            for p0, p1, ev in plan:
                if ev is not None and p0 < c1 and p1 > c0:
                    cur.wait_event(ev)
        opts = dict(options)
        if rows is not None:
            opts["rows"] = rows[c0:c1]
        if cols is not None:
            opts["cols"] = cols[c0:c1]
        outs.append(_least_squares_batched(
            lib, fun, x0[c0:c1], jac, (bound(bounds[0], c0, c1), bound(bounds[1], c0, c1)),
            method, ftol, xtol, gtol, max_nfev, scaling, diff_step,
            tuple(part(v, c0, c1) for v in args),
            {k: part(v, c0, c1) for k, v in dict(kwargs).items()}, opts))
    res = OptimizeResult(outs[0])
    for key, v in outs[0].items():
        if isinstance(v, torch.Tensor) and v.dim() >= 1 and v.shape[0] == outs[0].x.shape[0]:
            res[key] = torch.cat([o[key] for o in outs])
    for key in ("rounds", "kernel_launches"):
        if key in res:
            res[key] = sum(o[key] for o in outs)
    return res


def _least_squares_batched(lib, fun, x0, jac, bounds, method, ftol, xtol, gtol,
                           max_nfev, scaling, diff_step, args, kwargs, options):
    if not isinstance(x0, torch.Tensor):
        dev = _default_device() if lib.requires_cuda else torch.device("cpu")
        x0 = torch.as_tensor(x0, dtype=torch.float64, device=dev)
        options.pop("h2d_chunks", None)
        options.pop("device", None)
    elif lib.requires_cuda and not x0.is_cuda:
        # HOST inputs (x0 and the PerProblem data on the CPU, ideally pinned):
        # they are streamed to the device in chunks and the first rounds of
        # each chunk overlap the transfer of the next one
        x0, args, kwargs, plan = _stage_host_inputs(x0, args, kwargs, options)
        if plan is not None and "trace" not in options and options.get("cols") is None:
            options["prologue"] = plan
        elif plan is not None:
            # not streamed (the trace hook wants whole-batch rounds; `cols`
            # runs the problems segment by segment, not in their original
            # order): the copies were queued on the side stream, wait for the
            # last one
            torch.cuda.current_stream(x0.device).wait_event(plan[-1][2])
    else:
        options.pop("h2d_chunks", None)
        options.pop("device", None)
    ev0 = getattr(options.get("prologue"), "x0_event", None)
    if ev0 is not None:                      # staged inputs: x0 is on the copy stream
        torch.cuda.current_stream(x0.device).wait_event(ev0)
    x0 = x0.to(torch.float64).contiguous()
    if x0.dim() != 2:
        raise ValueError("batched `x0` must be (B, n).")
    B, n = x0.shape
    lb, ub = prepare_bounds(bounds, x0)
    for b in (lb, ub):
        if b.shape != (n,) and b.shape != (B, n):
            raise ValueError("Inconsistent shapes between bounds and `x0`.")
    if lb.shape != ub.shape:
        lb = lb.expand(B, n).contiguous()
        ub = ub.expand(B, n).contiguous()
    cols = options.pop("cols", None)
    used = None
    if cols is not None:
        # the coordinates past cols[b] are held fixed: their bounds and
        # scaling are never read and not checked
        cols = _check_cols(cols, B, n, x0.device)
        used = torch.arange(n, device=x0.device)[None, :] < cols[:, None]
    bad = lb >= ub
    if used is not None:
        bad = bad & (used if bad.dim() == 2 else used.any(0))
    if bool(torch.any(bad).item()):
        raise ValueError("Each lower bound mush be strictly less than each "
                         "upper bound.")
    scaling = check_scaling(scaling, x0,
                            None if cols is None else int(cols.max().item()) if B else 0)
    ftol, xtol, gtol = check_tolerance(ftol, xtol, gtol)
    if used is None:
        feasible = lib.in_bounds(x0, lb, ub)
    else:
        inf = torch.tensor(float("inf"), dtype=torch.float64, device=x0.device)
        feasible = lib.in_bounds(torch.where(used, x0, 0.0).contiguous(),
                                 torch.where(used, lb, -inf).contiguous(),
                                 torch.where(used, ub, inf).contiguous())
    if not bool(feasible.all().item()):
        raise ValueError("`x0` is infeasible.")
    for v in list(args) + list(dict(kwargs).values()):
        if isinstance(v, PerProblem):
            lib.same_device(x0, PerProblem=v.tensor)
    rows = options.pop("rows", None)
    if rows is not None:
        rows = _check_rows(rows, B, x0.device)

    cb = BatchedCallbacks(fun, jac, args, kwargs, B)
    jarg = jac if isinstance(jac, str) else cb.j
    out = solve_batched(lib, method, cb.f, jarg, x0, lb, ub, ftol, xtol, gtol,
                        max_nfev, scaling, diff_step=diff_step, rows=rows, cols=cols,
                        **options)
    res = OptimizeResult(out)
    res.fun = cb.f(res.x, None)
    if rows is not None:
        # the padding of a ragged batch is not part of the residual vector
        m = res.fun.shape[1]
        pad = torch.arange(m, device=res.fun.device)[None, :] >= rows[:, None].to(res.fun.device)
        res.fun = res.fun.masked_fill(pad, 0.0)
    release = getattr(fun, "blsq_release", None)
    if callable(release):
        release()                          # callbacks that cache between fun and jac
    # per-problem texts: res.message[int(res.status[b])]
    res.message = dict(TERMINATION_MESSAGES)
    res.message[L.STATUS_ERR_TR_ZERO] = "ValueError: `s` is zero."
    res.message[L.STATUS_ERR_TR_OUTSIDE] = \
        "ValueError: `x` is not within the trust region."
    res.success = res.status > 0
    return res


def _check_rows(rows, B, dev):
    """``options['rows']``: an integer tensor of shape (B,) with every count
    >= 1 (the upper limit m is checked at the first residual evaluation), as
    a contiguous int32 tensor on ``dev``."""
    if not isinstance(rows, torch.Tensor):
        try:
            rows = torch.as_tensor(rows)
        except (TypeError, ValueError, RuntimeError):
            raise ValueError("`rows` must be an integer tensor of shape (B,).")
    if rows.dtype.is_floating_point or rows.dtype.is_complex or rows.dtype == torch.bool:
        raise ValueError(f"`rows` must be an integer tensor, got {rows.dtype}.")
    if tuple(rows.shape) != (B,):
        raise ValueError(f"`rows` must have shape (B,) = ({B},), got {tuple(rows.shape)}.")
    if B:
        if int(rows.min().item()) < 1:
            raise ValueError("`rows` must be at least 1 for every problem.")
        if int(rows.max().item()) > 2 ** 31 - 1:
            raise ValueError("`rows` exceeds the number of residuals.")
    return rows.to(device=dev, dtype=torch.int32).contiguous()


def _check_cols(cols, B, n, dev):
    """``options['cols']``: an integer tensor of shape (B,) with every count
    in 1 .. n, as a contiguous int32 tensor on ``dev``."""
    if not isinstance(cols, torch.Tensor):
        try:
            cols = torch.as_tensor(cols)
        except (TypeError, ValueError, RuntimeError):
            raise ValueError("`cols` must be an integer tensor of shape (B,).")
    if cols.dtype.is_floating_point or cols.dtype.is_complex or cols.dtype == torch.bool:
        raise ValueError(f"`cols` must be an integer tensor, got {cols.dtype}.")
    if tuple(cols.shape) != (B,):
        raise ValueError(f"`cols` must have shape (B,) = ({B},), got {tuple(cols.shape)}.")
    if B:
        if int(cols.min().item()) < 1:
            raise ValueError("`cols` must be at least 1 for every problem.")
        if int(cols.max().item()) > n:
            raise ValueError(f"`cols` exceeds the number of parameters n = {n}.")
    return cols.to(device=dev, dtype=torch.int32).contiguous()


_COPY_STREAM = {}


class _StagePlan(list):
    """[(c0, c1, event)] chunks of a staged batch + the event of the x0 copy."""
    x0_event = None


def stage_host_inputs(x0, args=(), kwargs=None, device=None, h2d_chunks=4, out=None):
    """Start the host-to-device copies of a batched problem's inputs and return
    at once: ``(x0_dev, args_dev, kwargs_dev, plan)``.

    x0 (small) and every CPU ``PerProblem`` tensor (ideally pinned) are copied
    on a side stream, the per-problem data in ``h2d_chunks`` chunks of problems
    with one event per chunk.  Hand the results to ``least_squares_batched(fun,
    x0_dev, args=args_dev, kwargs=kwargs_dev, options={'prologue': plan})``:
    each chunk then runs its first rounds while the next one is still on the
    wire.  ``least_squares_batched`` does exactly this itself when it is called
    with CPU tensors; calling it directly lets a serving loop start the copies
    of the NEXT batch while the current one is being solved.

    out : optional ``(x0_buffer, {id(host tensor): device buffer})`` of
    preallocated device tensors that are not in use (a double-buffering
    caller's second set); without it fresh buffers are allocated and the copy
    stream first waits for the work queued on the current stream.
    """
    dev = torch.device(device) if device is not None else _default_device()
    kwargs = dict(kwargs or {})
    B = x0.shape[0]
    host = [v for v in list(args) + list(kwargs.values())
            if isinstance(v, PerProblem) and not v.tensor.is_cuda]
    for v in host:
        if v.tensor.shape[0] != B:
            raise ValueError("PerProblem data must have leading dimension B.")
    nch = max(1, min(int(h2d_chunks), B // 65536))
    step = -(-B // nch)
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        copy = _COPY_STREAM.get(dev)
        if copy is None:
            copy = _COPY_STREAM[dev] = torch.cuda.Stream(dev)
        if out is None:
            x0d = torch.empty(x0.shape, dtype=x0.dtype, device=dev)
            bufs = {id(v): torch.empty(v.tensor.shape, dtype=v.tensor.dtype, device=dev)
                    for v in host}
            copy.wait_stream(main)          # the buffers were allocated on main
        else:
            x0d, given = out
            bufs = {id(v): given[id(v.tensor)] for v in host}
        plan = _StagePlan()
        with torch.cuda.stream(copy):
            x0d.copy_(x0, non_blocking=True)
            plan.x0_event = torch.cuda.Event()
            plan.x0_event.record(copy)
            for c0 in range(0, B, step):
                c1 = min(B, c0 + step)
                for v in host:
                    bufs[id(v)][c0:c1].copy_(v.tensor[c0:c1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
                plan.append((c0, c1, ev))

    def swap(v):
        return PerProblem(bufs[id(v)]) if id(v) in bufs else v
    return (x0d, tuple(swap(v) for v in args), {k: swap(v) for k, v in kwargs.items()},
            plan)


def _stage_host_inputs(x0, args, kwargs, options):
    """least_squares_batched called with CPU tensors: stage them (see
    stage_host_inputs).  Returns the device x0, the rewritten args / kwargs and
    the [(c0, c1, event)] plan for ``solve_batched(prologue=...)``."""
    dev = options.pop("device", None) or _default_device()
    nch = int(options.pop("h2d_chunks", 4))
    return stage_host_inputs(x0, args, kwargs, device=dev, h2d_chunks=nch)


# A single problem with n <= SINGLE_BATCHED_MAX_N goes to the batched kernels
# (B = 1) unless it is tall: from TALL_FROM_ROWS rows on, the row-sharded Gram
# kernels of tall mode (n >= 2) are the faster path -- one warp folding m rows
# chunk by chunk is not.  Batched mode takes n up to L.MAX_BATCHED_N = 16, but
# a single problem with 9 <= n <= 16 stays on the tall kernels unless
# options={'mode': 'batched'} asks for them.
SINGLE_BATCHED_MAX_N = 8
TALL_FROM_ROWS = 32768


class _RouteToTall(Exception):
    """Raised by the first residual evaluation of a B = 1 batched solve when m
    turns out to be tall (m is only known once `fun` has been called)."""


def _single_callbacks(fun, jac, args, kwargs, dev, tall_from=None):
    """least_squares.py:351-371 on top of the (A=1, ...) batched protocol."""
    seen = [tall_from is None]

    def fun_b(X, idx=None):
        f = fun(X[0], *args, **kwargs)
        f = _to_f64(f, dev)
        if f.dim() == 0:
            f = f.reshape(1)
        if f.dim() > 1:
            raise RuntimeError("`fun` must return at most 1-d array_like.")
        if not seen[0]:
            seen[0] = True
            if f.shape[0] >= tall_from:
                raise _RouteToTall()
        return f.reshape(1, -1)

    if not callable(jac):
        return fun_b, jac

    def jac_b(X, idx=None):
        J = jac(X[0], *args, **kwargs)
        J = _to_f64(J, dev)
        if J.dim() > 2:
            raise RuntimeError("`jac` must return at most 2-d array_like.")
        while J.dim() < 2:
            J = J.unsqueeze(0)
        return J.unsqueeze(0)

    return fun_b, jac_b


def least_squares(fun, x0, jac='2-point', bounds=(-float('inf'), float('inf')),
                  method='trf', ftol=SQRT_EPS, xtol=SQRT_EPS, gtol=SQRT_EPS,
                  max_nfev=None, scaling=1.0, diff_step=None, args=(),
                  kwargs={}, options={}, _lib=None):
    """Drop-in for ``bounded_lsq.least_squares`` (least_squares.py:120-383),
    methods 'trf' and 'dogbox'.

    ``fun(x, *args, **kwargs)`` receives a 1-D float64 CUDA tensor and returns
    the residuals as a tensor (or scalar); ``jac`` likewise returns (m, n).
    Result fields that are arrays in the reference are CUDA tensors here.

    ``x_covariance`` is None as in the reference ('trf' / 'dogbox' leave it
    unset, trf.py:261,358); ``options={'x_covariance': True}`` fills it with
    the field's documented meaning (least_squares.py:248-252: the inverse of
    J^T J at the solution) from the triangular factor the solve already holds.

    Kernels: n <= 8 (SINGLE_BATCHED_MAX_N) runs on the batched kernels (B = 1)
    and n > 8 on the tall ones; a problem with 2 <= n <= 8 and TALL_FROM_ROWS
    or more residuals is moved to the tall kernels after its first residual
    evaluation (that one call is repeated; the solve is then local to this
    process).  ``options={'mode': 'batched' | 'tall'}`` pins the choice
    (batched: n <= 16); with ``mode='tall'`` and an initialised process group
    the callbacks return this rank's rows, as for n > 8.
    """
    lib = _lib if _lib is not None else L.get_lib()
    _validate_common(method, bounds, jac)
    if isinstance(x0, torch.Tensor):
        dev = x0.device
    else:
        dev = _default_device() if lib.requires_cuda else torch.device("cpu")
    with lib.device_guard(torch.empty(0, device=dev)):
        return _least_squares(lib, fun, x0, jac, bounds, method, ftol, xtol, gtol,
                              max_nfev, scaling, diff_step, args, kwargs, options,
                              dev)


def _least_squares(lib, fun, x0, jac, bounds, method, ftol, xtol, gtol, max_nfev,
                   scaling, diff_step, args, kwargs, options, dev):
    x0 = _to_f64(x0, dev)
    if x0.dim() == 0:
        x0 = x0.reshape(1)
    if x0.dim() > 1:
        raise ValueError("`x0` must have at most 1 dimension.")
    n = x0.shape[0]
    lb, ub = prepare_bounds(bounds, x0)
    if lb.shape != x0.shape or ub.shape != x0.shape:
        raise ValueError("Inconsistent shapes between bounds and `x0`.")
    if bool(torch.any(lb >= ub).item()):
        raise ValueError("Each lower bound mush be strictly less than each "
                         "upper bound.")
    scaling = check_scaling(scaling, x0)
    ftol, xtol, gtol = check_tolerance(ftol, xtol, gtol)
    X0 = x0.reshape(1, n).contiguous()
    if not bool(lib.in_bounds(X0, lb, ub).all().item()):
        raise ValueError("`x0` is infeasible.")

    # options['mode'] = 'batched' | 'tall' pins the kernels; by default n and
    # (for 2 <= n <= SINGLE_BATCHED_MAX_N) the number of residuals decide
    options = dict(options)
    mode = options.pop("mode", None)
    if mode not in (None, "batched", "tall"):
        raise ValueError("`options['mode']` must be 'batched' or 'tall'.")
    if mode == "batched" and n > L.MAX_BATCHED_N:
        raise ValueError("batched mode supports n <= %d" % L.MAX_BATCHED_N)
    if mode == "tall" and n < 2:
        raise ValueError("tall mode needs n >= 2")

    def tall():
        from .tall import solve_tall
        return solve_tall(lib, method, fun, jac, x0, lb, ub, ftol, xtol, gtol,
                          max_nfev, scaling, diff_step, args, kwargs, options)

    if mode == "tall" or (mode is None and n > SINGLE_BATCHED_MAX_N):
        return tall()

    probe = TALL_FROM_ROWS if (mode is None and n >= 2 and
                               not {"trace", "timers"} & set(options)) else None
    fun_b, jac_b = _single_callbacks(fun, jac, tuple(args), dict(kwargs), dev, probe)
    # single-problem callbacks are arbitrary user Python (often with host
    # round trips): no CUDA-graph capture unless asked for
    options.setdefault("graph_tail_rounds", 0)
    try:
        out = solve_batched(lib, method, fun_b, jac_b, X0, lb, ub, ftol, xtol,
                            gtol, max_nfev, scaling, diff_step=diff_step,
                            **options)
    except _RouteToTall:
        # m >= TALL_FROM_ROWS: the solve restarts in tall mode (one residual
        # evaluation at x0 was spent to learn m)
        options.pop("graph_tail_rounds", None)
        for k in ("check_every", "compact_below", "tail_below", "prologue",
                  "prologue_rounds"):
            options.pop(k, None)
        # the decision was taken from this process's rows alone, so the solve
        # is local too; rows sharded over ranks need mode='tall' (or n > 8)
        options.setdefault("group", False)
        return tall()
    x = out["x"][0]
    cov = out["x_covariance"]
    if cov is not None:
        # "if the inverse doesn't exist this field is set to None"
        cov = None if bool(torch.isnan(cov[0]).any().item()) else cov[0]
    res = OptimizeResult(
        x=x, fun=fun_b(x.reshape(1, n))[0], obj_value=float(out["obj_value"][0]),
        optimality=float(out["optimality"][0]),
        active_mask=out["active_mask"][0], nfev=int(out["nfev"][0]),
        njev=int(out["njev"][0]), status=int(out["status"][0]),
        x_covariance=cov)
    if callable(jac):
        res.jac = jac_b(x.reshape(1, n))[0]
    else:
        res.jac = fd_jacobian(lib, fun_b, x, res.fun, lb, ub, diff_step, jac)
    res.message = TERMINATION_MESSAGES[res.status]
    res.success = res.status > 0
    return res


def fd_jacobian(lib, fun_b, x, f0, lb, ub, diff_step=None, method='2-point'):
    """Dense finite-difference Jacobian (m, n) at one point through
    blsq_fd2_points / blsq_fd3_points (scipy _dense_difference)."""
    n = x.shape[0]
    f64 = torch.float64
    rel = float("nan") if diff_step is None else float(diff_step)
    xc = x.contiguous()
    if method == '2-point':
        Xp = torch.empty((n, 1, n), dtype=f64, device=x.device)
        dx = torch.empty((1, n), dtype=f64, device=x.device)
        lib.call("blsq_fd2_points", 1, None, n, xc.data_ptr(), lb.data_ptr(),
                 ub.data_ptr(), 0, rel, Xp.data_ptr(), dx.data_ptr(),
                 lib.stream(x))
        cols = [(fun_b(Xp[i])[0] - f0) / dx[0, i] for i in range(n)]
        return torch.stack(cols, dim=1)
    Xp = torch.empty((2 * n, 1, n), dtype=f64, device=x.device)
    dxo = torch.empty((1, 2 * n), dtype=f64, device=x.device)
    lib.call("blsq_fd3_points", 1, None, n, xc.data_ptr(), lb.data_ptr(),
             ub.data_ptr(), 0, rel, Xp.data_ptr(), dxo.data_ptr(), lib.stream(x))
    one = dxo[0, n:].tolist()
    cols = []
    for i in range(n):
        f1, f2 = fun_b(Xp[2 * i])[0], fun_b(Xp[2 * i + 1])[0]
        df = (-3.0 * f0 + 4 * f1 - f2) if one[i] else (f2 - f1)
        cols.append(df / dxo[0, i])
    return torch.stack(cols, dim=1)


def trf(fun, jac, x0, lb, ub, ftol, xtol, gtol, max_nfev, scaling, **options):
    """Positional signature of ``bounded_lsq.trf.trf`` (trf.py:173); ``jac``
    takes ``(x, f)`` like the reference's wrapped Jacobian."""
    return _method_entry('trf', fun, jac, x0, lb, ub, ftol, xtol, gtol,
                         max_nfev, scaling, options)


def dogbox(fun, jac, x0, lb, ub, ftol, xtol, gtol, max_nfev, scaling,
           **options):
    """Positional signature of ``bounded_lsq.dogbox.dogbox`` (dogbox.py:100)."""
    return _method_entry('dogbox', fun, jac, x0, lb, ub, ftol, xtol, gtol,
                         max_nfev, scaling, options)


def _method_entry(method, fun, jac, x0, lb, ub, ftol, xtol, gtol, max_nfev,
                  scaling, options):
    last_f = {}

    def fun_w(x):
        f = fun(x)
        last_f['f'] = f
        return f

    def jac_w(x):
        return jac(x, last_f.get('f'))

    res = least_squares(fun_w, x0, jac=jac_w, bounds=(lb, ub), method=method,
                        ftol=ftol, xtol=xtol, gtol=gtol, max_nfev=max_nfev,
                        scaling=scaling, options=options)
    del res['message'], res['success']
    return res
