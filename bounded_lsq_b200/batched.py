"""Lock-step driver for B independent bounded problems (batched mode).

One *round* = the user's residual/Jacobian callbacks on the current trial
points, then two CUDA kernels through the C ABI (``include/blsq.h``):

    blsq_linearise_batched   QR of [J | f] per problem      (HBM bound)
    blsq_round_batched       ratio test + accept + next trial step (FP64)

which together advance every running problem by exactly one trial evaluation
of the reference's loops (trf.py:238-352 / dogbox.py:164-267).  The Jacobian is
evaluated at every trial point (speculatively): an accepted step then needs no
second pass, a rejected one reuses the factor kept in the state record.
``nfev`` / ``njev`` are counted as the reference counts them (njev only on
accepted steps).

Finished problems are skipped inside the kernels; the host additionally
compacts the active set (``idx``) so the callbacks only see running problems.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings

import torch

from . import _lib as L

EPS = 2.220446049250313e-16
SQRT_EPS = EPS ** 0.5


class PerProblem:
    """Marks a callback argument as per-problem data with leading dimension B.

    ``args=(PerProblem(y),)``: the callbacks receive ``y`` itself while every
    problem is active and ``y[idx]`` once the active set has been compacted.
    """

    def __init__(self, tensor):
        self.tensor = tensor


def _gather_args(args, kwargs, idx):
    def g(a):
        if isinstance(a, PerProblem):
            if idx is None:
                return a.tensor
            if isinstance(idx, slice):             # contiguous range (prologue)
                return a.tensor[idx]
            return a.tensor.index_select(0, idx)
        return a
    return tuple(g(a) for a in args), {k: g(v) for k, v in kwargs.items()}


class BatchedCallbacks:
    """Adapts user callables ``fun(X, *args, **kwargs)`` to ``fun(X, idx)``."""

    def __init__(self, fun, jac, args=(), kwargs=None, B=None):
        self.fun, self.jac = fun, jac
        self.args, self.kwargs = tuple(args), dict(kwargs or {})
        self.B = B
        self._gathered = (None, None)     # (idx, gathered args) of the last call

    def _raw_args(self, sl):
        """args / kwargs with every per-problem tensor sliced to ``sl`` but not
        gathered: the indexed callbacks take the active ids themselves."""
        def raw(v):
            return v.tensor[sl] if isinstance(v, PerProblem) else v
        return (tuple(raw(v) for v in self.args),
                {n: raw(v) for n, v in self.kwargs.items()})

    def _call(self, fn, X, idx):
        if getattr(fn, "blsq_indexed", False):
            # indexed protocol: raw per-problem tensors + the active ids
            a, k = self._raw_args(idx if isinstance(idx, slice) else slice(None))
            return fn(X, None if isinstance(idx, slice) else idx, *a, **k)
        # the active set only changes when the driver compacts it: gather the
        # per-problem data once per compaction, not once per callback
        if self._gathered[0] is not idx or idx is None:
            self._gathered = (idx, _gather_args(self.args, self.kwargs, idx))
        a, k = self._gathered[1]
        return fn(X, *a, **k)

    def lin(self, X, idx32, off, A, p_istate, p_lin, stream):
        """Models compiled into the linearisation kernel (``fun.blsq_linearise``,
        bounded_lsq_b200.models): returns m when the callbacks of this round
        and blsq_linearise_batched were replaced by that one launch, else None."""
        fn = getattr(self.fun, "blsq_linearise", None)
        if fn is None:
            return None
        sl = slice(off, off + A) if (idx32 is None and (off or A != self.B)) else slice(None)
        a, k = self._raw_args(sl)
        return fn(X, idx32, p_istate, p_lin, stream, *a, **k)

    def f(self, X, idx):
        return self._call(self.fun, X, idx)

    def j(self, X, idx):
        return self._call(self.jac, X, idx)


_SIDE = {}


def _side_stream(dev):
    s = _SIDE.get(dev)
    if s is None:
        s = _SIDE[dev] = torch.cuda.Stream(dev)
    return s


_POOL = {}


def _graph_pool(dev):
    """One private allocator pool per device shared by all tail graphs: its
    segments are reused by the next capture instead of going back to
    cudaMalloc / cudaFree."""
    p = _POOL.get(dev)
    if p is None:
        p = _POOL[dev] = torch.cuda.graph_pool_handle()
    return p


# the allocator drops a pool when the last graph that used it is destroyed:
# the most recent tail graph of each device is kept alive until the next one
# has been captured
_LAST_GRAPH = {}


# callbacks whose capture failed once are not tried again (a failed capture
# costs a device synchronisation and an allocator flush)
_NOT_CAPTURABLE = set()


def _cb_key(fun, jac):
    def k(f):
        f = getattr(f, "__self__", f)             # BatchedCallbacks.f / .j
        return (id(getattr(f, "fun", f)), id(getattr(f, "jac", None)))
    return (k(fun), jac if isinstance(jac, str) else k(jac))


def _as_f64(t, like, what):
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t, dtype=torch.float64, device=like.device)
    if t.dtype != torch.float64:
        t = t.to(torch.float64)
    if t.device != like.device:
        t = t.to(like.device)
    return t


def solve_batched(lib, method, fun, jac, X0, lb, ub, ftol, xtol, gtol,
                  max_nfev, scaling, diff_step=None, check_every=2,
                  compact_below=0.75, tail_below=8192, trace=None,
                  timers=None, graph_tail_rounds=None, prologue=None,
                  prologue_rounds=6, x_covariance=False, rows=None):
    """Run ``method`` ('trf' | 'dogbox') on B problems.

    fun(X, idx) -> (A, m); jac is a callable jac(X, idx) -> (A, m, n) or the
    string '2-point'.  X0 (B, n); lb/ub (n,) or (B, n); scaling (n,) tensor or
    'jac'.  rows: None, or an int32 (B,) tensor on X0's device -- problem b
    has residuals 0 .. rows[b]-1 of the (A, m) callback outputs (ragged batch,
    blsq_linearise_batched_rows / blsq_round_batched_rows).  Returns a dict
    of device tensors (see least_squares_batched).
    """
    meth = {"trf": L.METHOD_TRF, "dogbox": L.METHOD_DOGBOX}[method]
    dev = X0.device
    f64 = torch.float64
    B, n = X0.shape
    if n > L.MAX_BATCHED_N:
        raise ValueError(f"batched mode supports n <= {L.MAX_BATCHED_N}")
    lib.check_tensor(X0, f64, "x0")
    lib.check_tensor(lb, f64, "lb")
    lib.check_tensor(ub, f64, "ub")
    bstride = 0 if lb.dim() == 1 else n
    lay = lib.state_layout(meth, n)
    S = lay["size"]
    LS = lib.lin_record_size(n)
    if max_nfev is None:
        max_nfev = 100 * n                           # trf.py:234-235
    max_nfev = int(max_nfev)
    jac_scaling = isinstance(scaling, str)
    sc_ptr = None if jac_scaling else scaling.data_ptr()
    if not jac_scaling:
        lib.check_tensor(scaling, f64, "scaling")
    fd = isinstance(jac, str)
    fd3 = fd and jac == '3-point'
    npts = 2 * n if fd3 else n                       # callback calls per FD Jacobian
    rel = float("nan") if diff_step is None else float(diff_step)
    rows_max = None
    if rows is not None:
        lib.check_tensor(rows, torch.int32, "rows")
        if rows.shape != (B,):
            raise ValueError("`rows` must have shape (B,).")
        rows_max = int(rows.max().item()) if B else 0

    state = torch.zeros((B, S), dtype=f64, device=dev)
    istate = torch.zeros((B, L.ISTATE_SIZE), dtype=torch.int32, device=dev)
    Xnew = torch.empty((B, n), dtype=f64, device=dev)
    # dogbox evaluates J at the bound-snapped trial (dogbox.py:256-261)
    Xjac = torch.empty((B, n), dtype=f64, device=dev) if method == "dogbox" \
        else None
    lin = torch.empty((B, LS), dtype=f64, device=dev)
    # count[2] = problems still running after the last round (written by the
    # round kernel itself, blsq_round_batched `count`)
    count = torch.zeros(4, dtype=torch.int32, device=dev)
    # TRF: worklist of the problems that leave the Gauss-Newton shortcut
    # (blsq_round_batched `work`)
    rwork = None
    if method == "trf":
        rwork = torch.empty(B + 1, dtype=torch.int32, device=dev)
    rwork_ptr = None if rwork is None else rwork.data_ptr()
    # latency-sized rounds are faster as ONE kernel (measured: the second
    # launch costs the tail what the shortcut saves the bulk)
    TWO_KERNELS_ABOVE = 32768
    if fd:
        Xp = torch.empty((npts, B, n), dtype=f64, device=dev)
        dx = torch.empty((B, 2 * n if fd3 else n), dtype=f64, device=dev)
    stream = lib.stream(X0)
    lib.call("blsq_init_batched", meth, B, n, X0.data_ptr(), lb.data_ptr(),
             ub.data_ptr(), bstride, state.data_ptr(), istate.data_ptr(),
             Xnew.data_ptr(), stream)

    # optional instrumentation (bench.py): CUDA events around every stage
    def tick():
        if timers is None or not X0.is_cuda:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def tock(kind, e0, running):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        timers.setdefault(kind, []).append((e0, e1, running))
    if timers is not None:
        timers["shape"] = (n, None, LS, S)
    nrun = B

    idx = None          # int64 for torch gathers
    idx32 = None        # int32 copy handed to the kernels
    pong, flip, cwork = None, 0, None
    A = B
    first = 1
    m = None
    rounds = 0
    launches = 0

    # the dense entry points unless the batch is ragged (same kernels as
    # before for a dense batch, bit for bit)
    def lin_call(*a):
        if rows is None:
            lib.call("blsq_linearise_batched", *a[:-2], a[-1])
        else:
            lib.call("blsq_linearise_batched_rows", *a)

    def round_call(*a):
        if rows is None:
            lib.call("blsq_round_batched", *a[:-2], a[-1])
        else:
            lib.call("blsq_round_batched_rows", *a)

    def one_round(A, idx, idx32, first, nrun, off=0, count_here=True):
        """Callbacks + linearise + round for the A compacted slots (or, in the
        streaming prologue, for the A problems starting at problem `off`)."""
        nonlocal m, launches
        stream = lib.stream(X0)            # the capture stream inside a graph
        Xa = Xnew[off:off + A]
        Xj = Xa if (Xjac is None or first) else Xjac[off:off + A]
        if idx is None and (off or A != B):
            idx = slice(off, off + A)
        # base pointers of this range of problems
        p_ist = istate.data_ptr() + off * L.ISTATE_SIZE * 4
        p_lin = lin.data_ptr() + off * LS * 8
        p_st = state.data_ptr() + off * S * 8
        p_x0 = X0.data_ptr() + off * n * 8
        p_lb = lb.data_ptr() + off * bstride * 8
        p_ub = ub.data_ptr() + off * bstride * 8
        p_xn = Xnew.data_ptr() + off * n * 8
        p_xj = None if Xjac is None else Xjac.data_ptr() + off * n * 8
        # rows is indexed by problem id like istate: shifted the same way
        p_rows = None if rows is None else rows.data_ptr() + off * 4
        ip = None if idx32 is None else idx32.data_ptr()
        # a model compiled into the linearisation kernel replaces the two
        # callbacks and blsq_linearise_batched of this round by one launch
        cbs = getattr(fun, "__self__", None)
        mm = None
        if not fd and Xjac is None and rows is None and hasattr(cbs, "lin"):
            t0 = tick()
            mm = cbs.lin(Xa, idx32, off, A, p_ist, p_lin, stream)
            if mm is not None:
                m = mm
                launches += 1
                tock("linearise", t0, nrun)
        if mm is None:
            t0 = tick()
            F = _as_f64(fun(Xa, idx), X0, "fun")
            if F.dim() != 2 or F.shape[0] != A:
                raise RuntimeError("batched `fun` must return an (A, m) tensor, "
                                   f"got {tuple(F.shape)} for A={A}")
            F = F.contiguous()
            if m is None:
                m = F.shape[1]
                if rows_max is not None and rows_max > m:
                    raise ValueError(f"`rows` exceeds the {m} residuals `fun` returns "
                                     f"(max(rows) = {rows_max}).")
            elif F.shape[1] != m:
                raise RuntimeError("`fun` changed its number of residuals")
            if not fd:
                J = _as_f64(jac(Xj, idx), X0, "jac")
                if J.dim() != 3 or J.shape[0] != A or J.shape[2] != n:
                    raise RuntimeError("batched `jac` must return an (A, m, n) "
                                       f"tensor, got {tuple(J.shape)}")
                if J.shape[1] != m:
                    raise RuntimeError(
                        "Inconsistent dimensions between the returns of `fun` "
                        "and `jac` on the first iteration.")
                J = L.aligned(J.contiguous(), 32 if n % 4 == 0 else (16 if n % 2 == 0 else 8))
                tock("callbacks", t0, nrun)
                t0 = tick()
                lin_call(A, ip, m, n, F.data_ptr(), J.data_ptr(), None, None, 0,
                         p_ist, p_lin, p_rows, stream)
                tock("linearise", t0, nrun)
            else:
                Xpa = Xp.view(-1)[: npts * A * n].view(npts, A, n)
                lib.call("blsq_fd3_points" if fd3 else "blsq_fd2_points", A, ip, n,
                         Xj.data_ptr(), p_lb, p_ub, bstride, rel,
                         Xpa.data_ptr(), dx.data_ptr(), stream)
                launches += 1
                Fp = []
                for i in range(npts):
                    Fi = _as_f64(fun(Xpa[i], idx), X0, "fun").contiguous()
                    if Fi.shape != F.shape:
                        raise RuntimeError("`fun` changed its output shape")
                    Fp.append(Fi)
                plist = (C.c_void_p * npts)(*[t.data_ptr() for t in Fp])
                tock("callbacks", t0, nrun)
                t0 = tick()
                lin_call(A, ip, m, n, F.data_ptr(), None,
                         C.cast(plist, C.c_void_p), dx.data_ptr(), 2 if fd3 else 1,
                         p_ist, p_lin, p_rows, stream)
                tock("linearise", t0, nrun)
        t0 = tick()
        round_call(meth, A, ip, m, n, p_lin,
                   p_x0, p_lb, p_ub, bstride, sc_ptr,
                   float(ftol), float(xtol), float(gtol), max_nfev, first,
                   p_st, p_ist, p_xn, p_xj,
                   rwork_ptr if A >= TWO_KERNELS_ABOVE else None,
                   count.data_ptr() if count_here else None, p_rows, stream)
        tock("round", t0, nrun)
        if timers is not None:
            timers["shape"] = (n, m, LS, S)
        launches += (2 if (rwork is None or A < TWO_KERNELS_ABOVE) else 3) - \
            (1 if mm is not None else 0)

    def graph_tail(A, idx, idx32, nrun):
        """The latency-sized tail of the batch (A <= tail_below slots, often a
        hundred more rounds for the slowest problems): GRAPH_ROUNDS rounds +
        the status count are captured ONCE into a CUDA graph and replayed, so
        a tail round costs the GPU a few microseconds instead of the host's
        launch path.  Finished problems are skipped inside the kernels, extra
        rounds after the last one finishes are no-ops.  Returns the rounds
        run, or None if the callbacks cannot be captured (host syncs,
        data-dependent shapes): the caller then carries on eagerly."""
        nonlocal launches
        one_round(A, idx, idx32, 0, nrun)       # eager: errors surface here
        r = 1
        l1 = launches
        # torch.cuda.graph() synchronises the device and flushes the caching
        # allocator on entry (every later allocation of the batch would go
        # back to cudaMalloc); capture_begin / capture_end on a side stream
        # do neither.
        # drain the (latency-sized) queue first: measured on the B200, a
        # capture that starts while the eager round is still in flight costs
        # ~16 ms more per solve than the microseconds this wait takes
        torch.cuda.current_stream(dev).synchronize()
        g = torch.cuda.CUDAGraph()
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        side.wait_stream(cur)
        try:
            with torch.cuda.stream(side):
                # thread_local: other threads (NCCL watchdog, NVML sampler)
                # keep making CUDA calls during the capture
                g.capture_begin(pool=_graph_pool(dev),
                                capture_error_mode="thread_local")
                try:
                    for _ in range(GRAPH_ROUNDS):
                        one_round(A, idx, idx32, 0, nrun)
                finally:
                    g.capture_end()
            cur.wait_stream(side)
            _LAST_GRAPH[dev] = g
        except Exception as e:                 # noqa: BLE001
            torch.cuda.synchronize(dev)
            # a capture that died half way leaves the allocator routing this
            # stream to the shared pool: stop that and start a fresh pool
            try:
                torch._C._cuda_endAllocateToPool(dev.index or 0, _graph_pool(dev))
            except Exception:                  # noqa: BLE001
                pass
            _POOL.pop(dev, None)
            _LAST_GRAPH.pop(dev, None)
            launches = l1
            _NOT_CAPTURABLE.add(_cb_key(fun, jac))
            warnings.warn("bounded_lsq_b200: the callbacks could not be "
                          "captured into a CUDA graph (%r); the tail of the "
                          "batch runs as eager rounds" % (e,), RuntimeWarning)
            return r, False
        per_replay = launches - l1
        launches = l1
        while True:
            g.replay()
            launches += per_replay
            r += GRAPH_ROUNDS
            if int(count[2].item()) == 0 or rounds + r > max_nfev + 1:
                return r, True

    if graph_tail_rounds is None:                  # BLSQ_GRAPH_TAIL=0 turns it off
        graph_tail_rounds = int(os.environ.get("BLSQ_GRAPH_TAIL", "8"))
    use_graph = (graph_tail_rounds > 0 and X0.is_cuda and trace is None
                 and timers is None
                 and _cb_key(fun, jac) not in _NOT_CAPTURABLE)
    GRAPH_ROUNDS = int(graph_tail_rounds)
    if prologue:
        # streaming start: the per-problem data arrives from the host in
        # chunks; each chunk runs its first rounds alone while the next one is
        # still on the wire, then the whole batch carries on in lock step
        K = max(1, min(int(prologue_rounds), max_nfev))
        if all(ev is None or ev.query() for _, _, ev in prologue):
            # everything has landed already (a pipelined caller staged this
            # batch under the previous solve): one lock-step start, full-size
            # launches
            prologue = [(0, B, None)]
        for c0, c1, ev in prologue:
            if ev is not None:
                torch.cuda.current_stream(dev).wait_event(ev)
            for r in range(K):
                one_round(c1 - c0, None, None, 1 if r == 0 else 0, c1 - c0, off=c0,
                          count_here=False)
        first = 0
        rounds = K

    def compact(A, idx32, nrun):
        """Ordered compaction on the device (3 small launches) into the other
        half of a ping-pong pair; the nrun problems still running (the round
        kernel's count) fill its first slots."""
        nonlocal pong, flip, cwork, launches, Xnew, Xjac
        if pong is None:
            pong = [dict(X=torch.empty_like(Xnew),
                         J=None if Xjac is None else torch.empty_like(Xjac),
                         i32=torch.empty(A, dtype=torch.int32, device=dev),
                         i64=torch.empty(A, dtype=torch.int64, device=dev)),
                    dict(X=Xnew, J=Xjac,
                         i32=torch.empty(A, dtype=torch.int32, device=dev),
                         i64=torch.empty(A, dtype=torch.int64, device=dev))]
            cwork = torch.empty(int(lib._dll.blsq_compact_work_size(A)),
                                dtype=torch.int32, device=dev)
        o = pong[flip]
        flip ^= 1
        lib.call("blsq_compact_batched", A,
                 None if idx32 is None else idx32.data_ptr(),
                 istate.data_ptr(), n, Xnew.data_ptr(),
                 None if Xjac is None else Xjac.data_ptr(),
                 o["i32"].data_ptr(), o["i64"].data_ptr(),
                 o["X"].data_ptr(),
                 None if Xjac is None else o["J"].data_ptr(),
                 cwork.data_ptr(), lib.stream(X0))
        launches += 3
        Xnew, Xjac = o["X"], o["J"]
        return nrun, o["i64"][:nrun], o["i32"][:nrun]

    while A > 0:
        one_round(A, idx, idx32, first, nrun)
        first = 0
        rounds += 1
        if trace is not None:
            trace(rounds, idx, Xnew[:A], state, istate)
        # host look at the status flags: every second round while the rounds
        # are bandwidth-sized, every 4th once they are launch-latency sized
        every = check_every if A > tail_below else max(check_every, 4)
        if rounds % every == 0 or rounds >= max_nfev:
            nrun = int(count[2].item())               # the one host sync
            if nrun == 0:
                break
            if nrun <= compact_below * A:
                A, idx, idx32 = compact(A, idx32, nrun)
            if use_graph and A <= tail_below:
                r, done = graph_tail(A, idx, idx32, nrun)
                rounds += r
                if done:
                    break
                use_graph = False                     # not capturable: eager
        if rounds > max_nfev + 1:                     # cannot happen
            raise RuntimeError("batched driver failed to terminate")

    status = istate[:, 0].to(torch.int64)
    bad = status < L.STATUS_RUNNING
    if bool(bad.any().item()):
        # trust_region.py:28-35 raises these from inside trf.  One problem:
        # the same exception.  A batch: the other B - 1 fits are valid, so the
        # failing ones keep their negative status (success = False) and the
        # caller is told which they are.
        which = torch.nonzero(bad).view(-1)
        code = int(status[which[0]].item())
        if B == 1:
            if code == L.STATUS_ERR_TR_ZERO:
                raise ValueError("`s` is zero.")
            if code == L.STATUS_ERR_TR_OUTSIDE:
                raise ValueError("`x` is not within the trust region.")
            raise RuntimeError(f"internal status {code}")
        warnings.warn(
            "bounded_lsq_b200: %d of %d problems stopped where the reference "
            "raises ValueError from intersect_trust_region (status %d = `s` is "
            "zero, %d = `x` is not within the trust region); first indices %s"
            % (which.numel(), B, L.STATUS_ERR_TR_ZERO, L.STATUS_ERR_TR_OUTSIDE,
               which[:8].tolist()), RuntimeWarning)

    x = state[:, lay["x"]:lay["x"] + n].contiguous()
    if method == "trf":
        # trf.py:257,354: find_active_constraints(x, lb, ub, rtol=xtol)
        mask = lib.find_active_constraints(x, lb, ub, xtol)
    else:
        mask = torch.empty((B, n), dtype=torch.int64, device=dev)
        lib.call("blsq_dogbox_on_bound", B, n, istate.data_ptr(),
                 mask.data_ptr(), stream)
    cov = None
    if x_covariance:
        # (J^T J)^-1 at the returned x from the triangle the solve holds
        cov = torch.empty((B, n, n), dtype=f64, device=dev)
        lib.call("blsq_covariance", B, n, state.data_ptr(), S, lay["R"], 1,
                 cov.data_ptr(), stream)
    return dict(
        x_covariance=cov,
        x=x, obj_value=state[:, lay["obj"]].clone(),
        optimality=state[:, lay["gnorm"]].clone(), active_mask=mask,
        nfev=istate[:, 1].to(torch.int64), njev=istate[:, 2].to(torch.int64),
        status=status, m=m, rounds=rounds, kernel_launches=launches)


def summarize_timers(timers):
    """Per-kernel totals from the events collected with ``timers=``.

    Algorithmic bytes per running problem (DESIGN.md "Roofline accounting"):
      linearise  8*m*(n+1) read ([J | f]) + 8*LS written (the record)
      round      8*LS read + 2*8*S state read/write + 2*32 istate + 8*n x_new
    """
    if not timers or "linearise" not in timers:
        return {}
    n, m, LS, S = timers["shape"]
    per = {"linearise": 8 * m * (n + 1) + 8 * LS,
           "round": 8 * LS + 16 * S + 64 + 8 * n}
    out = {}
    tot = {}
    for kind in ("callbacks", "linearise", "round"):
        ev = timers.get(kind, [])
        ms = [a.elapsed_time(b) for a, b, _ in ev]
        tot[kind] = sum(ms)
        if kind in per and ms:
            byts = sum(r * per[kind] for _, _, r in ev)
            out[kind] = dict(launches=len(ms), total_ms=tot[kind],
                             avg_ms=tot[kind] / len(ms),
                             gbs=byts / (tot[kind] * 1e-3) / 1e9,
                             bytes_per_problem=per[kind])
            # the launches that still see the whole batch (bandwidth sized)
            rmax = max(r for _, _, r in ev)
            full = [t for t, (_, _, r) in zip(ms, ev) if r == rmax]
            out[kind]["full_batch"] = dict(
                launches=len(full), running=rmax,
                avg_ms=sum(full) / len(full),
                gbs=rmax * per[kind] * len(full) / (sum(full) * 1e-3) / 1e9)
    kt = tot["linearise"] + tot["round"]
    for kind in ("linearise", "round"):
        if kind in out:
            out[kind]["share"] = tot[kind] / kt if kt else None
    out["callbacks_ms"] = tot["callbacks"]
    out["kernels_ms"] = kt
    return out
