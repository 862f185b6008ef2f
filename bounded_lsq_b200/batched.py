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


class _Segment:
    """The problems of one parameter count N: a dense lock-step solve of its
    own (state and lin records, istate, active set, count buffer, compaction)
    whose active slots are one contiguous range of every round's callback
    batch."""


def solve_batched(lib, method, fun, jac, X0, lb, ub, ftol, xtol, gtol,
                  max_nfev, scaling, diff_step=None, check_every=2,
                  compact_below=0.75, tail_below=8192, trace=None,
                  timers=None, graph_tail_rounds=None, prologue=None,
                  prologue_rounds=6, x_covariance=False, rows=None, cols=None):
    """Run ``method`` ('trf' | 'dogbox') on B problems.

    fun(X, idx) -> (A, m); jac is a callable jac(X, idx) -> (A, m, n) or the
    string '2-point'.  X0 (B, n); lb/ub (n,) or (B, n); scaling (n,) tensor or
    'jac'.  rows: None, or an int32 (B,) tensor on X0's device -- problem b
    has residuals 0 .. rows[b]-1 of the (A, m) callback outputs (ragged batch,
    blsq_linearise_batched_rows / blsq_round_batched_rows).  Returns a dict
    of device tensors (see least_squares_batched).

    cols: None, or an int32 (B,) tensor on X0's device with 1 <= cols[b] <= n
    -- problem b has parameters 0 .. cols[b]-1, the others are held at
    X0[b].  The problems are permuted once into segment-major order (a stable
    sort on cols), and each distinct count N is a *segment*: a dense solve
    of N-parameter problems run by the dense N kernels.  The segments share
    one callback call per round: blsq_pad_points writes their active points
    into one padded (A, n) batch (segment after segment, so the callbacks get
    the original problem ids as idx), and each segment linearises its slots
    of the outputs in place (blsq_linearise_batched_ld).  Without cols the
    batch is one segment and the calls are those of a dense solve.
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
    jac_scaling = isinstance(scaling, str)
    sc_ptr = None if jac_scaling else scaling.data_ptr()
    if not jac_scaling:
        lib.check_tensor(scaling, f64, "scaling")
    fd = isinstance(jac, str)
    fd3 = fd and jac == '3-point'
    rel = float("nan") if diff_step is None else float(diff_step)
    rows_max = None
    if rows is not None:
        lib.check_tensor(rows, torch.int32, "rows")
        if rows.shape != (B,):
            raise ValueError("`rows` must have shape (B,).")
        rows_max = int(rows.max().item()) if B else 0
    padded = cols is not None
    if padded:
        lib.check_tensor(cols, torch.int32, "cols")
        if cols.shape != (B,):
            raise ValueError("`cols` must have shape (B,).")

    # latency-sized rounds are faster as ONE kernel (measured: the second
    # launch costs the tail what the shortcut saves the bulk)
    TWO_KERNELS_ABOVE = 32768
    stream = lib.stream(X0)
    perm = None
    if not padded:
        parts = [(n, 0, B)]
    else:
        ch = cols.cpu().to(torch.int64)
        order = torch.argsort(ch, stable=True)
        vals, cnt = torch.unique_consecutive(ch[order], return_counts=True)
        perm = order.to(dev)
        X0p = X0.index_select(0, perm)
        if bstride:
            lbp, ubp = lb.index_select(0, perm), ub.index_select(0, perm)
        rowsp = None if rows is None else rows.index_select(0, perm)
        parts, b0 = [], 0
        for N, c in zip(vals.tolist(), cnt.tolist()):
            parts.append((N, b0, c))
            b0 += c
    # count[k, 2] = problems of segment k still running after the last round
    # (written by the round kernel itself, blsq_round_batched `count`)
    count = torch.zeros((len(parts), 4), dtype=torch.int32, device=dev)
    segs = []
    for k, (N, b0, Bk) in enumerate(parts):
        g = _Segment()
        g.N, g.b0 = N, b0
        if not padded:
            g.x0, g.lb, g.ub, g.bs, g.rows = X0, lb, ub, bstride, rows
        else:
            sl = slice(b0, b0 + Bk)
            g.x0 = X0p[sl, :N].contiguous()
            g.x0pad = X0p[sl]                  # the held coordinates
            g.lb = lbp[sl, :N].contiguous() if bstride else lb[:N]
            g.ub = ubp[sl, :N].contiguous() if bstride else ub[:N]
            g.bs = N if bstride else 0
            g.rows = None if rows is None else rowsp[sl].contiguous()
            g.perm = perm[sl]
        g.lay = lib.state_layout(meth, N)
        g.S = g.lay["size"]
        g.LS = lib.lin_record_size(N)
        g.max_nfev = int(100 * N if max_nfev is None else max_nfev)    # trf.py:234-235
        g.npts = 2 * N if fd3 else N           # callback calls per FD Jacobian
        g.state = torch.zeros((Bk, g.S), dtype=f64, device=dev)
        g.istate = torch.zeros((Bk, L.ISTATE_SIZE), dtype=torch.int32, device=dev)
        g.Xnew = torch.empty((Bk, N), dtype=f64, device=dev)
        # dogbox evaluates J at the bound-snapped trial (dogbox.py:256-261)
        g.Xjac = torch.empty((Bk, N), dtype=f64, device=dev) if method == "dogbox" \
            else None
        g.lin = torch.empty((Bk, g.LS), dtype=f64, device=dev)
        g.count = count[k]
        # TRF: worklist of the problems that leave the Gauss-Newton shortcut
        # (blsq_round_batched `work`)
        g.rwork = torch.empty(Bk + 1, dtype=torch.int32, device=dev) \
            if method == "trf" else None
        if fd:
            g.Xp = torch.empty((g.npts, Bk, N), dtype=f64, device=dev)
            g.dx = torch.empty((Bk, 2 * N if fd3 else N), dtype=f64, device=dev)
        g.A, g.idx, g.idx32 = Bk, None, None   # idx: int64 for torch gathers
        g.pong, g.flip, g.cwork = None, 0, None
        lib.call("blsq_init_batched", meth, Bk, N, g.x0.data_ptr(), g.lb.data_ptr(),
                 g.ub.data_ptr(), g.bs, g.state.data_ptr(), g.istate.data_ptr(),
                 g.Xnew.data_ptr(), stream)
        segs.append(g)
    max_nfev = max(g.max_nfev for g in segs)
    if padded:
        # the padded callback batches, slots in segment order
        Xcb = torch.empty((B, n), dtype=f64, device=dev)
        Xjcb = torch.empty((B, n), dtype=f64, device=dev) if method == "dogbox" else None
        if fd:
            Xpcb = torch.empty((2 * n if fd3 else n, B, n), dtype=f64, device=dev)
    gid = perm              # the callbacks' idx: original ids in slot order

    # optional instrumentation (bench.py): CUDA events around every stage;
    # a ragged-parameter batch keeps the linearise / round events per
    # segment, under timers["segments"][N]
    def tick():
        if timers is None or not X0.is_cuda:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def tock(kind, e0, running, g=None):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        if g is None:
            timers.setdefault(kind, []).append((e0, e1, running))
        else:
            timers.setdefault("segments", {}).setdefault(g.N, {}).setdefault(
                kind, []).append((e0, e1, g.A))
    if timers is not None and not padded:
        timers["shape"] = (n, None, segs[0].LS, segs[0].S)
    nrun = B

    first = 1
    m = None
    rounds = 0
    launches = 0

    # the dense entry points unless the batch is ragged (same kernels as
    # before for a dense batch, bit for bit)
    def lin_call(g, *a):
        if padded:
            lib.call("blsq_linearise_batched_ld", *a[:4], n, *a[4:])
        elif g.rows is None:
            lib.call("blsq_linearise_batched", *a[:-2], a[-1])
        else:
            lib.call("blsq_linearise_batched_rows", *a)

    def round_call(g, *a):
        if g.rows is None:
            lib.call("blsq_round_batched", *a[:-2], a[-1])
        else:
            lib.call("blsq_round_batched_rows", *a)

    def pad(out, fdm, pick, counted=True):
        """blsq_pad_points: the active points of every segment (pick(g) ->
        (X, Xp or None)) into the padded batch `out`."""
        nonlocal launches
        live = [g for g in segs if g.A > 0]
        tab = (L.PadSegment * len(live))()
        s0 = 0
        for i, g in enumerate(live):
            X, Xp = pick(g)
            tab[i] = L.PadSegment(s0, g.A, g.N, None if g.idx32 is None else g.idx32.data_ptr(),
                                  g.x0pad.data_ptr(), X.data_ptr(),
                                  None if Xp is None else Xp.data_ptr())
            s0 += g.A
        lib.call("blsq_pad_points", len(live), C.cast(tab, C.c_void_p), s0, n, fdm,
                 out.data_ptr(), lib.stream(X0))
        launches += counted

    def one_round(first, nrun, pro=None, count_here=True):
        """Callbacks + linearise + round for the active slots of every segment
        (or, in the streaming prologue, pro = (off, A): for the A problems
        starting at problem `off` of the one segment of a dense batch)."""
        nonlocal m, launches
        stream = lib.stream(X0)            # the capture stream inside a graph
        off = 0
        if pro is not None:
            off, A = pro
            live = [(segs[0], A)]
        else:
            live = [(g, g.A) for g in segs if g.A > 0]
            A = sum(a for _, a in live)

        def xj(g):                         # the points J is evaluated at
            return g.Xnew if (g.Xjac is None or first) else g.Xjac
        if padded:
            idx = gid
            Xa = Xcb[:A]
            pad(Xa, 0, lambda g: (g.Xnew, None))
            Xj = Xa
            if Xjcb is not None and not first:
                Xj = Xjcb[:A]
                pad(Xj, 0, lambda g: (g.Xjac, None))
        else:
            g = segs[0]
            Xa = g.Xnew[off:off + A]
            Xj = Xa if (g.Xjac is None or first) else g.Xjac[off:off + A]
            idx = g.idx
            if idx is None and (off or A != B):
                idx = slice(off, off + A)

        # base pointers of this range of problems of each segment
        def ptrs(g):
            return dict(
                ist=g.istate.data_ptr() + off * L.ISTATE_SIZE * 4,
                lin=g.lin.data_ptr() + off * g.LS * 8,
                st=g.state.data_ptr() + off * g.S * 8,
                x0=g.x0.data_ptr() + off * g.N * 8,
                lb=g.lb.data_ptr() + off * g.bs * 8,
                ub=g.ub.data_ptr() + off * g.bs * 8,
                xn=g.Xnew.data_ptr() + off * g.N * 8,
                xj=None if g.Xjac is None else g.Xjac.data_ptr() + off * g.N * 8,
                # rows is indexed by problem id like istate: shifted the same way
                rows=None if g.rows is None else g.rows.data_ptr() + off * 4,
                ip=None if g.idx32 is None else g.idx32.data_ptr())
        P = [ptrs(g) for g, _ in live]
        # a model compiled into the linearisation kernel replaces the two
        # callbacks and blsq_linearise_batched of this round by one launch
        cbs = getattr(fun, "__self__", None)
        mm = None
        if not padded and not fd and segs[0].Xjac is None and segs[0].rows is None \
                and hasattr(cbs, "lin"):
            t0 = tick()
            mm = cbs.lin(Xa, segs[0].idx32, off, A, P[0]["ist"], P[0]["lin"], stream)
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
                # aligned for width n is aligned for every segment's N
                # (lin_ld_width(N, n) divides n)
                J = L.aligned(J.contiguous(), 32 if n % 4 == 0 else (16 if n % 2 == 0 else 8))
                tock("callbacks", t0, nrun)
                s0 = 0
                for (g, a), p in zip(live, P):
                    t0 = tick()
                    lin_call(g, a, p["ip"], m, g.N, F.data_ptr() + s0 * m * 8,
                             J.data_ptr() + s0 * m * n * 8, None, None, 0,
                             p["ist"], p["lin"], p["rows"], stream)
                    tock("linearise", t0, nrun, g if padded else None)
                    s0 += a
            else:
                for (g, a), p in zip(live, P):
                    Xpa = g.Xp.view(-1)[: g.npts * a * g.N].view(g.npts, a, g.N)
                    lib.call("blsq_fd3_points" if fd3 else "blsq_fd2_points", a, p["ip"],
                             g.N, (xj(g) if padded else Xj).data_ptr(),
                             p["lb"], p["ub"], g.bs, rel, Xpa.data_ptr(), g.dx.data_ptr(),
                             stream)
                    launches += 1
                npts = 2 * n if fd3 else n
                if padded:
                    Xpa = Xpcb.view(-1)[: npts * A * n].view(npts, A, n)
                    pad(Xpa, 2 if fd3 else 1, lambda g: (xj(g), g.Xp))
                Fp = []
                for i in range(npts):
                    Fi = _as_f64(fun(Xpa[i], idx), X0, "fun").contiguous()
                    if Fi.shape != F.shape:
                        raise RuntimeError("`fun` changed its output shape")
                    Fp.append(Fi)
                tock("callbacks", t0, nrun)
                s0 = 0
                for (g, a), p in zip(live, P):
                    # segment g reads its slots of the batches of its own N
                    # coordinates; the other batches are not read
                    plist = (C.c_void_p * g.npts)(*[t.data_ptr() + s0 * m * 8
                                                    for t in Fp[:g.npts]])
                    t0 = tick()
                    lin_call(g, a, p["ip"], m, g.N, F.data_ptr() + s0 * m * 8, None,
                             C.cast(plist, C.c_void_p), g.dx.data_ptr(), 2 if fd3 else 1,
                             p["ist"], p["lin"], p["rows"], stream)
                    tock("linearise", t0, nrun, g if padded else None)
                    s0 += a
        for (g, a), p in zip(live, P):
            t0 = tick()
            round_call(g, meth, a, p["ip"], m, g.N, p["lin"],
                       p["x0"], p["lb"], p["ub"], g.bs, sc_ptr,
                       float(ftol), float(xtol), float(gtol), g.max_nfev, first,
                       p["st"], p["ist"], p["xn"], p["xj"],
                       g.rwork.data_ptr() if (g.rwork is not None and a >= TWO_KERNELS_ABOVE)
                       else None,
                       g.count.data_ptr() if count_here else None, p["rows"], stream)
            tock("round", t0, nrun, g if padded else None)
            launches += 2 if (g.rwork is None or a < TWO_KERNELS_ABOVE) else 3
        if timers is not None and not padded:
            timers["shape"] = (n, m, segs[0].LS, segs[0].S)
        launches -= 1 if mm is not None else 0

    def running():
        """Problems still running per segment: the one host sync."""
        return count.cpu()[:, 2].tolist()

    def graph_tail(nrun):
        """The latency-sized tail of the batch (A <= tail_below slots, often a
        hundred more rounds for the slowest problems): GRAPH_ROUNDS rounds +
        the status count are captured ONCE into a CUDA graph and replayed, so
        a tail round costs the GPU a few microseconds instead of the host's
        launch path.  Finished problems are skipped inside the kernels, extra
        rounds after the last one finishes are no-ops.  Returns the rounds
        run, or None if the callbacks cannot be captured (host syncs,
        data-dependent shapes): the caller then carries on eagerly."""
        nonlocal launches
        one_round(0, nrun)                     # eager: errors surface here
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
                        one_round(0, nrun)
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
            if sum(running()) == 0 or rounds + r > max_nfev + 1:
                return r, True

    if graph_tail_rounds is None:                  # BLSQ_GRAPH_TAIL=0 turns it off
        graph_tail_rounds = int(os.environ.get("BLSQ_GRAPH_TAIL", "8"))
    use_graph = (graph_tail_rounds > 0 and X0.is_cuda and trace is None
                 and timers is None
                 and _cb_key(fun, jac) not in _NOT_CAPTURABLE)
    GRAPH_ROUNDS = int(graph_tail_rounds)
    if prologue and padded:
        # the streaming prologue runs the problems in their original order,
        # not in segments: wait for every copy and start in lock step
        for _, _, ev in prologue:
            if ev is not None:
                torch.cuda.current_stream(dev).wait_event(ev)
        prologue = None
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
                one_round(1 if r == 0 else 0, c1 - c0, pro=(c0, c1 - c0), count_here=False)
        first = 0
        rounds = K

    def compact(g, nrun):
        """Ordered compaction of segment g on the device (3 small launches)
        into the other half of a ping-pong pair; the nrun problems still
        running (the round kernel's count) fill its first slots."""
        nonlocal launches
        if g.pong is None:
            g.pong = [dict(X=torch.empty_like(g.Xnew),
                           J=None if g.Xjac is None else torch.empty_like(g.Xjac),
                           i32=torch.empty(g.A, dtype=torch.int32, device=dev),
                           i64=torch.empty(g.A, dtype=torch.int64, device=dev)),
                      dict(X=g.Xnew, J=g.Xjac,
                           i32=torch.empty(g.A, dtype=torch.int32, device=dev),
                           i64=torch.empty(g.A, dtype=torch.int64, device=dev))]
            g.cwork = torch.empty(int(lib._dll.blsq_compact_work_size(g.A)),
                                  dtype=torch.int32, device=dev)
        o = g.pong[g.flip]
        g.flip ^= 1
        lib.call("blsq_compact_batched", g.A,
                 None if g.idx32 is None else g.idx32.data_ptr(),
                 g.istate.data_ptr(), g.N, g.Xnew.data_ptr(),
                 None if g.Xjac is None else g.Xjac.data_ptr(),
                 o["i32"].data_ptr(), o["i64"].data_ptr(),
                 o["X"].data_ptr(),
                 None if g.Xjac is None else o["J"].data_ptr(),
                 g.cwork.data_ptr(), lib.stream(X0))
        launches += 3
        g.Xnew, g.Xjac = o["X"], o["J"]
        g.A, g.idx, g.idx32 = nrun, o["i64"][:nrun], o["i32"][:nrun]

    def trace_view():
        """trace(rounds, idx, X, state, istate) arguments: the next trial
        points of the active slots in callback order, with istate indexed by
        problem id (state: the segments' records of a ragged-parameter batch)."""
        if not padded:
            g = segs[0]
            return g.idx, g.Xnew[:g.A], g.state, g.istate
        X = torch.empty((A, n), dtype=f64, device=dev)
        pad(X, 0, lambda g: (g.Xnew, None), counted=False)
        ist = torch.empty((B, L.ISTATE_SIZE), dtype=torch.int32, device=dev)
        ist[perm] = torch.cat([g.istate for g in segs])
        return gid, X, [g.state for g in segs], ist

    A = B
    while A > 0:
        one_round(first, nrun)
        first = 0
        rounds += 1
        if trace is not None:
            trace(rounds, *trace_view())
        # host look at the status flags: every second round while the rounds
        # are bandwidth-sized, every 4th once they are launch-latency sized
        every = check_every if A > tail_below else max(check_every, 4)
        if rounds % every == 0 or rounds >= max_nfev:
            nrs = running()                           # the one host sync
            nrun = sum(nrs)
            if nrun == 0:
                break
            moved = []
            for g, nr in zip(segs, nrs):
                if g.A and nr <= compact_below * g.A:
                    moved.append((g, int(lib._dll.blsq_compact_work_size(g.A)) - 1))
                    compact(g, nr)
            if moved and padded:
                # the round kernel counts before the deferred TRF pass, which
                # can still finish problems: the slots past the survivors
                # would hold stale ids, and a segment's ids only index its own
                # problems.  The compaction's own survivor counts, one sync.
                surv = torch.stack([g.cwork[w] for g, w in moved]).cpu().tolist()
                for (g, _), s in zip(moved, surv):
                    g.A, g.idx, g.idx32 = s, g.idx[:s], g.idx32[:s]
                    if s == 0:
                        g.count.zero_()       # no longer launched: not running
            A = sum(g.A for g in segs)
            if moved and padded:
                gid = torch.cat([g.perm if g.idx is None else g.perm.index_select(0, g.idx)
                                 for g in segs if g.A > 0])
            if use_graph and A <= tail_below:
                r, done = graph_tail(nrun)
                rounds += r
                if done:
                    break
                use_graph = False                     # not capturable: eager
        if rounds > max_nfev + 1:                     # cannot happen
            raise RuntimeError("batched driver failed to terminate")

    if padded:
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(B, device=dev)

    def gather(t):                                    # segment order -> problem order
        return t if not padded else t.index_select(0, inv)

    def field(f):
        return gather(f(segs[0]) if not padded else torch.cat([f(g) for g in segs]))
    status = field(lambda g: g.istate[:, 0].to(torch.int64))
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

    # per segment; a ragged-parameter batch pads x with x0, active_mask and
    # x_covariance with zeros
    if padded:
        x = X0p.clone()
        mask = torch.zeros((B, n), dtype=torch.int64, device=dev)
        cov = torch.zeros((B, n, n), dtype=f64, device=dev) if x_covariance else None
    for g in segs:
        N, Bk, b1 = g.N, g.state.shape[0], g.b0 + g.state.shape[0]
        xg = g.state[:, g.lay["x"]:g.lay["x"] + N].contiguous()
        if method == "trf":
            # trf.py:257,354: find_active_constraints(x, lb, ub, rtol=xtol)
            mg = lib.find_active_constraints(xg, g.lb, g.ub, xtol)
        else:
            mg = torch.empty((Bk, N), dtype=torch.int64, device=dev)
            lib.call("blsq_dogbox_on_bound", Bk, N, g.istate.data_ptr(),
                     mg.data_ptr(), stream)
        cg = None
        if x_covariance:
            # (J^T J)^-1 at the returned x from the triangle the solve holds
            cg = torch.empty((Bk, N, N), dtype=f64, device=dev)
            lib.call("blsq_covariance", Bk, N, g.state.data_ptr(), g.S, g.lay["R"], 1,
                     cg.data_ptr(), stream)
        if not padded:
            x, mask, cov = xg, mg, cg
        else:
            x[g.b0:b1, :N] = xg
            mask[g.b0:b1, :N] = mg
            if x_covariance:
                cov[g.b0:b1, :N, :N] = cg
    return dict(
        x_covariance=None if cov is None else gather(cov),
        x=gather(x), obj_value=field(lambda g: g.state[:, g.lay["obj"]].clone()),
        optimality=field(lambda g: g.state[:, g.lay["gnorm"]].clone()),
        active_mask=gather(mask),
        nfev=field(lambda g: g.istate[:, 1].to(torch.int64)),
        njev=field(lambda g: g.istate[:, 2].to(torch.int64)),
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
