"""Driver for ONE tall problem (tall mode): m up to 1e8 rows, 8 < n <= 256.

The callbacks return this rank's rows of the residual vector / Jacobian
(``fun(x) -> (m_local,)``, ``jac(x) -> (m_local, n)``, CUDA float64, row
major); x, the bounds and every n-sized quantity are replicated on all ranks.
Per accepted step the rank runs CholeskyQR2 on ``[J | f]`` through the C ABI
(``include/blsq.h``, "tall mode"):

    blsq_tall_gram(1) -> all-gather -> blsq_tall_factor(1)      R1, g, f.f
    blsq_tall_gram(2) -> all-gather -> blsq_tall_factor(2)      R, Q^T f

and per trial point ``blsq_tall_sumsq`` + ``blsq_tall_round`` (judge, then
propose).  Everything after the factorisation is n x n (SURVEY section 7: with
J = QR the hat-space SVD, the quadratic models and the Gauss-Newton /
Cauchy steps only need R, Q^T f and g), so a trial costs one ``fun`` call.

Multi-GPU (one process per GPU, ``torch.distributed``): rows are split by
rank, the only exchanges are the two all-gathers of the (n*n + n + 1)-double
Gram records per Jacobian and one all-gather of a double per trial; every rank
sums the gathered records in rank order, so all ranks take bit-identical
steps.  The loop follows trf.py:238-352 / dogbox.py:164-267; counters and
statuses are the reference's.
"""
from __future__ import annotations

import torch

from . import _lib as L


def _dist(group):
    import torch.distributed as dist
    if group is False:                    # this process alone, whatever is initialised
        return None, 1, 0
    if group is None and not (dist.is_available() and dist.is_initialized()):
        return None, 1, 0
    return dist, dist.get_world_size(group), dist.get_rank(group)


class _Gather:
    """All-gather of small per-rank records into a preallocated (nranks, k)
    tensor: ONE collective call, no list of outputs and no stack."""

    def __init__(self, group):
        self.group = group
        self.dist, self.nranks, self.rank = _dist(group)
        self._out = {}

    def __call__(self, rec):
        if self.nranks == 1:
            return rec.view(1, -1)
        rec = rec.contiguous()
        key = (rec.numel(), rec.dtype, rec.device)
        out = self._out.get(key)
        if out is None:
            out = self._out[key] = torch.empty((self.nranks, rec.numel()),
                                               dtype=rec.dtype, device=rec.device)
        self.dist.all_gather_into_tensor(out.view(-1), rec.view(-1), group=self.group)
        return out

    def sum_int(self, v, device):
        if self.nranks == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device=device)
        self.dist.all_reduce(t, group=self.group)
        return int(t.item())


def _fd_jacobian_tall(lib, fun, x, f0, lb, ub, diff_step, st, method='2-point'):
    """Finite-difference Jacobian of this rank's rows (least_squares.py:
    357-365): n ('2-point') or 2n ('3-point') extra ``fun`` calls at scipy's
    bound-aware points (blsq_fd2_points / blsq_fd3_points, bit exact)."""
    n = x.shape[0]
    f64 = torch.float64
    rel = float("nan") if diff_step is None else float(diff_step)
    J = torch.empty((f0.shape[0], n), dtype=f64, device=x.device)
    xc = x.contiguous()
    if method == '2-point':
        Xp = torch.empty((n, 1, n), dtype=f64, device=x.device)
        dx = torch.empty((1, n), dtype=f64, device=x.device)
        lib.call("blsq_fd2_points", 1, None, n, xc.data_ptr(), lb.data_ptr(),
                 ub.data_ptr(), 0, rel, Xp.data_ptr(), dx.data_ptr(), st)
        for i in range(n):
            J[:, i] = (fun(Xp[i, 0]) - f0) / dx[0, i]
        return J
    Xp = torch.empty((2 * n, 1, n), dtype=f64, device=x.device)
    dxo = torch.empty((1, 2 * n), dtype=f64, device=x.device)
    lib.call("blsq_fd3_points", 1, None, n, xc.data_ptr(), lb.data_ptr(),
             ub.data_ptr(), 0, rel, Xp.data_ptr(), dxo.data_ptr(), st)
    one = dxo[0, n:].tolist()                            # host sync (n flags)
    for i in range(n):
        f1, f2 = fun(Xp[2 * i, 0]), fun(Xp[2 * i + 1, 0])
        df = (-3.0 * f0 + 4 * f1 - f2) if one[i] else (f2 - f1)
        J[:, i] = df / dxo[0, i]
    return J


def solve_tall(lib, method, fun, jac, x0, lb, ub, ftol, xtol, gtol, max_nfev,
               scaling, diff_step=None, args=(), kwargs=None, options=None):
    """Run 'trf' | 'dogbox' on one tall problem.  Returns an OptimizeResult
    with the reference's fields (tensors for the array-valued ones)."""
    from .least_squares import OptimizeResult, TERMINATION_MESSAGES
    opts = dict(options or {})
    group = opts.pop("group", None)
    timers = opts.pop("timers", None)
    trace = opts.pop("trace", None)
    want_cov = bool(opts.pop("x_covariance", False))
    if opts:
        # trf.py:173 / dogbox.py:100 accept no extra options
        raise TypeError(f"{method}() got an unexpected keyword argument "
                        f"'{sorted(opts)[0]}'")
    kwargs = dict(kwargs or {})
    args = tuple(args)
    meth = {"trf": L.METHOD_TRF, "dogbox": L.METHOD_DOGBOX}[method]
    dev = x0.device
    f64 = torch.float64
    n = x0.shape[0]
    if n > 256:
        raise ValueError("tall mode supports n <= 256")
    lay = lib.tall_layout(n)
    gather = _Gather(group)
    nranks = gather.nranks
    if max_nfev is None:
        max_nfev = 100 * n                              # trf.py:234-235
    max_nfev = int(max_nfev)
    jac_scaling = isinstance(scaling, str)
    sc_ptr = None if jac_scaling else scaling.data_ptr()
    st = lib.stream(x0)

    def call_fun(x):
        f = fun(x, *args, **kwargs)
        if not isinstance(f, torch.Tensor):
            f = torch.as_tensor(f, dtype=f64, device=dev)
        if f.dim() == 0:
            f = f.reshape(1)
        if f.dim() > 1:
            raise RuntimeError("`fun` must return at most 1-d array_like.")
        # blsq_tall_gram moves rows with 16-byte bulk copies
        return L.aligned(f.to(f64).contiguous(), 16)

    def call_jac(x, f):
        if callable(jac):
            J = jac(x, *args, **kwargs)
            if not isinstance(J, torch.Tensor):
                J = torch.as_tensor(J, dtype=f64, device=dev)
            if J.dim() > 2:
                raise RuntimeError("`jac` must return at most 2-d array_like.")
            while J.dim() < 2:
                J = J.unsqueeze(0)
            J = J.to(f64)
        else:
            J = _fd_jacobian_tall(lib, call_fun, x, f, lb, ub, diff_step, st, jac)
        return L.aligned(J.contiguous(), 16)

    state = torch.zeros(lay["state_size"], dtype=f64, device=dev)
    istate = torch.zeros(lay["istate_size"], dtype=torch.int32, device=dev)
    fac = torch.zeros(lay["fac_size"], dtype=f64, device=dev)
    gwork = torch.empty(max(lay["gram_work"], 1), dtype=f64, device=dev)
    swork = torch.empty(4096, dtype=f64, device=dev)
    rwork = torch.empty(n * n, dtype=f64, device=dev)
    GS = lay["record"]
    rec = torch.empty(GS, dtype=f64, device=dev)
    ssq = torch.empty(1, dtype=f64, device=dev)
    x_view = state[lay["x"]:lay["x"] + n]
    xnew_view = state[lay["x_new"]:lay["x_new"] + n]

    def tick():
        if timers is None or not x0.is_cuda:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def tock(kind, e0):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        timers.setdefault(kind, []).append((e0, e1))

    launches = [0]

    def round_(phase, first, new_lin, parts=None, m_total=0):
        launches[0] += 1
        lib.call("blsq_tall_round", meth, phase, n, m_total, nranks,
                 None if parts is None else parts.data_ptr(), fac.data_ptr(),
                 x0.data_ptr(), lb.data_ptr(), ub.data_ptr(), sc_ptr,
                 float(ftol), float(xtol), float(gtol), max_nfev, first,
                 new_lin, state.data_ptr(), istate.data_ptr(),
                 rwork.data_ptr(), st)

    def gram(p, J, f, sstride):
        launches[0] += 2                        # gram + reduce
        t0 = tick()
        lib.call("blsq_tall_gram", p, J.shape[0], n, J.data_ptr(), f.data_ptr(),
                 fac[lay["rinvp"]:].data_ptr(), sstride, gwork.data_ptr(),
                 rec.data_ptr(), st)
        tock("gram%d" % p, t0)
        return gather(rec)

    def factor(p, recs):
        launches[0] += 1
        t0 = tick()
        lib.call("blsq_tall_factor", p, n, nranks, GS,
                 None if recs is None else recs.data_ptr(), fac.data_ptr(), st)
        tock("factor", t0)

    def factorise(J, f):
        # preconditioner from a sample of the row tiles (all of them for
        # small m: then this is CholeskyQR2), one exact pass, verified
        sstride = int(lib._fn["blsq_tall_sample_stride"](J.shape[0], n))
        if nranks > 1:
            # every rank must take the same decision below
            sstride = max(int(s) for s in gather(torch.tensor(
                [float(sstride)], dtype=f64, device=dev)).view(-1).tolist())
        factor(1, gram(1, J, f, sstride))
        factor(2, gram(2, J, f, 1))
        # the verification of pass 2 asks for another pass when cond(J R1^-1)
        # is not O(1): a sampled first pass that missed rows that matter, or
        # an ill-conditioned J whose first Cholesky needed a diagonal shift
        # (shifted CholeskyQR3: kappa up to ~1e12 comes out as accurate as a
        # Householder factor; trf.py:272 / dogbox.py:197 never fail there)
        for _ in range(3):
            if float(fac[lay["refine"]].item()) == 0.0:         # host sync
                break
            factor(3, None)
            factor(2, gram(2, J, f, 1))

    round_(0, 1, 0)
    first = 1
    m_total = None
    f_cur = J_cur = None
    while True:
        t0 = tick()
        f_new = call_fun(xnew_view)
        tock("fun", t0)
        if m_total is None:
            m_total = gather.sum_int(f_new.shape[0], dev)
        elif f_cur is not None and f_new.shape != f_cur.shape:
            raise RuntimeError("`fun` changed its number of residuals")
        launches[0] += 2
        t0 = tick()
        lib.call("blsq_tall_sumsq", f_new.shape[0], f_new.data_ptr(),
                 swork.data_ptr(), ssq.data_ptr(), st)
        parts = gather(ssq).view(-1)
        round_(1, first, 0, parts, m_total)
        tock("judge", t0)
        head = istate[:4].tolist()                       # host sync
        status, accepted = head[0], head[3]
        new_lin = 0
        if accepted:
            f_cur = f_new
            if status == L.STATUS_RUNNING:
                t0 = tick()
                J_cur = call_jac(x_view, f_cur)
                tock("jac", t0)
                if J_cur.dim() != 2 or J_cur.shape[1] != n:
                    raise RuntimeError("`jac` must return an (m, n) tensor, "
                                       f"got {tuple(J_cur.shape)}")
                if J_cur.shape[0] != f_cur.shape[0]:
                    raise RuntimeError(
                        "Inconsistent dimensions between the returns of `fun` "
                        "and `jac` on the first iteration.")
                factorise(J_cur, f_cur)
                new_lin = 1
            else:
                J_cur = None                              # evaluated below
        if status != L.STATUS_RUNNING:
            break
        t0 = tick()
        round_(2, first, new_lin, None, m_total)
        tock("propose", t0)
        first = 0
        if trace is not None:
            trace(xnew_view.clone(), state, istate)
        # (reading the status here instead of calling `fun` once more than the
        # reference does: a 20 us look against a 1.5 ms callback at C4)
        status = int(istate[0].item())                   # host sync
        if status != L.STATUS_RUNNING:
            break

    if status < L.STATUS_RUNNING:
        if status == L.STATUS_ERR_TR_ZERO:
            raise ValueError("`s` is zero.")
        if status == L.STATUS_ERR_TR_OUTSIDE:
            raise ValueError("`x` is not within the trust region.")
        raise RuntimeError(f"internal status {status}")
    info = float(fac[lay["info"]].item())
    gnorm = float(state[lay["gnorm"]].item())
    if info != 0.0 and not (status == 1 and gnorm == 0.0):
        # the shifted Cholesky only gives up on a Jacobian with NaN / inf
        # entries (scipy.linalg.svd, trf.py:272, raises on those too); an
        # all-zero Jacobian ends above with g = 0 -> status 1 like the reference
        raise ValueError(
            "tall mode: the Jacobian contains infs or NaNs "
            f"(factorisation info {info:.0f})")

    x = x_view.clone()
    if J_cur is None:
        J_cur = call_jac(x, f_cur)
    if method == "trf":
        mask = lib.find_active_constraints(x.view(1, n), lb, ub, xtol)[0]
    else:
        ob = lay["on_bound"]
        mask = istate[ob:ob + n].to(torch.int64)
    ist = istate[:4].tolist()
    cov = None
    if want_cov and info == 0.0:
        # (J^T J)^-1 = R^-1 R^-T from the factor at the returned x
        cov = torch.empty((n, n), dtype=f64, device=dev)
        lib.call("blsq_covariance", 1, n, fac.data_ptr(), 0, lay["R"], 0,
                 cov.data_ptr(), st)
        if bool(torch.isnan(cov).any().item()):
            cov = None
    res = OptimizeResult(
        x=x, fun=f_cur, jac=J_cur, obj_value=float(state[lay["obj"]].item()),
        optimality=float(state[lay["gnorm"]].item()), active_mask=mask,
        nfev=ist[1], njev=ist[2], status=ist[0], x_covariance=cov)
    res.message = TERMINATION_MESSAGES[res.status]
    res.success = res.status > 0
    res.kernel_launches = launches[0]
    res.m_total = m_total
    return res
