"""Batched mode for 9 <= n <= 16 parameters per problem.

The instances for N = 9..16 (csrc/blsq_batched_wide.cu) have their own
lin_kernel class table: lane groups of 16 or 32 and MULTI, no 8-lane class
(lane k stores row k of R), with LinCfg<N, true>::RPL rows per lane.  The
round kernel runs the per-thread code of N <= 8.

Every check takes ``lib`` and a torch device: the unmarked tests run them on
the host emulation built from tests/host_emul/emul_wide.cpp (emul.cpp and the
ragged entry points of emul_rows.cpp, dispatching n = 1..16), the
``gpu``-marked ones on the CUDA library.  A single problem with n > 8 still goes to the tall kernels unless
options={'mode': 'batched'} asks for the batched ones."""
import contextlib
import ctypes as C
import os
import subprocess
import warnings

import numpy as np
import pytest
import torch

import cases
import hostemul
import test_linearise_accuracy as tla
from cases import T, bits
from test_ragged_batches import FIELDS, RandModel, same
from bounded_lsq_b200 import PerProblem, least_squares, least_squares_batched
from bounded_lsq_b200 import _lib as L

EMUL_WIDE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emul",
                         "emul_wide.cpp")
WIDE = range(9, 17)
CLASSES = ("G16", "G32", "MULTI")


def quiet(fn, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return fn(*a, **k)


# --------------------------------------------------- lin_kernel class table --

def rpl(N):
    """Rows per lane of lin_kernel for N = 9..16 (LinCfg<N, true>::RPL)."""
    return 4 if N <= 12 else 2


def lin_class(N, m):
    """The class launch_lin picks for N > 8: the smallest group of 16 or 32
    lanes whose registers hold all m rows, else MULTI."""
    for G, name in ((16, "G16"), (32, "G32")):
        if m <= G * rpl(N):
            return name
    return "MULTI"


def widths(N):
    """m at both sides of both class edges of N, a MULTI width with a partial
    last chunk, plus m = 1 < n, m = n - 1 and m = n."""
    e16, e32 = 16 * rpl(N), 32 * rpl(N)
    return sorted({1, N - 1, N, e16, e16 + 1, e32, e32 + 1, 3 * e32 + 5})


_gate_record = tla.gate_record


def gate_record(rec, N, m, G, ref, fam, stats, fails, key):
    """test_linearise_accuracy.gate_record with the R gate at 8 N u |a_j|
    (64 at N = 8): each of the N projections of modified Gram-Schmidt adds
    O(u |a_j|) to column j of R.  Measured: the serial host emulation reaches
    84 u |a_j| at N = 16, kappa = 1e12."""
    n0 = len(fails)
    _gate_record(rec, N, m, G, ref, fam, stats, fails, key)
    fails[n0:] = [f for f in fails[n0:] if not (f[1] == "R" and f[3] <= 8 * N)]


@contextlib.contextmanager
def wide_tables():
    """test_linearise_accuracy's checks with the N > 8 class table and R gate."""
    saved = tla.lin_class, tla.widths, tla.gate_record
    tla.lin_class, tla.widths, tla.gate_record = lin_class, widths, gate_record
    try:
        yield
    finally:
        tla.lin_class, tla.widths, tla.gate_record = saved


# ------------------------------------------------------------------ checks --

def check_layouts(lib, dev):
    """The state and record layouts of n = 9..16 keep the invariants of
    n <= 8 (TRF records and their blocks on multiples of 4 doubles), and n = 17
    is refused."""
    assert L.MAX_BATCHED_N == 16
    for method in (L.METHOD_TRF, L.METHOD_DOGBOX):
        for n in WIDE:
            lay = lib.state_layout(method, n)
            assert lay["size"] > 3 * n and lay["x"] == 0 and lay["x_new"] >= n
            if method == L.METHOD_TRF:
                assert lay["size"] % 4 == 0 and lay["x_new"] % 4 == 0
                assert all(lay[k] % 4 == 0 for k in ("scale", "delta")), lay
            assert lib.lin_record_size(n) % 4 == 0
        with pytest.raises(L.BlsqError):
            lib.state_layout(method, 17)
    assert lib._dll.blsq_lin_record_size(17) < 0


def check_single_problem_routing(lib, dev):
    """least_squares with 9 <= n <= 16 runs on the tall kernels by default and
    on the batched ones with options={'mode': 'batched'}; the trace callback
    shows which: (x_new, state, istate) for tall, (round, idx, Xnew, state,
    istate) for batched.  Both give the oracle's status and x."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(3)
    for n in WIDE:
        m = 2 * n + 3
        A = rng.standard_normal((m, n))
        y = A @ rng.uniform(-1, 1, n) + 0.01 * rng.standard_normal(m)
        lb, ub, x0 = np.full(n, -0.5), np.full(n, 0.6), np.zeros(n)
        At, yt = T(A, dev), T(y, dev)
        ref = orc.least_squares(lambda x: A @ x - y, x0, jac=lambda x: A,
                                bounds=(lb, ub))
        for mode, nargs in ((None, 3), ("batched", 5)):
            seen = []
            opts = dict(trace=lambda *a, s=seen: s.append(len(a)))
            if mode:
                opts["mode"] = mode
            r = least_squares(lambda x: At @ x - yt, T(x0, dev), jac=lambda x: At,
                              bounds=(T(lb, dev), T(ub, dev)), options=opts, _lib=lib)
            assert seen and set(seen) == {nargs}, (n, mode, seen)
            assert r.status == ref.status, (n, mode)
            assert np.allclose(r.x.cpu().numpy(), ref.x, rtol=1e-8, atol=1e-10), (n, mode)
    with pytest.raises(ValueError):
        least_squares(lambda x: x, T(np.zeros(17), dev), options=dict(mode="batched"),
                      _lib=lib)
    with pytest.raises(ValueError):
        least_squares_batched(lambda X: X, T(np.zeros((2, 17)), dev), _lib=lib)


def check_lin_records(lib, dev, Ns=WIDE):
    """test_linearise_accuracy.check_every_instance for N = 9..16 with the
    N > 8 class table: the exact-Gram / mpmath reference, the R, Q^T f,
    backward, g and f.f gates and the bit-exact invariances, at both sides of
    every class edge and at m < n and m = n."""
    with wide_tables():
        return tla.check_every_instance(lib, dev, Ns=Ns)


def check_all_lin_instances(lib, dev):
    report, run = check_lin_records(lib, dev)
    want = {(N, c, mo) for N in WIDE for c in CLASSES for mo in (0, 1, 2)}
    assert run.dense == want and len(want) == 72, sorted(want - run.dense)
    if lib.requires_cuda:
        assert run.rows == want, sorted(want - run.rows)
    return report


def check_corpus(lib, dev, copies=3):
    """Every corpus.npz instance with 9 <= n <= 16, solved as ONE batch of
    `copies` identical problems with per-problem (B, n) bounds, under the gates
    of cases.check_corpus_single and its measured waivers; the copies agree
    bit for bit."""
    cs, z, probs = cases.corpus_cases(max_n=16)
    cs = [c for c in cs if probs[c[0]].n >= 9]
    assert cs
    stats = dict(total=0, exact_status=0, waived=0, fd_total=0, fd_exact=0)
    for name, method, jm, sc in cs:
        p = probs[name]
        key = f"{name}|{method}|{jm}|{sc}|"
        obj, status, nfev, njev, opt, ntr = z[key + "scalars"]

        def evaluate(X, what, p=p):
            Xh = X.cpu().numpy()
            return T(np.stack([np.asarray(p.fun(x) if what == "fun" else p.jac(x), dtype=float)
                               for x in Xh]), dev)
        trials = []

        def trace(r, idx, Xn, state, istate):
            if not trials:
                trials.append(Xn.cpu().numpy().copy())
        tile = lambda v: T(np.tile(v, (copies, 1)), dev)            # noqa: E731
        res = quiet(least_squares_batched, lambda X: evaluate(X, "fun"), tile(p.x0),
                    jac=(lambda X: evaluate(X, "jac")) if jm == "exact" else jm,
                    bounds=(tile(p.lb), tile(p.ub)), method=method,
                    scaling='jac' if sc == 'jac' else 1.0,
                    options=dict(trace=trace, graph_tail_rounds=0), _lib=lib)
        for f in ("x", "obj_value", "status", "nfev", "njev", "active_mask"):
            v = getattr(res, f).cpu().numpy()
            assert all(bits(v[b], v[0]) for b in range(copies)), (key, f)
        x = res.x[0].cpu().numpy()
        st, nf, nj = int(res.status[0]), int(res.nfev[0]), int(res.njev[0])
        ob = float(res.obj_value[0])
        stats["total"] += 1
        assert np.all(x >= p.lb) and np.all(x <= p.ub), key
        assert st >= 0, key
        gt = z[key + "trials"]
        if trials and not np.isnan(gt[0]).any() and \
                not cases.first_step_sensitive(z, name, method, sc):
            stepn = max(np.abs(gt[0] - p.x0).max(), 1e-300)
            e0 = float(np.abs(trials[0][0] - gt[0]).max() / stepn)
            stats["first_step_rel"] = max(stats.get("first_step_rel", 0.0), e0)
            assert e0 < 1e-10, (key, e0)
        waived, tol = cases.self_sensitive(z, key)
        if jm != "exact":
            base_waived, _ = cases.self_sensitive(z, f"{name}|{method}|exact|{sc}|")
            if status > 0 and st > 0 and obj > 1e-20 and not base_waived:
                assert abs(ob - obj) <= 1e-3 * max(obj, 1e-9), (key, ob, obj)
            if not base_waived:
                stats["fd_total"] += 1
                stats["fd_exact"] += (st == int(status) and nf == int(nfev))
            continue
        if waived:
            stats["waived"] += 1
            if status > 0 and st > 0 and obj > 1e-20:
                assert abs(ob - obj) <= tol * max(obj, 1e-9), (key, ob, obj, tol)
            continue
        assert st == int(status), (key, st, status)
        assert nf == int(nfev) and nj == int(njev), key
        assert bits(res.active_mask[0].cpu().numpy(), z[key + "mask"]), key
        gx = z[key + "x"]
        assert np.allclose(x, gx, rtol=1e-8, atol=1e-8 * np.abs(gx).max()), (key, x, gx)
        assert abs(ob - obj) <= 1e-8 * obj + 1e-18, key
        stats["exact_status"] += 1
    # finite differences: status and nfev are counted.  Over the 33 counted runs
    # of n >= 9 the tall kernels match 31 and this path 30 on the host
    # emulation; the misses are runs of 89 - 339 evaluations (PenaltyII10_B,
    # Trigonometric_B) whose count the 1e-8 noise of the difference quotient
    # decides.  check_corpus_single's 0.93 is a fraction over all n.
    assert stats["fd_exact"] >= 0.9 * stats["fd_total"], stats
    print("corpus 9 <= n <= 16:", stats)
    return stats


def check_vs_oracle(lib, dev, B=8, seed=42):
    """Random bounded problems for n = 9..16, both methods, scaling 1.0 and
    'jac', analytic / 2-point / 3-point Jacobians, bounds active at many
    solutions: the gates of cases.check_random_small_vs_oracle (cost 1e-8 for
    every problem; status, nfev, x and the active set identical for >= 99 %;
    finite differences: the cost only).  Every eighth batch has m < n: status
    -102 where the oracle raises, its status and nfev otherwise."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    tot = dict(total=0, exact=0, under=0, under_ok=0)
    k = 0
    for n in WIDE:
        for method in ("trf", "dogbox"):
            for scaling in (1.0, "jac"):
                for jac in ("exact", "2-point", "3-point"):
                    k += 1
                    W = n - 2 if k % 8 == 0 else int(rng.integers(n, 3 * n + 6))
                    mdl = RandModel(n, W, B, np.full(B, W), seed=int(rng.integers(1 << 30)))
                    res = mdl.solve(lib, dev, jac, method, rows=False, scaling=scaling)
                    X = res.x.cpu().numpy()
                    assert np.all(X >= mdl.lb) and np.all(X <= mdl.ub)
                    st, nf = res.status.cpu().numpy(), res.nfev.cpu().numpy()
                    ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
                    for b in range(B):
                        yb = mdl.y[b]
                        try:
                            ref = quiet(
                                orc.least_squares,
                                lambda x: mdl.A @ x + 0.3 * np.sin(mdl.Bm @ x) - yb, mdl.x0,
                                jac=(lambda x: mdl.A + 0.3 * np.cos(mdl.Bm @ x)[:, None] * mdl.Bm)
                                if jac == "exact" else jac,
                                bounds=(mdl.lb, mdl.ub), method=method, scaling=scaling)
                        except ValueError as e:
                            assert "not within the trust region" in str(e)
                            tot["under"] += 1
                            tot["under_ok"] += st[b] == -102
                            continue
                        if W < n:
                            tot["under"] += 1
                            if st[b] >= 0:
                                assert abs(ob[b] - ref.obj_value) <= \
                                    1e-6 * ref.obj_value + 1e-18, (n, method, b)
                            tot["under_ok"] += (st[b] == ref.status and nf[b] == ref.nfev)
                            continue
                        tot["total"] += 1
                        assert abs(ob[b] - ref.obj_value) <= 1e-8 * ref.obj_value + 1e-18, \
                            (n, method, scaling, jac, b)
                        if jac == "exact":
                            tot["exact"] += (
                                st[b] == ref.status and nf[b] == ref.nfev and
                                np.allclose(X[b], ref.x, rtol=1e-8, atol=1e-9) and
                                np.array_equal(mk[b], np.asarray(ref.active_mask)))
                        else:
                            tot["exact"] += 1 if np.array_equal(
                                mk[b], np.asarray(ref.active_mask)) else 0
    assert tot["exact"] >= 0.99 * tot["total"], tot
    assert tot["under"] > 0 and tot["under_ok"] >= 0.83 * tot["under"], tot
    print("random n = 9..16 vs oracle:", tot)
    return tot


def check_coordinate_15(lib, dev, B=12):
    """n = 16 with the target of coordinate 15 below its lower bound in half
    of the problems and above its upper bound in the other half: the last 2-bit
    field of istate (bits 30-31) decodes to active_mask[:, 15] = -1 / +1, equal
    to the oracle's, for dogbox (on_bound) and TRF (find_active_constraints)."""
    from oracle import blsq_oracle as orc
    n, m = 16, 40
    rng = np.random.default_rng(15)
    A = rng.standard_normal((m, n))
    xt = rng.uniform(-0.4, 0.4, (B, n))
    xt[:, 15] = np.where(np.arange(B) % 2 == 0, -3.0, 3.0)
    y = xt @ A.T
    lb, ub, x0 = np.full(n, -1.0), np.full(n, 1.0), np.zeros(n)
    At = T(A, dev)
    for method in ("dogbox", "trf"):
        res = least_squares_batched(
            lambda X, Y: X @ At.T - Y, T(np.tile(x0, (B, 1)), dev),
            jac=lambda X, Y: At[None].expand(X.shape[0], m, n),
            bounds=(T(lb, dev), T(ub, dev)), method=method, args=(PerProblem(T(y, dev)),),
            _lib=lib)
        mk = res.active_mask.cpu().numpy()
        want = np.where(np.arange(B) % 2 == 0, -1, 1)
        assert np.array_equal(mk[:, 15], want), (method, mk[:, 15])
        for b in range(B):
            ref = orc.least_squares(lambda x: A @ x - y[b], x0, jac=lambda x: A,
                                    bounds=(lb, ub), method=method)
            assert np.array_equal(mk[b], np.asarray(ref.active_mask)), (method, b)


def check_invariances(lib, dev, graph=False):
    """n = 12 and 16: permutation and subsets of the batch, chunk, the
    compaction thresholds and (graph) the CUDA-graph tail give the same bits
    per problem; a ragged problem gives the bits of the dense solve of its
    truncated residuals within one lane-group class; NaN instead of zeros in
    the padding changes no bit."""
    rng = np.random.default_rng(12)
    for n in (12, 16):
        B = 160
        W = 16 * rpl(n)                         # G16 for every count
        for jac, method in (("exact", "trf"), ("2-point", "dogbox"), ("3-point", "trf")):
            mdl = RandModel(n, W, B, np.full(B, W), seed=n + B)
            base = mdl.solve(lib, dev, jac, method, rows=False, graph_tail_rounds=0,
                             compact_below=0.0, x_covariance=True)
            perm = rng.permutation(B)
            same(mdl.solve(lib, dev, jac, method, sel=perm, rows=False, x_covariance=True),
                 base, "perm", sel2=perm)
            sub = np.sort(rng.choice(B, 37, replace=False))
            same(mdl.solve(lib, dev, jac, method, sel=sub, rows=False, x_covariance=True),
                 base, "subset", sel2=sub)
            same(mdl.solve(lib, dev, jac, method, rows=False, chunk=48, x_covariance=True),
                 base, "chunk")
            for opts in (dict(compact_below=1.0), dict(check_every=3, compact_below=0.5)):
                same(mdl.solve(lib, dev, jac, method, rows=False, graph_tail_rounds=0,
                               x_covariance=True, **opts), base, opts)
            if graph:
                for opts in (dict(), dict(graph_tail_rounds=3, tail_below=100)):
                    same(mdl.solve(lib, dev, jac, method, rows=False, x_covariance=True,
                                   **opts), base, ("graph", opts))
        # ragged: counts n - 1 .. W, all in the G16 class of width W
        Br = 24
        rows = rng.integers(n - 1, W + 1, Br)
        rows[0], rows[-1] = n - 1, W
        for jac, method in (("exact", "dogbox"), ("2-point", "trf")):
            rag = RandModel(n, W, Br, rows, seed=7 * n)
            zero = RandModel(n, W, Br, rows, seed=7 * n, pad=0.0)
            r1 = rag.solve(lib, dev, jac, method, x_covariance=True)
            same(zero.solve(lib, dev, jac, method, x_covariance=True), r1, ("nan pad", n))
            for r in np.unique(rows)[:4]:
                sel = np.nonzero(rows == r)[0]
                solo = np.concatenate([sel, sel]) if len(sel) == 1 else sel
                den = rag.solve(lib, dev, jac, method, sel=solo, r=int(r), x_covariance=True)
                same(r1, den, (n, jac, method, int(r)), sel1=sel, sel2=slice(0, len(sel)))


def check_covariance(lib, dev):
    """blsq_covariance on packed records (the batched x_covariance) for
    n = 9..16 against test_linearise_accuracy's exact-integer inverse, same
    gate: 4 x NumPy's error + 4 n u max|C|."""
    rng = np.random.default_rng(29)
    for n in WIDE:
        B = 6
        Rs = np.triu(rng.standard_normal((B, n, n)))
        for b in range(B):
            Rs[b][np.diag_indices(n)] = np.ldexp(rng.uniform(1, 2, n), rng.integers(-8, 9, n))
        NT = n * (n + 1) // 2
        rec = np.zeros((B, NT + 3))
        for b in range(B):
            rec[b, :NT] = [Rs[b, i, j] for i in range(n) for j in range(i, n)]
        rt = T(rec, dev)
        ct = torch.empty((B, n, n), dtype=torch.float64, device=dev)
        lib.call("blsq_covariance", B, n, rt.data_ptr(), NT + 3, 0, 1, ct.data_ptr(),
                 lib.stream(rt))
        got = ct.cpu().numpy()
        for b in range(B):
            Cs = tla.exact_cov(Rs[b])
            Ri = np.linalg.inv(Rs[b])
            gate = 4 * np.abs(Ri @ Ri.T - Cs).max() + 4 * n * tla.U * np.abs(Cs).max()
            assert np.abs(got[b] - Cs).max() <= gate, (n, b)
    # end to end: x_covariance of a batched solve against (J^T J)^-1 at its x
    for n in (9, 12, 16):
        mdl = RandModel(n, 3 * n, 6, np.full(6, 3 * n), seed=n)
        r = mdl.solve(lib, dev, "exact", "trf", rows=False, x_covariance=True)
        X, Cv = r.x.cpu().numpy(), r.x_covariance.cpu().numpy()
        for b in range(6):
            J = mdl.A + 0.3 * np.cos(mdl.Bm @ X[b])[:, None] * mdl.Bm
            Ti = np.linalg.inv(np.linalg.qr(J, mode="r"))
            ref = Ti @ Ti.T
            assert np.abs(Cv[b] - ref).max() <= 1e-8 * np.abs(ref).max(), (n, b)


# ------------------------------------------------------- GPU-only checks --

def check_abi_errors(lib, dev):
    """blsq_linearise_batched: a J misaligned for the vector loads of n = 10,
    14 (16 bytes) and 12, 16 (32 bytes) and a null Fp_host[j] return
    BLSQ_E_BADARG before any launch."""
    dll = lib._dll
    for n in (10, 12, 14, 16):
        m, A = 8, 4
        buf = torch.zeros(A * m * n + 8, dtype=torch.float64, device=dev)
        F = torch.zeros((A, m), dtype=torch.float64, device=dev)
        ist = torch.full((A, 8), -1, dtype=torch.int32, device=dev)
        lin = torch.zeros((A, lib.lin_record_size(n)), dtype=torch.float64, device=dev)
        base = buf.data_ptr()
        assert base % 256 == 0
        ok = dll.blsq_linearise_batched(A, None, m, n, C.c_void_p(F.data_ptr()),
                                        C.c_void_p(base), None, None, 0,
                                        C.c_void_p(ist.data_ptr()),
                                        C.c_void_p(lin.data_ptr()), None)
        assert ok == 0, (n, ok)
        offs = (8, 16, 24) if n % 4 == 0 else (8,)
        for off in offs:
            rc = dll.blsq_linearise_batched(A, None, m, n, C.c_void_p(F.data_ptr()),
                                            C.c_void_p(base + off), None, None, 0,
                                            C.c_void_p(ist.data_ptr()),
                                            C.c_void_p(lin.data_ptr()), None)
            assert rc == -1, (n, off, rc)
        dx = torch.ones((A, 2 * n), dtype=torch.float64, device=dev)
        for mode in (1, 2):
            ptrs = [F.data_ptr()] * (mode * n)
            ptrs[-1] = 0
            arr = (C.c_void_p * len(ptrs))(*ptrs)
            rc = dll.blsq_linearise_batched(A, None, m, n, C.c_void_p(F.data_ptr()), None,
                                            arr, C.c_void_p(dx.data_ptr()), mode,
                                            C.c_void_p(ist.data_ptr()),
                                            C.c_void_p(lin.data_ptr()), None)
            assert rc == -1, (n, mode, rc)
    torch.cuda.synchronize()


def check_host_inputs(lib, dev):
    """n = 12: host (pinned CPU) x0 and data through the streaming prologue
    give the bits of the device-input solve."""
    B, n, W = 50000, 12, 40
    mdl = RandModel(n, W, 64, np.full(64, W), seed=4)
    y = np.tile(mdl.y, (B // 64 + 1, 1))[:B].copy()
    At, Bt = T(mdl.A, dev), T(mdl.Bm, dev)

    def fun(X, Y):
        return X @ At.T + 0.3 * torch.sin(X @ Bt.T) - Y

    def jac(X, Y):
        return At[None] + 0.3 * torch.cos(X @ Bt.T)[:, :, None] * Bt[None]
    X0 = np.zeros((B, n))
    base = least_squares_batched(fun, T(X0, dev), jac=jac, bounds=(mdl.lb, mdl.ub),
                                 args=(PerProblem(T(y, dev)),))
    r = least_squares_batched(fun, torch.as_tensor(X0).pin_memory(), jac=jac,
                              bounds=(mdl.lb, mdl.ub),
                              args=(PerProblem(torch.as_tensor(y).pin_memory()),),
                              options=dict(h2d_chunks=3, prologue_rounds=4))
    same(r, base, "host inputs", fields=FIELDS[:-1])


# ------------------------------------------------------------------ tests --

CHECKS = [check_layouts, check_single_problem_routing, check_all_lin_instances, check_corpus,
          check_vs_oracle, check_coordinate_15, check_invariances, check_covariance]
CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/host_emul/emul_wide.cpp built into a temporary directory."""
    out = str(tmp_path_factory.mktemp("emul_wide") / "libblsq_hostemul_wide.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC",
                           "-ffp-contract=off", "-mfma", "-x", "c++", EMUL_WIDE, "-o", out])
    return hostemul.HostEmulLib(out)


@pytest.fixture(scope="module")
def cuda_lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bounded_lsq_b200 import get_lib
    return get_lib()


@pytest.mark.parametrize("check", CHECKS, ids=lambda c: c.__name__[6:])
def test_hostemul(emul, check):
    check(emul, CPU)


@pytest.mark.gpu
@pytest.mark.parametrize("check", CHECKS + [check_abi_errors, check_host_inputs],
                         ids=lambda c: c.__name__[6:])
def test_gpu(cuda_lib, check):
    dev = torch.device("cuda:0")
    if check is check_invariances:
        return check(cuda_lib, dev, graph=True)
    check(cuda_lib, dev)
