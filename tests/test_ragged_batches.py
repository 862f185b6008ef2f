"""Ragged batches: ``least_squares_batched(..., options={'rows': rows})``.

Every check takes ``lib`` and a torch device like the checks of cases.py: the
unmarked tests run them on the host emulation with the ragged entry points
(tests/host_emul/emul_rows.cpp), the ``gpu``-marked ones on the CUDA library.  Problem b of a ragged batch of
width W must be solved exactly as the dense problem made of its first
rows[b] residuals; the padding past rows[b] is never read (it holds NaN in
most checks below)."""
import os
import subprocess
import warnings

import numpy as np
import pytest
import torch

import cases
import hostemul
from cases import T, bits
from bounded_lsq_b200 import least_squares_batched, PerProblem

EMUL_ROWS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emul",
                         "emul_rows.cpp")
FIELDS = ("x", "obj_value", "status", "nfev", "njev", "active_mask", "x_covariance")


def same(r1, r2, label, fields=FIELDS, sel1=None, sel2=None):
    for f in fields:
        a, b = getattr(r1, f), getattr(r2, f)
        if a is None and b is None:
            continue
        a = a.cpu().numpy() if sel1 is None else a[sel1].cpu().numpy()
        b = b.cpu().numpy() if sel2 is None else b[sel2].cpu().numpy()
        assert bits(a, b), (label, f)


def quiet(fn, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return fn(*a, **k)


# ------------------------------------------------------ a random test model --

class RandModel:
    """f_b(x) = A x + 0.3 sin(Bm x) - y_b on the first rows[b] rows of a width-W
    design; y past rows[b] is NaN, so any read of the padding shows up."""

    def __init__(self, n, W, B, rows, seed, pad=float("nan")):
        rng = np.random.default_rng(seed)
        self.n, self.W, self.B = n, W, B
        self.A = rng.standard_normal((W, n))
        self.Bm = rng.standard_normal((W, n)) * 0.5
        xt = rng.uniform(-1, 1, (B, n))
        self.rows = np.asarray(rows, dtype=np.int64)
        y = xt @ self.A.T + 0.3 * np.sin(xt @ self.Bm.T) + 0.01 * rng.standard_normal((B, W))
        for b in range(B):
            y[b, self.rows[b]:] = pad
        self.y = y
        self.lb, self.ub = np.full(n, -0.6), np.full(n, 0.7)
        self.x0 = np.zeros(n)

    def torch_callbacks(self, dev, r=None):
        At, Bt = T(self.A[:r], dev), T(self.Bm[:r], dev)
        n = self.n

        def dot(X, M):
            # elementwise in a fixed order: a row's value does not depend on
            # how many rows there are (a matmul may block differently)
            acc = X[:, 0:1] * M[None, :, 0]
            for j in range(1, n):
                acc = acc + X[:, j:j + 1] * M[None, :, j]
            return acc

        def fun(X, Y):
            return dot(X, At) + 0.3 * torch.sin(dot(X, Bt)) - Y

        def jac(X, Y):
            return At[None] + 0.3 * torch.cos(dot(X, Bt))[:, :, None] * Bt[None]
        return fun, jac

    def solve(self, lib, dev, jac="exact", method="trf", sel=None, r=None, rows=True,
              scaling=1.0, **opts):
        """The ragged batch (r None) or the dense truncation to r rows."""
        sel = np.arange(self.B) if sel is None else np.asarray(sel)
        fun, jacf = self.torch_callbacks(dev, r)
        y = self.y[sel] if r is None else self.y[sel, :r]
        options = dict(opts)
        if r is None and rows:
            options["rows"] = torch.as_tensor(self.rows[sel])
        return quiet(least_squares_batched, fun, T(np.tile(self.x0, (len(sel), 1)), dev),
                     jac=jacf if jac == "exact" else jac,
                     bounds=(T(self.lb, dev), T(self.ub, dev)), method=method,
                     scaling=scaling, args=(PerProblem(T(y, dev)),), options=options,
                     _lib=lib)


# ------------------------------------------------------------------ checks --

def check_full_rows_is_dense(lib, dev):
    """rows = m for every problem gives the bits of the dense solve."""
    for name in ("c2_trf_exact", "c2_dogbox_exact", "c3_trf_2point", "c3_dogbox_2point",
                 "rat_trf_3point", "rat_dogbox_3point"):
        base, z, _ = cases.run_golden_batched(lib, dev, name, x_covariance=True)
        B, m = z["y"].shape
        rows = torch.full((B,), m, dtype=torch.int64)
        r, _, _ = cases.run_golden_batched(lib, dev, name, x_covariance=True, rows=rows)
        same(r, base, name)


def check_ragged_equals_truncated(lib, dev):
    """Problem b of a ragged batch == the dense solve of its first rows[b]
    residuals, bit for bit, when W and rows[b] share a lane-group class: n = 4,
    W = 64 (G = 8 for every count) and n = 4, W = 600 (MULTI for 260 .. 600)."""
    rng = np.random.default_rng(5)
    out = {}
    for W, lo, B, jac, method in ((64, 1, 40, "exact", "trf"), (64, 1, 40, "2-point", "dogbox"),
                                  (64, 1, 40, "3-point", "trf"),
                                  (600, 260, 10, "exact", "dogbox"),
                                  (600, 260, 10, "2-point", "trf")):
        rows = rng.integers(lo, W + 1, B)
        rows[0], rows[-1] = lo, W
        mdl = RandModel(4, W, B, rows, seed=W + B)
        rag = mdl.solve(lib, dev, jac, method, x_covariance=True)
        for r in np.unique(rows):
            sel = np.nonzero(rows == r)[0]
            # B = 1 raises for the reference's ValueError statuses: solve >= 2
            solo = np.concatenate([sel, sel]) if len(sel) == 1 else sel
            den = mdl.solve(lib, dev, jac, method, sel=solo, r=int(r), x_covariance=True)
            same(rag, den, (W, jac, method, int(r)), sel1=sel, sel2=slice(0, len(sel)))
        out[(W, jac, method)] = len(np.unique(rows))
    return out


def check_padding_never_read(lib, dev):
    """NaN instead of zeros in the padding of y (so of F, J and the perturbed
    F) changes no bit of any result field."""
    for jac, method in (("exact", "trf"), ("2-point", "dogbox"), ("3-point", "trf"),
                        ("exact", "dogbox")):
        rows = np.random.default_rng(3).integers(1, 49, 30)
        a = RandModel(3, 48, 30, rows, seed=9, pad=0.0).solve(lib, dev, jac, method,
                                                             x_covariance=True)
        b = RandModel(3, 48, 30, rows, seed=9).solve(lib, dev, jac, method, x_covariance=True)
        same(a, b, (jac, method))
        fa, fb = a.fun.cpu().numpy(), b.fun.cpu().numpy()
        assert bits(fa, fb) and not np.isnan(fb).any()


def check_vs_oracle(lib, dev, B=16, seed=42):
    """Random bounded problems for n = 1..8, both methods, scaling 1.0 and
    'jac', per-problem rows including 1, counts below n and the width W: each
    problem against the oracle on its truncated rows, with the gates of
    check_random_small_vs_oracle (rows >= n) and check_edge_cases_vs_oracle
    (rows < n: cost 1e-6, status -102 where the oracle raises)."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    tot = dict(full=0, full_exact=0, under=0, under_ok=0)
    for n in range(1, 9):
        for method in ("trf", "dogbox"):
            for scaling in (1.0, "jac"):
                W = int(rng.integers(n + 2, 3 * n + 8))
                rows = rng.integers(1, W + 1, B)
                rows[0], rows[1], rows[2] = 1, max(1, n - 1), W
                mdl = RandModel(n, W, B, rows, seed=int(rng.integers(1 << 30)))
                res = mdl.solve(lib, dev, "exact", method, scaling=scaling)
                X = res.x.cpu().numpy()
                assert np.all(X >= mdl.lb) and np.all(X <= mdl.ub)
                st, nf = res.status.cpu().numpy(), res.nfev.cpu().numpy()
                ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
                for b in range(B):
                    r = int(rows[b])
                    A, Bm, yb = mdl.A[:r], mdl.Bm[:r], mdl.y[b, :r]
                    try:
                        ref = orc.least_squares(
                            lambda x: A @ x + 0.3 * np.sin(Bm @ x) - yb, mdl.x0,
                            jac=lambda x: A + 0.3 * np.cos(Bm @ x)[:, None] * Bm,
                            bounds=(mdl.lb, mdl.ub), method=method, scaling=scaling)
                    except ValueError as e:
                        assert "not within the trust region" in str(e)
                        tot["under"] += 1
                        tot["under_ok"] += st[b] == -102
                        continue
                    if r >= n:
                        tot["full"] += 1
                        assert abs(ob[b] - ref.obj_value) <= 1e-8 * ref.obj_value + 1e-18, \
                            (n, method, scaling, b, r)
                        tot["full_exact"] += (
                            st[b] == ref.status and nf[b] == ref.nfev and
                            np.allclose(X[b], ref.x, rtol=1e-8, atol=1e-9) and
                            np.array_equal(mk[b], np.asarray(ref.active_mask)))
                    else:
                        tot["under"] += 1
                        if st[b] >= 0:
                            assert abs(ob[b] - ref.obj_value) <= \
                                1e-6 * ref.obj_value + 1e-18, (n, method, b, r)
                        tot["under_ok"] += (st[b] == ref.status and nf[b] == ref.nfev)
    assert tot["full_exact"] >= 0.99 * tot["full"], tot
    assert tot["under_ok"] >= 0.83 * tot["under"], tot
    return tot


def check_corpus_ragged(lib, dev):
    """The n <= 8 instances of the reference's corpus, grouped by (n, method,
    jac mode, scaling), each group solved as ONE ragged batch padded (with NaN)
    to its largest m: per-problem x0 and bounds, a per-instance callback
    dispatched through PerProblem(ids).  Same gates and measured waivers as
    check_corpus_single."""
    cs, z, probs = cases.corpus_cases(max_n=8)
    groups = {}
    for name, method, jm, sc in cs:
        groups.setdefault((probs[name].n, method, jm, sc), []).append(name)
    stats = dict(total=0, exact_status=0, waived=0, fd_total=0, fd_exact=0, batches=0)
    for (n, method, jm, sc), names in sorted(groups.items()):
        ps = [probs[nm] for nm in names]
        ms = [len(p.fun(p.x0)) for p in ps]
        W, B = max(ms), len(ps)

        def evaluate(X, ids, what):
            out = np.full((X.shape[0], W) + ((n,) if what == "jac" else ()), np.nan)
            Xh = X.cpu().numpy()
            for a, i in enumerate(ids.cpu().numpy()):
                p = ps[int(i)]
                v = np.asarray(p.fun(Xh[a]) if what == "fun" else p.jac(Xh[a]), dtype=float)
                out[a, :len(v)] = v.reshape(len(v), -1)[:, 0] if what == "fun" else v
            return T(out, dev)

        trials = []

        def trace(r, idx, Xn, state, istate):
            if not trials:
                trials.append(Xn.cpu().numpy().copy())
        ids = T(np.arange(B), dev, torch.int64)
        res = least_squares_batched(
            lambda X, i: evaluate(X, i, "fun"),
            T(np.stack([p.x0 for p in ps]), dev),
            jac=(lambda X, i: evaluate(X, i, "jac")) if jm == "exact" else jm,
            bounds=(T(np.stack([p.lb for p in ps]), dev), T(np.stack([p.ub for p in ps]), dev)),
            method=method, scaling='jac' if sc == 'jac' else 1.0, args=(PerProblem(ids),),
            options=dict(rows=torch.as_tensor(ms), graph_tail_rounds=0, trace=trace),
            _lib=lib)
        stats["batches"] += 1
        for b, (name, p) in enumerate(zip(names, ps)):
            key = f"{name}|{method}|{jm}|{sc}|"
            obj, status, nfev, njev, opt, ntr = z[key + "scalars"]
            x = res.x[b].cpu().numpy()
            st, nf, nj = int(res.status[b]), int(res.nfev[b]), int(res.njev[b])
            ob = float(res.obj_value[b])
            stats["total"] += 1
            assert np.all(x >= p.lb) and np.all(x <= p.ub), key
            assert st >= 0, key
            gt = z[key + "trials"]
            if trials and not np.isnan(gt[0]).any() and \
                    not cases.first_step_sensitive(z, name, method, sc):
                stepn = max(np.abs(gt[0] - p.x0).max(), 1e-300)
                e0 = float(np.abs(trials[0][b] - gt[0]).max() / stepn)
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
            assert bits(res.active_mask[b].cpu().numpy(), z[key + "mask"]), key
            gx = z[key + "x"]
            assert np.allclose(x, gx, rtol=1e-8, atol=1e-8 * np.abs(gx).max()), (key, x, gx)
            assert abs(ob - obj) <= 1e-8 * obj + 1e-18, key
            stats["exact_status"] += 1
    assert stats["fd_exact"] >= 0.93 * stats["fd_total"], stats
    return stats


def check_invariance(lib, dev, graph=False):
    """With rows set: permuting the problems, solving a subset at the same
    width, chunk, the compaction thresholds and (graph) the CUDA-graph tail
    give the same bits per problem."""
    rng = np.random.default_rng(17)
    B, W = 300, 40
    rows = rng.integers(1, W + 1, B)
    for jac, method in (("exact", "trf"), ("2-point", "dogbox")):
        mdl = RandModel(5, W, B, rows, seed=23)
        base = mdl.solve(lib, dev, jac, method, graph_tail_rounds=0, compact_below=0.0)
        perm = rng.permutation(B)
        same(mdl.solve(lib, dev, jac, method, sel=perm), base, "perm", sel2=perm)
        sub = np.sort(rng.choice(B, 77, replace=False))
        same(mdl.solve(lib, dev, jac, method, sel=sub), base, "subset", sel2=sub)
        same(mdl.solve(lib, dev, jac, method, chunk=64), base, "chunk")
        for opts in (dict(compact_below=1.0), dict(check_every=3, compact_below=0.5)):
            same(mdl.solve(lib, dev, jac, method, graph_tail_rounds=0, **opts), base, opts)
        if graph:
            for opts in (dict(), dict(graph_tail_rounds=3, tail_below=200)):
                same(mdl.solve(lib, dev, jac, method, **opts), base, ("graph", opts))


def check_api_errors(lib, dev):
    """ValueError for a bad `rows`; res.fun is zero past rows[b] and its
    squared norm is obj_value."""
    mdl = RandModel(2, 10, 6, [1, 2, 3, 10, 7, 5], seed=1)

    def bad(rows, match, fun=None):
        f, j = mdl.torch_callbacks(dev)
        if fun is not None:
            f = fun
        with pytest.raises(ValueError, match=match):
            least_squares_batched(f, T(np.zeros((6, 2)), dev), jac=j,
                                  args=(PerProblem(T(mdl.y, dev)),),
                                  options=dict(rows=rows), _lib=lib)
    bad(torch.ones(5, dtype=torch.int64), "shape")
    bad(torch.ones((6, 1), dtype=torch.int64), "shape")
    bad(torch.ones(6, dtype=torch.float64), "integer")
    bad(torch.ones(6, dtype=torch.bool), "integer")
    bad(torch.tensor([1, 2, 0, 4, 5, 6]), "at least 1")
    bad(torch.tensor([1, 2, 3, 11, 5, 6]), "exceeds")
    f, _ = mdl.torch_callbacks(dev)

    def inlined(X, Y):
        return f(X, Y)
    inlined.blsq_linearise = lambda *a: None
    bad(torch.ones(6, dtype=torch.int64), "compiled into", fun=inlined)
    res = mdl.solve(lib, dev)
    F = res.fun.cpu().numpy()
    for b in range(6):
        assert np.all(F[b, mdl.rows[b]:] == 0.0) and not np.isnan(F[b]).any()
        # obj_value is f.f (the reference's obj_value, twice its cost)
        assert abs(float(F[b] @ F[b]) - float(res.obj_value[b])) <= \
            1e-12 * float(res.obj_value[b]) + 1e-300


# ------------------------------------------------------- GPU-only checks --

def check_fused_model_rows(dev):
    """models.callbacks('ExpDecay2', rows=True) (fused, writes only r < rows[b])
    against the torch ExpDecay2 callbacks on NaN-padded data, bit for bit."""
    from bounded_lsq_b200 import models
    from bounded_lsq_b200.synthetic import ExpDecay2
    model = ExpDecay2()
    B = 4096
    _, y = model.make_data(B, seed=31)
    rows = np.random.default_rng(2).integers(24, model.m + 1, B)
    for b in range(B):
        y[b, rows[b]:] = np.nan
    yt, rt = T(y, dev), T(rows, dev, torch.int32)
    X0 = T(np.tile(model.x0, (B, 1)), dev)
    for jk, method in (("exact", "trf"), ("2-point", "dogbox")):
        fun, jac = models.callbacks("ExpDecay2", jk, rows=True)
        r1 = least_squares_batched(fun, X0, jac=jac, bounds=(model.lb, model.ub),
                                   method=method, args=(PerProblem(yt), PerProblem(rt)),
                                   options=dict(rows=rt, x_covariance=True))
        r2 = least_squares_batched(model.fun_t, X0,
                                   jac=model.jac_t if jk == "exact" else jk,
                                   bounds=(model.lb, model.ub), method=method,
                                   args=(PerProblem(yt),),
                                   options=dict(rows=rt, x_covariance=True))
        same(r1, r2, ("fused", jk, method))
        assert bits(r1.fun.cpu().numpy(), r2.fun.cpu().numpy())


def check_host_inputs_rows(dev):
    """Host (pinned CPU) x0, data and rows through the streaming prologue:
    same bits as the device-input solve."""
    from bounded_lsq_b200 import models
    from bounded_lsq_b200.synthetic import ExpDecay2
    model = ExpDecay2()
    B = 140000
    _, y = model.make_data(4096, seed=5)
    y = np.tile(y, (-(-B // 4096), 1))[:B].copy()
    rows = np.random.default_rng(8).integers(24, model.m + 1, B)
    X0 = np.tile(model.x0, (B, 1))
    fun, jac = models.callbacks("ExpDecay2", rows=True)
    yt, rt = T(y, dev), T(rows, dev, torch.int32)
    base = least_squares_batched(fun, T(X0, dev), jac=jac, bounds=(model.lb, model.ub),
                                 args=(PerProblem(yt), PerProblem(rt)), options=dict(rows=rt))
    yh = torch.as_tensor(y).pin_memory()
    rh = torch.as_tensor(rows, dtype=torch.int32).pin_memory()
    r = least_squares_batched(fun, torch.as_tensor(X0).pin_memory(), jac=jac,
                              bounds=(model.lb, model.ub),
                              args=(PerProblem(yh), PerProblem(rh)),
                              options=dict(rows=rh, h2d_chunks=2, prologue_rounds=4))
    same(r, base, "host inputs", fields=FIELDS[:-1])
    r = least_squares_batched(fun, torch.as_tensor(X0).pin_memory(), jac=jac,
                              bounds=(model.lb, model.ub),
                              args=(PerProblem(yh), PerProblem(rh)),
                              options=dict(rows=rh, h2d_chunks=2, chunk=70000))
    same(r, base, "host inputs + chunk", fields=FIELDS[:-1])


# ------------------------------------------------------------------ tests --

CHECKS = [check_full_rows_is_dense, check_ragged_equals_truncated, check_padding_never_read,
          check_vs_oracle, check_corpus_ragged, check_invariance, check_api_errors]
CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/host_emul/emul_rows.cpp (the host emulation plus the ragged entry
    points), built into a temporary directory."""
    out = str(tmp_path_factory.mktemp("emul_rows") / "libblsq_hostemul_rows.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC",
                           "-ffp-contract=off", "-mfma", "-x", "c++", EMUL_ROWS, "-o", out])
    return hostemul.HostEmulLib(out)


@pytest.fixture(scope="module")
def cuda_lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bounded_lsq_b200 import get_lib
    return get_lib()


@pytest.mark.parametrize("check", CHECKS, ids=lambda c: c.__name__[6:])
def test_hostemul(emul, check):
    print(check(emul, CPU))


@pytest.mark.gpu
@pytest.mark.parametrize("check", CHECKS, ids=lambda c: c.__name__[6:])
def test_gpu(cuda_lib, check):
    dev = torch.device("cuda:0")
    if check is check_invariance:
        print(check(cuda_lib, dev, graph=True))
    else:
        print(check(cuda_lib, dev))


@pytest.mark.gpu
def test_gpu_fused_model_rows(cuda_lib):
    check_fused_model_rows(torch.device("cuda:0"))


@pytest.mark.gpu
def test_gpu_host_inputs_rows(cuda_lib):
    check_host_inputs_rows(torch.device("cuda:0"))
