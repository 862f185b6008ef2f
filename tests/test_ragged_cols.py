"""Ragged parameter counts: ``least_squares_batched(..., options={'cols': cols})``.

Every check takes ``lib`` and a torch device like the checks of
test_ragged_batches.py: the unmarked tests run them on the host emulation with
the ragged-parameter entry points (tests/host_emul/emul_cols.cpp), the
``gpu``-marked ones on the CUDA library.  Problem b of a batch of width n must
be solved exactly as the dense problem made of its first cols[b] parameters,
with the others held at x0[b]: the batch runs one dense solve per distinct
count, so the comparisons below are bit for bit.  The padded Jacobian columns
hold NaN in most checks."""
import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import cases
import hostemul
from cases import T, bits
from test_ragged_batches import FIELDS, same, quiet
from bounded_lsq_b200 import least_squares_batched, PerProblem

EMUL_COLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emul",
                         "emul_cols.cpp")


# ------------------------------------------------------ a random test model --

class ColModel:
    """f_b(x) = A x + 0.3 sin(Bm x) - y_b over all n coordinates of x; problem
    b fits its first cols[b] and holds the others at x0[b] (nonzero, so they
    enter every residual).  With `rows`, y past rows[b] is NaN.  The Jacobian
    callback writes `jpad` (NaN) into the columns past cols[b]."""

    def __init__(self, n, W, B, cols, seed, rows=None, per_bounds=False):
        rng = np.random.default_rng(seed)
        self.n, self.W, self.B = n, W, B
        self.A = rng.standard_normal((W, n))
        self.Bm = rng.standard_normal((W, n)) * 0.5
        xt = rng.uniform(-1, 1, (B, n))
        self.x0 = rng.uniform(-0.2, 0.2, (B, n))
        self.cols = np.asarray(cols, dtype=np.int64)
        self.rows = None if rows is None else np.asarray(rows, dtype=np.int64)
        y = xt @ self.A.T + 0.3 * np.sin(xt @ self.Bm.T) + 0.01 * rng.standard_normal((B, W))
        if self.rows is not None:
            for b in range(B):
                y[b, self.rows[b]:] = np.nan
        self.y = y
        self.lb, self.ub = np.full(n, -0.6), np.full(n, 0.7)
        if per_bounds:
            self.lb = self.lb - rng.uniform(0, 0.4, (B, n))
            self.ub = self.ub + rng.uniform(0, 0.4, (B, n))

    def callbacks(self, dev, jpad=float("nan")):
        At, Bt = T(self.A, dev), T(self.Bm, dev)
        n = self.n

        def dot(X, M):
            # elementwise in a fixed order: a row's value does not depend on
            # how many rows there are (a matmul may block differently)
            acc = X[:, 0:1] * M[None, :, 0]
            for j in range(1, n):
                acc = acc + X[:, j:j + 1] * M[None, :, j]
            return acc

        def fun(X, Y, C=None):
            return dot(X, At) + 0.3 * torch.sin(dot(X, Bt)) - Y

        def jac(X, Y, C=None):
            J = At[None] + 0.3 * torch.cos(dot(X, Bt))[:, :, None] * Bt[None]
            if C is not None:
                pad = torch.arange(n, device=J.device)[None, None, :] >= C[:, None, None]
                J = J.masked_fill(pad, jpad)
            return J
        return fun, jac

    def solve(self, lib, dev, jac="exact", method="trf", sel=None, N=None, scaling=1.0,
              jpad=float("nan"), bounds=None, **opts):
        """The ragged batch (N None) or the dense solve of its first N
        parameters with the others fixed at x0."""
        sel = np.arange(self.B) if sel is None else np.asarray(sel)
        fun, jacf = self.callbacks(dev, jpad)
        lb, ub = bounds if bounds is not None else (self.lb, self.ub)
        lb = lb if lb.ndim == 1 else lb[sel]
        ub = ub if ub.ndim == 1 else ub[sel]
        y = PerProblem(T(self.y[sel], dev))
        options = dict(opts)
        if self.rows is not None:
            options["rows"] = torch.as_tensor(self.rows[sel])
        sc = T(scaling, dev) if isinstance(scaling, np.ndarray) else scaling
        if N is None:
            options["cols"] = torch.as_tensor(self.cols[sel])
            args = (y, PerProblem(T(self.cols[sel], dev, torch.int64)))
            f, j, x0 = fun, jacf, self.x0[sel]
        else:
            args = (y, PerProblem(T(self.x0[sel, N:], dev)))

            def f(X, Y, P):
                return fun(torch.cat([X, P], 1), Y)

            def j(X, Y, P):
                return jacf(torch.cat([X, P], 1), Y)[:, :, :N]
            x0, lb, ub = self.x0[sel, :N], lb[..., :N], ub[..., :N]
            if isinstance(scaling, np.ndarray):
                sc = T(scaling[:N], dev)
        return quiet(least_squares_batched, f, T(x0, dev), jac=j if jac == "exact" else jac,
                     bounds=(T(lb, dev), T(ub, dev)), method=method, scaling=sc, args=args,
                     options=options, _lib=lib)


def part(res, sel, N):
    """The fields of problems `sel` on their first N coordinates."""
    cov = res.x_covariance
    return SimpleNamespace(
        x=res.x[sel, :N], obj_value=res.obj_value[sel], status=res.status[sel],
        nfev=res.nfev[sel], njev=res.njev[sel], active_mask=res.active_mask[sel, :N],
        x_covariance=None if cov is None else cov[sel, :N, :N])


def check_reduced(mdl, rag, lib, dev, jac, method, label, **kw):
    """Every cols group of `rag` against the dense solve of its first N
    parameters, bit for bit; the padded coordinates of x are x0, those of
    active_mask and x_covariance are 0."""
    x0 = mdl.x0
    for N in np.unique(mdl.cols):
        sel = np.nonzero(mdl.cols == N)[0]
        # B = 1 raises for the reference's ValueError statuses: solve >= 2
        solo = np.concatenate([sel, sel]) if len(sel) == 1 else sel
        den = mdl.solve(lib, dev, jac, method, sel=solo, N=int(N), **kw)
        same(part(rag, sel, N), part(den, slice(0, len(sel)), N), (label, int(N)))
        assert bits(rag.x[sel, N:].cpu().numpy(), x0[sel, N:]), (label, int(N))
        assert not rag.active_mask[sel, N:].any(), (label, int(N))
        if rag.x_covariance is not None:
            cv = rag.x_covariance[sel].cpu().numpy()
            assert not cv[:, N:, :].any() and not cv[:, :, N:].any(), (label, int(N))
    return len(np.unique(mdl.cols))


def mixed_cols(rng, n, B):
    cols = rng.integers(1, n + 1, B)
    cols[0], cols[-1] = 1, n
    return cols


# ------------------------------------------------------------------ checks --

def check_full_cols_is_dense(lib, dev):
    """cols = n for every problem gives the bits of the solve without cols."""
    for name in ("c2_trf_exact", "c2_dogbox_exact", "c3_trf_2point", "c3_dogbox_2point",
                 "rat_trf_3point", "rat_dogbox_3point"):
        base, z, _ = cases.run_golden_batched(lib, dev, name, x_covariance=True)
        B, n = base.x.shape
        cols = torch.full((B,), n, dtype=torch.int64)
        r, _, _ = cases.run_golden_batched(lib, dev, name, x_covariance=True, cols=cols)
        same(r, base, name)


def check_ragged_equals_reduced(lib, dev):
    """Problem b of a batch of mixed cols == the dense solve of its first
    cols[b] parameters, bit for bit: TRF and dogbox, analytic / 2-point /
    3-point Jacobians, scaling 1.0, (n,) and 'jac', shared and per-problem
    bounds, x_covariance, with and without ragged rows; n up to 16, cols
    down to 1."""
    rng = np.random.default_rng(11)
    groups = {}
    for n, W, B, jac, method, sc, per_b, ragged in (
            (6, 30, 40, "exact", "trf", 1.0, False, False),
            (6, 30, 40, "2-point", "dogbox", "jac", True, True),
            (6, 30, 40, "3-point", "trf", "vec", True, False),
            (8, 24, 40, "exact", "dogbox", "vec", True, True),
            (8, 200, 24, "exact", "trf", "jac", False, False),
            (12, 40, 30, "2-point", "trf", 1.0, False, True),
            (16, 40, 36, "exact", "dogbox", "vec", False, True),
            (16, 48, 36, "exact", "trf", "jac", True, False),
            (16, 20, 24, "3-point", "dogbox", 1.0, True, False)):
        cols = mixed_cols(rng, n, B)
        rows = None
        if ragged:
            rows = rng.integers(max(1, W // 3), W + 1, B)
            rows[1] = W
        mdl = ColModel(n, W, B, cols, seed=n * 100 + W, rows=rows, per_bounds=per_b)
        scaling = rng.uniform(0.5, 2.0, n) if sc == "vec" else sc
        rag = mdl.solve(lib, dev, jac, method, scaling=scaling, x_covariance=True)
        label = (n, W, jac, method, sc, per_b, ragged)
        groups[label] = check_reduced(mdl, rag, lib, dev, jac, method, label, scaling=scaling,
                                      x_covariance=True)
    return groups


def check_padding_never_read(lib, dev):
    """NaN instead of zeros in the padded Jacobian columns, and bounds with
    lb >= ub and an infeasible x0 in the padded coordinates, change no bit of
    any result field; the padded coordinates of res.x are x0."""
    rng = np.random.default_rng(3)
    n, B = 7, 30
    cols = mixed_cols(rng, n, B)
    for jac, method in (("exact", "trf"), ("exact", "dogbox"), ("2-point", "dogbox"),
                        ("3-point", "trf")):
        mdl = ColModel(n, 25, B, cols, seed=9, per_bounds=True)
        a = mdl.solve(lib, dev, jac, method, jpad=0.0, x_covariance=True)
        b = mdl.solve(lib, dev, jac, method, x_covariance=True)
        same(a, b, (jac, method, "NaN J"))
        lb, ub = mdl.lb.copy(), mdl.ub.copy()
        for i in range(B):
            lb[i, cols[i]:], ub[i, cols[i]:] = 1.0, -1.0       # x0 in between is ~0
        c = mdl.solve(lib, dev, jac, method, bounds=(lb, ub), x_covariance=True)
        same(c, b, (jac, method, "bounds"))
        x = b.x.cpu().numpy()
        for i in range(B):
            assert bits(x[i, cols[i]:], mdl.x0[i, cols[i]:])
        assert not np.isnan(b.fun.cpu().numpy()).any()


def check_vs_oracle(lib, dev, B=12, seed=42):
    """Random bounded problems with mixed cols for n = 3, 8, 11, 16, both
    methods, scaling 1.0 and 'jac', rows below cols[b] included: each problem
    against the oracle on its reduced problem (first rows[b] residuals, first
    cols[b] parameters, the others fixed at x0), with the gates of
    test_ragged_batches.check_vs_oracle (rows >= cols: cost 1e-8, status,
    nfev, x and the active set for >= 99 %; rows < cols: cost 1e-6, status
    -102 where the oracle raises, status and nfev for >= 83 %)."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    tot = dict(full=0, full_exact=0, under=0, under_ok=0)
    for n in (3, 8, 11, 16):
        for method in ("trf", "dogbox"):
            for scaling in (1.0, "jac"):
                W = int(rng.integers(n + 2, 3 * n + 8))
                cols = mixed_cols(rng, n, B)
                rows = rng.integers(1, W + 1, B)
                rows[0], rows[1], rows[2] = W, 1, max(1, cols[2] - 1)
                mdl = ColModel(n, W, B, cols, seed=int(rng.integers(1 << 30)), rows=rows)
                res = mdl.solve(lib, dev, "exact", method, scaling=scaling)
                X = res.x.cpu().numpy()
                assert np.all(X >= mdl.lb) and np.all(X <= mdl.ub)
                st, nf = res.status.cpu().numpy(), res.nfev.cpu().numpy()
                ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
                for b in range(B):
                    r, N = int(rows[b]), int(cols[b])
                    A, Bm, yb, xp = mdl.A[:r], mdl.Bm[:r], mdl.y[b, :r], mdl.x0[b, N:]

                    def fun(x, A=A, Bm=Bm, yb=yb, xp=xp):
                        xf = np.concatenate([x, xp])
                        return A @ xf + 0.3 * np.sin(Bm @ xf) - yb

                    def jac(x, A=A, Bm=Bm, xp=xp, N=N):
                        xf = np.concatenate([x, xp])
                        return (A + 0.3 * np.cos(Bm @ xf)[:, None] * Bm)[:, :N]
                    try:
                        ref = quiet(orc.least_squares, fun, mdl.x0[b, :N], jac=jac,
                                    bounds=(mdl.lb[:N], mdl.ub[:N]), method=method,
                                    scaling=scaling)
                    except ValueError as e:
                        assert "not within the trust region" in str(e)
                        tot["under"] += 1
                        tot["under_ok"] += st[b] == -102
                        continue
                    if r >= N:
                        tot["full"] += 1
                        assert abs(ob[b] - ref.obj_value) <= 1e-8 * ref.obj_value + 1e-18, \
                            (n, method, scaling, b, r, N)
                        tot["full_exact"] += (
                            st[b] == ref.status and nf[b] == ref.nfev and
                            np.allclose(X[b, :N], ref.x, rtol=1e-8, atol=1e-9) and
                            np.array_equal(mk[b, :N], np.asarray(ref.active_mask)))
                    else:
                        tot["under"] += 1
                        if st[b] >= 0:
                            assert abs(ob[b] - ref.obj_value) <= \
                                1e-6 * ref.obj_value + 1e-18, (n, method, b, r, N)
                        tot["under_ok"] += (st[b] == ref.status and nf[b] == ref.nfev)
    assert tot["full_exact"] >= 0.99 * tot["full"], tot
    assert tot["under"] > 0 and tot["under_ok"] >= 0.83 * tot["under"], tot
    return tot


def check_corpus_ragged_cols(lib, dev):
    """Every instance of the reference's corpus with n <= 16, grouped by
    (method, jac mode, scaling) only: each group is ONE batch padded to its
    largest n (cols) and its largest m (rows), NaN in the padded Jacobian
    columns and residuals, NaN bounds in the padded coordinates.  The gates
    and measured waivers of test_ragged_batches.check_corpus_ragged (status
    and nfev of the finite-difference runs: 139 of 146 on the host
    emulation, gate 0.93)."""
    cs, z, probs = cases.corpus_cases(max_n=16)
    groups = {}
    for name, method, jm, sc in cs:
        groups.setdefault((method, jm, sc), []).append(name)
    stats = dict(total=0, exact_status=0, waived=0, fd_total=0, fd_exact=0, batches=0,
                 widths=0)
    for (method, jm, sc), names in sorted(groups.items()):
        ps = [probs[nm] for nm in names]
        ns = [p.n for p in ps]
        ms = [len(p.fun(p.x0)) for p in ps]
        n, W, B = max(ns), max(ms), len(ps)

        def evaluate(X, ids, what):
            out = np.full((X.shape[0], W) + ((n,) if what == "jac" else ()), np.nan)
            Xh = X.cpu().numpy()
            for a, i in enumerate(ids.cpu().numpy()):
                p = ps[int(i)]
                x = Xh[a, :p.n]
                v = np.asarray(p.fun(x) if what == "fun" else p.jac(x), dtype=float)
                if what == "fun":
                    out[a, :len(v)] = v
                else:
                    out[a, :v.shape[0], :p.n] = v.reshape(v.shape[0], -1)
            return T(out, dev)

        def padded(v):
            return np.stack([np.concatenate([getattr(p, v), np.full(n - p.n, np.nan)])
                             for p in ps])
        first = {}

        def trace(r, idx, Xn, state, istate):
            if not first:
                first.update(zip(idx.cpu().numpy().tolist(), Xn.cpu().numpy()))
        x0 = np.stack([np.concatenate([p.x0, np.zeros(n - p.n)]) for p in ps])
        ids = T(np.arange(B), dev, torch.int64)
        res = least_squares_batched(
            lambda X, i: evaluate(X, i, "fun"), T(x0, dev),
            jac=(lambda X, i: evaluate(X, i, "jac")) if jm == "exact" else jm,
            bounds=(T(padded("lb"), dev), T(padded("ub"), dev)),
            method=method, scaling='jac' if sc == 'jac' else 1.0, args=(PerProblem(ids),),
            options=dict(rows=torch.as_tensor(ms), cols=torch.as_tensor(ns),
                         graph_tail_rounds=0, trace=trace), _lib=lib)
        stats["batches"] += 1
        stats["widths"] = max(stats["widths"], len(set(ns)))
        for b, (name, p) in enumerate(zip(names, ps)):
            key = f"{name}|{method}|{jm}|{sc}|"
            obj, status, nfev, njev, opt, ntr = z[key + "scalars"]
            x = res.x[b].cpu().numpy()
            assert bits(x[p.n:], x0[b, p.n:]), key
            x = x[:p.n]
            st, nf, nj = int(res.status[b]), int(res.nfev[b]), int(res.njev[b])
            ob = float(res.obj_value[b])
            stats["total"] += 1
            assert np.all(x >= p.lb) and np.all(x <= p.ub), key
            assert st >= 0, key
            gt = z[key + "trials"]
            if b in first and not np.isnan(gt[0]).any() and \
                    not cases.first_step_sensitive(z, name, method, sc):
                stepn = max(np.abs(gt[0] - p.x0).max(), 1e-300)
                e0 = float(np.abs(first[b][:p.n] - gt[0]).max() / stepn)
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
            assert bits(res.active_mask[b, :p.n].cpu().numpy(), z[key + "mask"]), key
            gx = z[key + "x"]
            assert np.allclose(x, gx, rtol=1e-8, atol=1e-8 * np.abs(gx).max()), (key, x, gx)
            assert abs(ob - obj) <= 1e-8 * obj + 1e-18, key
            stats["exact_status"] += 1
    assert stats["widths"] > 1, stats
    assert stats["fd_exact"] >= 0.93 * stats["fd_total"], stats
    return stats


def check_invariance(lib, dev, graph=False):
    """With cols (and rows) set: permuting the problems, solving a subset,
    chunk, the compaction thresholds and (graph) the CUDA-graph tail give the
    same bits per problem."""
    rng = np.random.default_rng(17)
    B, W, n = 300, 30, 8
    cols = mixed_cols(rng, n, B)
    rows = rng.integers(n, W + 1, B)
    for jac, method in (("exact", "trf"), ("2-point", "dogbox")):
        mdl = ColModel(n, W, B, cols, seed=23, rows=rows, per_bounds=True)
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
    """ValueError for a bad `cols` and for `cols` with an inlined model; the
    bound, feasibility and scaling checks still apply to the first cols[b]
    coordinates."""
    cols = [1, 2, 3, 3, 2, 1]
    mdl = ColModel(3, 10, 6, cols, seed=1)
    f, j = mdl.callbacks(dev)

    def run(cols, fun=f, x0=None, bounds=None, scaling=1.0):
        lb, ub = bounds if bounds is not None else (mdl.lb, mdl.ub)
        return quiet(least_squares_batched, fun, T(mdl.x0 if x0 is None else x0, dev), jac=j,
                     bounds=(T(lb, dev), T(ub, dev)), scaling=scaling,
                     args=(PerProblem(T(mdl.y, dev)),), options=dict(cols=cols), _lib=lib)

    def bad(match, cols=cols, **kw):
        with pytest.raises(ValueError, match=match):
            run(cols, **kw)
    bad("shape", cols=torch.ones(5, dtype=torch.int64))
    bad("shape", cols=torch.ones((6, 1), dtype=torch.int64))
    bad("integer", cols=torch.ones(6, dtype=torch.float64))
    bad("integer", cols=torch.ones(6, dtype=torch.bool))
    bad("at least 1", cols=torch.tensor([1, 2, 0, 3, 2, 1]))
    bad("exceeds", cols=torch.tensor([1, 2, 4, 3, 2, 1]))

    def inlined(X, Y):
        return f(X, Y)
    inlined.blsq_linearise = lambda *a: None
    bad("compiled into", fun=inlined)
    # a used coordinate is still checked, a padded one is not
    x0 = mdl.x0.copy()
    x0[1, 1] = 5.0
    bad("infeasible", x0=x0)
    x0 = mdl.x0.copy()
    x0[1, 2] = 5.0
    run(cols, x0=x0)
    lb, ub = np.tile(mdl.lb, (6, 1)), np.tile(mdl.ub, (6, 1))
    lb[2, 2] = ub[2, 2] = 0.0
    bad("strictly less", bounds=(lb, ub))
    lb[2, 2], ub[2, 2] = -0.6, 0.7
    lb[0, 1], ub[0, 1] = 1.0, -1.0
    run(cols, bounds=(lb, ub))
    bad("positive", scaling=T(np.array([1.0, 1.0, -1.0]), dev))
    run([1, 2, 2, 2, 2, 1], scaling=T(np.array([1.0, 1.0, -1.0]), dev))


def check_lin_ld_instances(lib, dev):
    """blsq_linearise_batched_ld at every N = 1..16, lane-group classes from
    m = 3 to MULTI, row strides ldj with every vector width, with and without
    rows: the records equal those of blsq_linearise_batched_rows on the
    contiguous first N columns, bit for bit, with NaN in the padded columns.
    ldj < n and (ldj == n) behave as documented."""
    dll = lib._dll
    rng = np.random.default_rng(5)
    A = 37
    for N in range(1, 17):
        LS = lib.lin_record_size(N)
        for ldj in sorted({N, N + 1, N + 2, 2 * N, 16, 17} - set(range(N))):
            for m in (3, 40, 150, 600):
                for ragged in (False, True):
                    J = rng.standard_normal((A, m, ldj))
                    J[:, :, N:] = np.nan
                    F = rng.standard_normal((A, m))
                    rows = rng.integers(1, m + 1, A).astype(np.int32) if ragged else None
                    ist = np.full((A, 8), -1, np.int32)
                    ist[::3, 0] = 0                           # stopped: skipped
                    Jt, Ft, It = T(J, dev), T(F, dev), T(ist, dev, torch.int32)
                    Jc = T(np.ascontiguousarray(J[:, :, :N]), dev)
                    Rt = None if rows is None else T(rows, dev, torch.int32)
                    rp = None if Rt is None else C.c_void_p(Rt.data_ptr())
                    out = []
                    for fn, Jp, extra in (("blsq_linearise_batched_ld", Jt, (N, ldj)),
                                          ("blsq_linearise_batched_rows", Jc, (N,))):
                        lin = torch.full((A, LS), 7.0, dtype=torch.float64, device=dev)
                        lib.call(fn, A, None, m, *extra, Ft.data_ptr(), Jp.data_ptr(), None,
                                 None, 0, It.data_ptr(), lin.data_ptr(), rp, lib.stream(Ft))
                        out.append(lin.cpu().numpy())
                    assert bits(out[0], out[1]), (N, ldj, m, ragged)
        lin = torch.zeros((A, LS), dtype=torch.float64, device=dev)
        F = torch.zeros((A, 4), dtype=torch.float64, device=dev)
        ist = torch.full((A, 8), -1, dtype=torch.int32, device=dev)
        if N > 1:
            rc = dll.blsq_linearise_batched_ld(
                A, None, 4, N, N - 1, C.c_void_p(F.data_ptr()), C.c_void_p(F.data_ptr()),
                None, None, 0, C.c_void_p(ist.data_ptr()), C.c_void_p(lin.data_ptr()), None,
                None)
            assert rc == -1, (N, rc)
    if dev.type == "cuda":
        torch.cuda.synchronize()


# ------------------------------------------------------- GPU-only checks --

def check_ld_alignment(lib, dev):
    """A J misaligned for the vector width of (n, ldj) returns BLSQ_E_BADARG
    before any launch; the widths follow from both n and ldj.  A solve whose
    jac returns a misaligned view gives the bits of the aligned solve."""
    dll = lib._dll
    m, A = 8, 4
    for n, ldj, width in ((4, 8, 4), (4, 6, 2), (8, 12, 4), (8, 10, 2), (2, 6, 2),
                          (2, 5, 1), (3, 8, 1), (12, 16, 4), (6, 16, 2), (16, 16, 4)):
        buf = torch.zeros(A * m * ldj + 8, dtype=torch.float64, device=dev)
        F = torch.zeros((A, m), dtype=torch.float64, device=dev)
        ist = torch.full((A, 8), -1, dtype=torch.int32, device=dev)
        lin = torch.zeros((A, lib.lin_record_size(n)), dtype=torch.float64, device=dev)
        base = buf.data_ptr()
        assert base % 256 == 0
        for off in (0, 8, 16, 24):
            rc = dll.blsq_linearise_batched_ld(A, None, m, n, ldj, C.c_void_p(F.data_ptr()),
                                               C.c_void_p(base + off), None, None, 0,
                                               C.c_void_p(ist.data_ptr()),
                                               C.c_void_p(lin.data_ptr()), None, None)
            assert rc == (0 if off % (8 * width) == 0 else -1), (n, ldj, off, rc)
    torch.cuda.synchronize()
    rng = np.random.default_rng(4)
    n, B, W = 8, 64, 20
    mdl = ColModel(n, W, B, mixed_cols(rng, n, B), seed=6)
    base = mdl.solve(lib, dev, x_covariance=True)
    fun, jac = mdl.callbacks(dev)

    def jac_view(X, Y, Cc):
        J = jac(X, Y, Cc)
        buf = torch.empty(J.numel() + 1, dtype=J.dtype, device=J.device)
        v = buf[1:].view(J.shape)
        v.copy_(J)
        return v
    r = quiet(least_squares_batched, fun, T(mdl.x0, dev), jac=jac_view,
              bounds=(T(mdl.lb, dev), T(mdl.ub, dev)),
              args=(PerProblem(T(mdl.y, dev)), PerProblem(T(mdl.cols, dev, torch.int64))),
              options=dict(cols=torch.as_tensor(mdl.cols), x_covariance=True), _lib=lib)
    same(r, base, "misaligned J view")


def check_host_inputs_cols(lib, dev):
    """Host (pinned CPU) x0, data and cols give the bits of the device-input
    solve, whole and in chunks."""
    rng = np.random.default_rng(8)
    n, B, W = 8, 100000, 24
    mdl = ColModel(n, W, 64, mixed_cols(rng, n, 64), seed=12)
    y = np.tile(mdl.y, (B // 64 + 1, 1))[:B].copy()
    x0 = np.tile(mdl.x0, (B // 64 + 1, 1))[:B].copy()
    cols = rng.integers(1, n + 1, B)
    At, Bt = T(mdl.A, dev), T(mdl.Bm, dev)

    def fun(X, Y):
        return X @ At.T + 0.3 * torch.sin(X @ Bt.T) - Y

    def jac(X, Y):
        return At[None] + 0.3 * torch.cos(X @ Bt.T)[:, :, None] * Bt[None]
    base = least_squares_batched(fun, T(x0, dev), jac=jac, bounds=(mdl.lb, mdl.ub),
                                 args=(PerProblem(T(y, dev)),),
                                 options=dict(cols=T(cols, dev, torch.int32)))
    yh = torch.as_tensor(y).pin_memory()
    for opts in (dict(h2d_chunks=3, prologue_rounds=4), dict(h2d_chunks=2, chunk=40000)):
        r = least_squares_batched(fun, torch.as_tensor(x0).pin_memory(), jac=jac,
                                  bounds=(mdl.lb, mdl.ub), args=(PerProblem(yh),),
                                  options=dict(cols=torch.as_tensor(cols), **opts))
        same(r, base, ("host inputs", opts), fields=FIELDS[:-1])


# ------------------------------------------------------------------ tests --

CHECKS = [check_full_cols_is_dense, check_ragged_equals_reduced, check_padding_never_read,
          check_vs_oracle, check_corpus_ragged_cols, check_invariance, check_api_errors,
          check_lin_ld_instances]
CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    """tests/host_emul/emul_cols.cpp (the host emulation for n = 1..16 plus the
    ragged-parameter entry points), built into a temporary directory."""
    out = str(tmp_path_factory.mktemp("emul_cols") / "libblsq_hostemul_cols.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC",
                           "-ffp-contract=off", "-mfma", "-x", "c++", EMUL_COLS, "-o", out])
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
@pytest.mark.parametrize("check", CHECKS + [check_ld_alignment, check_host_inputs_cols],
                         ids=lambda c: c.__name__[6:])
def test_gpu(cuda_lib, check):
    dev = torch.device("cuda:0")
    if check is check_invariance:
        print(check(cuda_lib, dev, graph=True))
    else:
        print(check(cuda_lib, dev))
