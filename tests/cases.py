"""Parity cases shared by the CPU (host-emulated core) and GPU (C ABI) suites.

Every function takes ``lib`` (a bounded_lsq_b200._lib.Lib) and a torch device.
The GPU suite passes the CUDA library -- those are the parity tests proper;
the CPU suite passes tests/host_emul (same per-problem C++, host build) so the
branch logic is exercised in the GPU-less container.
"""
import json
import os
import warnings

import numpy as np
import pytest
import torch

import packed_npz
from bounded_lsq_b200 import least_squares, least_squares_batched, PerProblem
from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak, RatPoly5

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SQ = np.finfo(float).eps ** 0.5


def T(a, dev, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def bits(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


# ---------------------------------------------------------------- helpers --

def check_helpers_bit_exact(lib, dev):
    """bounds.py / dogbox.py:9-35 / FD steps against the reference's outputs
    (tests/golden/helpers.npz), bit for bit."""
    z = packed_npz.Packed(os.path.join(GOLDEN, "helpers.npz"))
    n_cases = int(z["ncases"])
    for i in range(n_cases):
        g = lambda k: z[f"c{i}_{k}"]            # noqa: E731
        x, xc, d, lb, ub = g("x"), g("xc"), g("d"), g("lb"), g("ub")
        n = x.size
        X, XC, D = T(x[None], dev), T(xc[None], dev), T(d[None], dev)
        LB, UB = T(lb, dev), T(ub, dev)
        step, hits = lib.step_size_to_bound(X, D, LB, UB)
        # the SIGN of a zero minimum is not defined by NumPy itself (its
        # SIMD min reduction picks either zero depending on n and the CPU),
        # so +0.0 == -0.0 here; everything else is compared bit for bit
        sv = step.cpu().numpy()[0]
        assert bits(sv, g("step")) or (sv == 0 and g("step") == 0), i
        assert bits(hits.cpu().numpy()[0], g("hits")), i
        for rtol, key in ((1e-3, "act_1e3"), (SQ, "act_sq")):
            m = lib.find_active_constraints(X, LB, UB, rtol)
            assert bits(m.cpu().numpy()[0], g(key)), (i, key)
        for rstep, key in ((0.0, "msf0"), (1e-10, "msf1")):
            y = lib.make_strictly_feasible(XC, LB, UB, rstep)
            assert bits(y.cpu().numpy()[0], g(key)), (i, key)
        v, jv = lib.scaling_vector(XC, T(g("g")[None], dev), LB, UB)
        assert bits(v.cpu().numpy()[0], g("v")) and bits(jv.cpu().numpy()[0], g("jv")), i
        ok = lib.in_bounds(X, LB, UB)
        assert bool(ok.cpu().numpy()[0]) == bool(g("inb")), i
        lo, hi, fl = lib.find_intersection(XC, T(g("tr")[None], dev), LB, UB)
        fl = fl.cpu().numpy()[0]
        assert bits(lo.cpu().numpy()[0], g("fi_lo")) and bits(hi.cpu().numpy()[0], g("fi_hi")), i
        for bit, key in enumerate(("fi_ol", "fi_ou", "fi_tl", "fi_tu")):
            assert bits(((fl >> bit) & 1).astype(bool), g(key)), (i, key)
        # FD steps (scipy _numdiff) through blsq_fd2_points
        for rel, key in ((float("nan"), "fd2"), (1e-2, "fd2_rel")):
            Xp = torch.empty((n, 1, n), dtype=torch.float64, device=dev)
            dx = torch.empty((1, n), dtype=torch.float64, device=dev)
            lib.call("blsq_fd2_points", 1, None, n, XC.data_ptr(),
                     LB.data_ptr(), UB.data_ptr(), 0, rel, Xp.data_ptr(),
                     dx.data_ptr(), lib.stream(XC))
            h = g(key)
            want_pts = xc[None, :] + np.diag(h)
            want_dx = (xc + h) - xc
            assert bits(Xp.cpu().numpy()[:, 0, :], want_pts), (i, key)
            assert bits(dx.cpu().numpy()[0], want_dx), (i, key)
        # 3-point scheme through blsq_fd3_points: h and the one-sided flags
        Xp = torch.empty((2 * n, 1, n), dtype=torch.float64, device=dev)
        dxo = torch.empty((1, 2 * n), dtype=torch.float64, device=dev)
        lib.call("blsq_fd3_points", 1, None, n, XC.data_ptr(), LB.data_ptr(),
                 UB.data_ptr(), 0, float("nan"), Xp.data_ptr(), dxo.data_ptr(),
                 lib.stream(XC))
        h, one = g("fd3"), g("fd3_one").astype(bool)
        x1 = np.where(one, xc + h, xc - h)
        x2 = np.where(one, xc + 2 * h, xc + h)
        pts = Xp.cpu().numpy()[:, 0, :]
        want1 = np.tile(xc, (n, 1))
        want2 = np.tile(xc, (n, 1))
        want1[np.arange(n), np.arange(n)] = x1
        want2[np.arange(n), np.arange(n)] = x2
        assert bits(pts[0::2], want1) and bits(pts[1::2], want2), (i, "fd3")
        want_dx = np.where(one, x2 - xc, x2 - x1)
        out = dxo.cpu().numpy()[0]
        assert bits(out[:n], want_dx), (i, "fd3 dx")
        assert np.array_equal(out[n:] != 0, one), (i, "fd3 one-sided")
    return n_cases


def check_helpers_batched_rows(lib, dev, B=4096, n=6, seed=3):
    """Same passes on a (B, n) batch with per-problem bounds against NumPy
    restatements row by row (bit-exact), incl. ties and infinities."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    lb = rng.uniform(-3, 0, (B, n))
    ub = lb + rng.uniform(0.1, 4, (B, n))
    lb[rng.random((B, n)) < 0.15] = -np.inf
    ub[rng.random((B, n)) < 0.15] = np.inf
    x = np.clip(rng.standard_normal((B, n)), lb, ub)
    d = rng.standard_normal((B, n))
    d[rng.random((B, n)) < 0.1] = 0.0
    d[::5, 1] = d[::5, 0]
    x[::5, 1], lb[::5, 1], ub[::5, 1] = x[::5, 0], lb[::5, 0], ub[::5, 0]
    g = rng.standard_normal((B, n))
    step, hits = lib.step_size_to_bound(T(x, dev), T(d, dev), T(lb, dev), T(ub, dev))
    act = lib.find_active_constraints(T(x, dev), T(lb, dev), T(ub, dev), 1e-3)
    msf = lib.make_strictly_feasible(T(x, dev), T(lb, dev), T(ub, dev), 0.0)
    v, jv = lib.scaling_vector(T(x, dev), T(g, dev), T(lb, dev), T(ub, dev))
    step, hits, act, msf, v, jv = (t.cpu().numpy() for t in (step, hits, act, msf, v, jv))
    for b in range(0, B, 7):
        s, h = orc.step_size_to_bound(x[b], d[b], lb[b], ub[b])
        assert (bits(step[b], s) or (step[b] == 0 and s == 0)) and bits(hits[b], h), b
        assert bits(act[b], orc.find_active_constraints(x[b], lb[b], ub[b], 1e-3)), b
        assert bits(msf[b], orc.make_strictly_feasible(x[b], lb[b], ub[b], 0)), b
        ov, ojv = orc.scaling_vector(x[b], g[b], lb[b], ub[b])
        assert bits(v[b], ov) and bits(jv[b], ojv), b


# ------------------------------------------------------------ batched fits --

MODELS = {"c2": ExpDecay2, "c3": GaussPeak, "rat": RatPoly5}


def run_golden_batched(lib, dev, name, **options):
    """Solve the problems stored in tests/golden/<name>.npz (produced by the
    unmodified reference) and return (result, golden, first trial points)."""
    cfg, method, jac = name.split("_")
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    model = MODELS[cfg](int(json.loads(str(z["meta"]))["m"]))
    y = T(z["y"], dev)
    B = y.shape[0]
    X0 = T(np.tile(model.x0, (B, 1)), dev)
    trials = []

    def trace(r, idx, Xn, state, istate):
        if len(trials) < 4:
            full = torch.full((B, model.n), float("nan"), dtype=torch.float64,
                              device=dev)
            run = istate[:, 0] == -1
            if idx is None:
                full[run] = Xn[run]
            else:
                sel = run[idx]
                full[idx[sel]] = Xn[sel]
            trials.append(full.cpu().numpy())

    opts = dict(options)
    opts["trace"] = trace
    j = model.jac_t if jac == "exact" else {"2point": "2-point",
                                            "3point": "3-point"}[jac]
    res = least_squares_batched(
        model.fun_t, X0, jac=j, bounds=(model.lb, model.ub), method=method,
        args=(PerProblem(y),), options=opts, _lib=lib)
    return res, z, trials


def summarize(res, z, trials):
    x = res.x.cpu().numpy()
    obj = res.obj_value.cpu().numpy()
    st = res.status.cpu().numpy()
    out = dict(
        status_eq=float((st == z["status"]).mean()),
        nfev_eq=float((res.nfev.cpu().numpy() == z["nfev"]).mean()),
        njev_eq=float((res.njev.cpu().numpy() == z["njev"]).mean()),
        mask_eq=float((res.active_mask.cpu().numpy() == z["mask"]).all(1).mean()),
        x_rel=float((np.abs(x - z["x"]).max(1) / np.abs(z["x"]).max(1)).max()),
        obj_rel=float((np.abs(obj - z["obj"]) / z["obj"]).max()),
    )
    # per-iteration trial points (relative to the size of the step taken)
    gt = z["trials"]
    K = min(len(trials), gt.shape[1], 3)
    worst = 0.0
    for k in range(K):
        ok = ~np.isnan(gt[:, k]).any(1) & ~np.isnan(trials[k]).any(1)
        if ok.any():
            err = np.abs(trials[k][ok] - gt[ok, k]).max(1) / np.abs(gt[ok, k]).max(1)
            worst = max(worst, float(err.max()))
    out["trial_rel"] = worst
    return out


def check_golden_exact_jac(lib, dev, name):
    """Analytic-Jacobian configs: the north-star gates, all problems."""
    res, z, trials = run_golden_batched(lib, dev, name)
    s = summarize(res, z, trials)
    assert s["status_eq"] == 1.0, s
    assert s["nfev_eq"] == 1.0 and s["njev_eq"] == 1.0, s
    assert s["mask_eq"] == 1.0, s            # active sets bit-exact
    assert s["x_rel"] < 1e-8 and s["obj_rel"] < 1e-8, s   # north-star rtol
    assert s["trial_rel"] < 1e-10, s         # per-iteration steps
    return s


def check_golden_fd_jac(lib, dev, name):
    """2-point configs.  The golden residuals come from NumPy's exp, ours from
    torch's; a 1-ulp difference in f is amplified by 1/h ~ 6.7e7 in the FD
    Jacobian, so iterates agree to ~1e-8 and a few borderline ftol/xtol
    decisions move (SURVEY 7 hard part 1).  Gates: final cost/x within the
    north-star 1e-8, active sets exact, >= 95% identical status/nfev."""
    res, z, trials = run_golden_batched(lib, dev, name)
    s = summarize(res, z, trials)
    assert s["mask_eq"] == 1.0, s
    assert s["x_rel"] < 1e-8 and s["obj_rel"] < 1e-8, s
    # 3-point: h ~ 6e-6, so the 1-ulp noise is amplified 10x less than 2-point
    assert s["status_eq"] >= 0.95 and s["nfev_eq"] >= 0.95, s
    assert s["trial_rel"] < (1e-8 if name.endswith("3point") else 1e-7), s
    return s


def check_golden_fd_exact(lib, dev, name):
    """Finite-difference configs on the transcendental-free model (RatPoly5:
    only + - * /, so the device residuals are NumPy's to the last bit).  With
    bit-identical inputs the FIRST trial step must meet the north-star 1e-10
    (measured: 8e-15) -- the FD Jacobian at x0 is scipy's bit for bit
    (check_fd_linearise_bit_exact).  From the second step on no implementation
    that is not bit-identical can do better than ~1e-8 * cond(J): the accepted
    point differs from the reference's in the last bit, and a forward
    difference with h ~ 1.5e-8 turns the rounding noise of f (1e-16) into 1e-8
    of J, a different realisation at a different point.  Measured on the
    REFERENCE ITSELF (oracle, 1-ulp noise on f, 48 fits): x changes by up to
    2e-4 (trf) / 6e-6 (dogbox), cost by 3e-9 / 2e-6, nfev or status of 1 fit in
    48.  Gates: first step 1e-10; active sets bit-exact, status / nfev / cost
    (1e-8) equal for >= 95 % of the fits."""
    res, z, trials = run_golden_batched(lib, dev, name)
    s = summarize(res, z, trials)
    gt = z["trials"]
    ok = ~np.isnan(gt[:, 0]).any(1) & ~np.isnan(trials[0]).any(1)
    x0 = MODELS[name.split("_")[0]].x0
    err = np.abs(trials[0][ok] - gt[ok, 0]).max(1) / np.abs(gt[ok, 0] - x0).max(1)
    s["first_step_rel"] = float(err.max())
    obj = res.obj_value.cpu().numpy()
    s["obj_1e8_frac"] = float((np.abs(obj - z["obj"]) <= 1e-8 * z["obj"]).mean())
    assert ok.sum() >= 0.9 * len(ok) and s["first_step_rel"] < 1e-10, s
    assert s["mask_eq"] >= 0.95 and s["status_eq"] >= 0.95 and s["nfev_eq"] >= 0.95, s
    assert s["obj_1e8_frac"] >= 0.95, s
    return s


def check_fd_linearise_bit_exact(lib, dev, seed=3):
    """SURVEY 8a row a24 at kernel level: blsq_fd2_points / blsq_fd3_points +
    blsq_linearise_batched in finite-difference mode must produce, bit for
    bit, the record the analytic mode produces from scipy's own
    approx_derivative Jacobian.  Residuals are computed by NumPy and handed
    to the kernel as arrays (no callback in between), so this isolates the
    device arithmetic: the points, dx = (x + h) - x, the 3-point stencils and
    the correctly rounded quotient."""
    from scipy.optimize._numdiff import approx_derivative
    from bounded_lsq_b200.synthetic import GaussPeak
    rng = np.random.default_rng(seed)
    out = {}
    for model in (RatPoly5(40), GaussPeak(128), RatPoly5(300)):
        n, m = model.n, model.m
        B = 24
        _, y = model.make_data(B, seed=seed)
        # points inside, on and next to the bounds
        X = rng.uniform(model.lb, model.ub, (B, n))
        X[::4, 0] = model.lb[0]
        X[1::4, n - 1] = model.ub[n - 1]
        X[2::4, 1] = np.nextafter(model.ub[1], -np.inf)
        LS = lib.lin_record_size(n)
        ist = torch.zeros((B, 8), dtype=torch.int32, device=dev)
        ist[:, 0] = -1
        F0 = np.stack([model.fun_np(X[b], y[b]) for b in range(B)])
        st = lib.stream(ist)
        for mode, meth in ((1, "2-point"), (2, "3-point")):
            npts = n * mode
            Xp = torch.empty((npts, B, n), dtype=torch.float64, device=dev)
            dx = torch.empty((B, npts), dtype=torch.float64, device=dev)
            Xt, lbt, ubt = T(X, dev), T(model.lb, dev), T(model.ub, dev)
            lib.call("blsq_fd3_points" if mode == 2 else "blsq_fd2_points", B, None, n,
                     Xt.data_ptr(), lbt.data_ptr(), ubt.data_ptr(), 0, float("nan"),
                     Xp.data_ptr(), dx.data_ptr(), st)
            P = Xp.cpu().numpy()
            Fp = [T(np.stack([model.fun_np(P[i, b], y[b]) for b in range(B)]), dev)
                  for i in range(npts)]
            import ctypes as C
            plist = (C.c_void_p * npts)(*[t.data_ptr() for t in Fp])
            Ft = T(F0, dev)
            lin_fd = torch.zeros((B, LS), dtype=torch.float64, device=dev)
            lib.call("blsq_linearise_batched", B, None, m, n, Ft.data_ptr(), None,
                     C.cast(plist, C.c_void_p), dx.data_ptr(), mode, ist.data_ptr(),
                     lin_fd.data_ptr(), st)
            J = np.stack([approx_derivative(lambda xx, b=b: model.fun_np(xx, y[b]), X[b],
                                            method=meth, f0=F0[b],
                                            bounds=(model.lb, model.ub))
                          for b in range(B)])
            lin_an = torch.zeros((B, LS), dtype=torch.float64, device=dev)
            Jt = T(J, dev)
            lib.call("blsq_linearise_batched", B, None, m, n, Ft.data_ptr(),
                     Jt.data_ptr(), None, None, 0, ist.data_ptr(),
                     lin_an.data_ptr(), st)
            assert bits(lin_fd.cpu().numpy(), lin_an.cpu().numpy()), (type(model).__name__, m, meth)
            out[(type(model).__name__, m, meth)] = True
    return out


def check_compaction_invariance(lib, dev):
    """Results must not depend on when the active set is compacted or how
    often the host looks at the status flags."""
    base, z, _ = run_golden_batched(lib, dev, "c2_trf_exact", compact_below=0.0)
    for opts in (dict(compact_below=1.0), dict(check_every=3, compact_below=0.5)):
        r, _, _ = run_golden_batched(lib, dev, "c2_trf_exact", **opts)
        assert bits(r.x.cpu().numpy(), base.x.cpu().numpy()), opts
        assert bits(r.status.cpu().numpy(), base.status.cpu().numpy()), opts
        assert bits(r.nfev.cpu().numpy(), base.nfev.cpu().numpy()), opts


def check_graph_tail_invariance(lib, dev):
    """The CUDA-graph tail (rounds captured once and replayed) must give the
    same bits as eager rounds, with torch callbacks, with the 2-point path, and
    must fall back to eager rounds when a callback cannot be captured."""
    out = {}
    for cfg, method, jac in (("c2", "trf", "exact"), ("c3", "dogbox", "2-point")):
        model = MODELS[cfg]()
        B = 3000
        _, y = model.make_data(B, seed=77)
        yt = T(y, dev)
        X0 = T(np.tile(model.x0, (B, 1)), dev)
        j = model.jac_t if jac == "exact" else jac

        def solve(fun=model.fun_t, **opts):
            return least_squares_batched(
                fun, X0, jac=j, bounds=(model.lb, model.ub), method=method,
                args=(PerProblem(yt),), options=opts, _lib=lib)

        def syncing_fun(X, yy):
            float(X[0, 0].item())              # host sync: not capturable
            return model.fun_t(X, yy)

        base = solve(graph_tail_rounds=0)
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            r_fallback = solve(fun=syncing_fun)
        assert any("could not be captured" in str(w.message) for w in caught)
        # ... and a failed capture must not poison the next one
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            r_g8 = solve()
            r_g3 = solve(graph_tail_rounds=3, tail_below=2000)
        assert not any("could not be captured" in str(w.message) for w in caught), \
            [str(w.message) for w in caught]
        for label, r in (("graph8", r_g8), ("graph3", r_g3), ("fallback", r_fallback)):
            for fld in ("x", "obj_value", "status", "nfev", "njev", "active_mask"):
                assert bits(getattr(r, fld).cpu().numpy(),
                            getattr(base, fld).cpu().numpy()), (cfg, label, fld)
            out[(cfg, label)] = (r.rounds, base.rounds)
        assert int((base.status > 0).sum()) == B
    return out


def check_prologue_invariance(lib, dev, host_inputs=False):
    """Streaming start (each chunk of problems runs its first rounds alone,
    then the batch carries on in lock step): same bits as the plain solve.
    With host_inputs the data is handed over as pinned CPU tensors and the
    front end stages it chunk by chunk."""
    for cfg, method, jac in (("c2", "trf", "exact"), ("c3", "dogbox", "2-point"),
                             ("c2", "dogbox", "exact")):
        model = MODELS[cfg]()
        B = 1500 if not host_inputs else 200000
        _, y = model.make_data(min(B, 4096), seed=5)
        y = np.tile(y, (-(-B // y.shape[0]), 1))[:B].copy()
        yt = T(y, dev)
        X0 = T(np.tile(model.x0, (B, 1)), dev)
        j = model.jac_t if jac == "exact" else jac
        lbt, ubt = T(model.lb, dev), T(model.ub, dev)

        def solve(x0=X0, yy=yt, **opts):
            return least_squares_batched(
                model.fun_t, x0, jac=j, bounds=(lbt, ubt), method=method,
                args=(PerProblem(yy),), options=opts, _lib=lib)

        base = solve()
        runs = [solve(prologue=[(0, 400, None), (400, 1001, None), (1001, B, None)],
                      prologue_rounds=3),
                solve(prologue=[(0, B, None)], prologue_rounds=50)]
        if host_inputs:
            runs.append(solve(x0=X0.cpu().pin_memory(), yy=yt.cpu().pin_memory(),
                              h2d_chunks=3, prologue_rounds=4))
        for k, r in enumerate(runs):
            for fld in ("x", "obj_value", "status", "nfev", "njev", "active_mask"):
                assert bits(getattr(r, fld).cpu().numpy(),
                            getattr(base, fld).cpu().numpy()), (cfg, method, k, fld)


def check_per_problem_bounds(lib, dev):
    """(B, n) bounds give the same answers as shared (n,) bounds."""
    model = ExpDecay2()
    z = np.load(os.path.join(GOLDEN, "c2_trf_exact.npz"))
    y = T(z["y"][:64], dev)
    B = 64
    X0 = T(np.tile(model.x0, (B, 1)), dev)
    for method in ("trf", "dogbox"):
        r1 = least_squares_batched(model.fun_t, X0, jac=model.jac_t,
                                   bounds=(model.lb, model.ub), method=method,
                                   args=(PerProblem(y),), _lib=lib)
        lbB = T(np.tile(model.lb, (B, 1)), dev)
        ubB = T(np.tile(model.ub, (B, 1)), dev)
        r2 = least_squares_batched(model.fun_t, X0, jac=model.jac_t,
                                   bounds=(lbB, ubB), method=method,
                                   args=(PerProblem(y),), _lib=lib)
        assert bits(r1.x.cpu().numpy(), r2.x.cpu().numpy())
        assert bits(r1.active_mask.cpu().numpy(), r2.active_mask.cpu().numpy())


# ------------------------------------------------------- small-n corpus ----

def corpus_cases(max_n=None):
    """(name, method, jacmode, scaling) of the golden corpus (config #1: the 58
    instances of the reference suite) with n <= max_n."""
    from problems import corpus
    z = np.load(os.path.join(GOLDEN, "corpus.npz"))
    probs = {p.name: p for p in corpus()}
    out = []
    for key in z.files:
        if not key.endswith("|x"):
            continue
        name, method, jm, sc, _ = key.split("|")
        p = probs[name]
        if (max_n is None or p.n <= max_n) and jm in ("exact", "2-point", "3-point"):
            out.append((name, method, jm, sc))
    return out, z, probs


def self_sensitive(z, key):
    """Is this run ulp-chaotic IN THE REFERENCE?  corpus.npz stores, for every
    analytic-Jacobian run, what the unmodified reference does to its own result
    when its residuals carry 1-ulp noise (make_golden.self_sensitivity): x_rel,
    obj_rel, runs whose nfev changed, runs whose status changed.  A run is
    waived from the x / nfev / status gates only on that measured evidence
    (SURVEY 7 hard part 1), never by name.  Returns (waived, cost tolerance)."""
    k = key + "sens"
    if k not in z.files:
        return False, 1e-8
    xr, orr, dn, ds, fs = z[k]
    waived = bool(dn > 0 or ds > 0 or xr > 1e-9 or fs > 1e-11)
    return waived, (min(0.5, max(1e-3, 10.0 * orr)) if waived else 1e-8)


def first_step_sensitive(z, name, method, sc):
    """The reference's own first step moves by more than 1e-11 under a few ulps
    of noise on f (an exact tie of a branch test at x0, see
    make_golden.self_sensitivity): the 1e-10 gate on the first step is waived."""
    k = f"{name}|{method}|exact|{sc}|sens"
    return k in z.files and z[k][4] > 1e-11


def check_corpus_single(lib, dev, max_n=None, names=None):
    """Config #1 (the reference's benchmark suite) through the single-problem
    front end: n <= 8 on the batched kernels (B = 1), larger n on the tall
    kernels."""
    cases, z, probs = corpus_cases(max_n)
    stats = dict(total=0, exact_status=0, waived=0, fd_total=0, fd_exact=0)
    for name, method, jm, sc in cases:
        if names is not None and name not in names:
            continue
        p = probs[name]
        key = f"{name}|{method}|{jm}|{sc}|"
        obj, status, nfev, njev, opt, ntr = z[key + "scalars"]

        def fun(x, p=p):
            return p.fun(x.cpu().numpy())

        def jac(x, p=p):
            return p.jac(x.cpu().numpy())

        scaling = 'jac' if sc == 'jac' else 1.0
        first_trial = []

        def trace(*a, ft=first_trial):
            # batched driver: (round, idx, Xnew, state, istate); tall: (x_new, state, istate)
            if not ft:
                xn = a[2][0] if len(a) == 5 else a[0]
                ft.append(xn.cpu().numpy().copy())

        res = least_squares(fun, p.x0, jac=jac if jm == "exact" else jm,
                            bounds=(p.lb, p.ub), method=method,
                            scaling=scaling, options=dict(trace=trace), _lib=lib)
        stats["total"] += 1
        x = res.x.cpu().numpy()
        assert np.all(x >= p.lb) and np.all(x <= p.ub), key
        assert res.status >= 0, key
        gt = z[key + "trials"]
        if first_trial and not np.isnan(gt[0]).any() and \
                not first_step_sensitive(z, name, method, sc):
            # the first step from x0 meets the north-star 1e-10 on EVERY run
            # (also the finite-difference and the self-sensitive ones): the
            # inputs of that step are bit-identical
            stepn = max(np.abs(gt[0] - p.x0).max(), 1e-300)
            e0 = float(np.abs(first_trial[0] - gt[0]).max() / stepn)
            stats["first_step_rel"] = max(stats.get("first_step_rel", 0.0), e0)
            assert e0 < 1e-10, (key, e0)
        waived, tol = self_sensitive(z, key)
        if jm != "exact":
            # finite differences: later Jacobians are taken at points that
            # differ in the last bit and carry another realisation of the 1e-8
            # rounding noise of the difference quotient (check_golden_fd_exact):
            # status and nfev are counted, the cost compared loosely
            base_waived, _ = self_sensitive(z, f"{name}|{method}|exact|{sc}|")
            if status > 0 and res.status > 0 and obj > 1e-20 and not base_waived:
                assert abs(res.obj_value - obj) <= 1e-3 * max(obj, 1e-9), \
                    (key, res.obj_value, obj)
            if not base_waived:
                stats["fd_total"] += 1
                stats["fd_exact"] += (res.status == int(status) and
                                      res.nfev == int(nfev))
            continue
        if waived:
            stats["waived"] += 1
            if status > 0 and res.status > 0 and obj > 1e-20:
                assert abs(res.obj_value - obj) <= tol * max(obj, 1e-9), \
                    (key, res.obj_value, obj, tol)
            continue
        assert res.status == int(status), (key, res.status, status)
        assert res.nfev == int(nfev) and res.njev == int(njev), key
        assert bits(res.active_mask.cpu().numpy(), z[key + "mask"]), key
        gx = z[key + "x"]
        assert np.allclose(x, gx, rtol=1e-8, atol=1e-8 * np.abs(gx).max()), \
            (key, x, gx)
        # zero-residual problems end at obj ~ 1e-30: absolute floor 1e-18
        assert abs(res.obj_value - obj) <= 1e-8 * obj + 1e-18, key
        stats["exact_status"] += 1
    assert stats["fd_exact"] >= 0.93 * stats["fd_total"], stats
    return stats


# ------------------------------------------------------------------ tall --

def run_tall_golden(lib, dev, tag, method, shards=1, file="tall.npz", **kw):
    """One tall problem of tests/golden/tall.npz (C4-like) or c5.npz (C5-like:
    n up to 256, lb = 0 so that half of the bounds are active), both written
    by the unmodified reference, through least_squares ->
    bounded_lsq_b200.tall."""
    from bounded_lsq_b200.synthetic import TallLinExp
    z = np.load(os.path.join(GOLDEN, file))
    meta = [m for m in json.loads(str(z["meta"]))
            if m["tag"] == tag and m["method"] == method][0]
    kw_wl = {} if meta.get("x0_tail") is None else dict(x0_tail=meta["x0_tail"])
    if "lb" in meta:
        kw_wl["lb"] = meta["lb"]
    wl = TallLinExp(meta["m"], meta["n"], seed=meta["seed"], **kw_wl).to_device(dev)
    assert bits(np.float64(np.sum(wl.y)), z[f"{tag}_y_checksum"])
    trials = []

    def trace(xn, state, istate):
        if len(trials) < 4:
            trials.append(xn.cpu().numpy())

    res = least_squares(wl.fun_t, T(wl.x0, dev), jac=wl.jac_t,
                        bounds=(T(wl.lb, dev), T(wl.ub, dev)), method=method,
                        options=dict(trace=trace), _lib=lib, **kw)
    pre = f"{tag}_{method}_"
    return res, z, pre, trials, wl


def check_tall_golden(lib, dev, tag, method, file="tall.npz"):
    res, z, pre, trials, wl = run_tall_golden(lib, dev, tag, method, file=file)
    obj, status, nfev, njev, opt, ntr = z[pre + "scalars"]
    gx = z[pre + "x"]
    x = res.x.cpu().numpy()
    s = dict(status=(res.status, int(status)), nfev=(res.nfev, int(nfev)),
             njev=(res.njev, int(njev)),
             x_rel=float(np.abs(x - gx).max() / np.abs(gx).max()),
             obj_rel=abs(res.obj_value - obj) / obj,
             mask_eq=bits(res.active_mask.cpu().numpy(), z[pre + "mask"]))
    gt = z[pre + "trials"]
    worst = 0.0
    prev = np.asarray(wl.x0, float)
    for k in range(min(len(trials), 3)):
        if np.isnan(gt[k]).any():
            break
        # relative to the size of the step taken (north star: 1e-10)
        stepn = max(np.abs(gt[k] - prev).max(), 1e-300)
        worst = max(worst, float(np.abs(trials[k] - gt[k]).max() / stepn))
        prev = gt[k]
    s["trial_rel"] = worst
    assert s["status"][0] == s["status"][1], s
    assert s["obj_rel"] < 1e-8, s                            # north-star rtol
    assert s["trial_rel"] < 1e-10, s                         # first iterations
    s["nactive"] = int(np.count_nonzero(z[pre + "mask"]))
    # h = the C5 benchmark start (identical exponentials, like a/b)
    chaotic = tag in ("a", "b", "h") and method == "trf"
    if not chaotic:
        # tags a/b start TRF at an exactly rank-deficient Jacobian (identical
        # exponentials): rounding decides which of the two mirror-image minima
        # (the exponentials swapped) is reached and after how many steps -- the
        # reference does not reproduce its own x / nfev / active set there
        # under 1-ulp noise on f (DESIGN.md section 5) -- so only the gates
        # above apply; everywhere else x, the counters and the active set must
        # match too
        assert s["mask_eq"], s                               # active set bit-exact
        assert s["nfev"][0] == s["nfev"][1] and s["njev"][0] == s["njev"][1], s
        assert s["x_rel"] < 1e-8, s
    # result fields of the reference (least_squares.py:206-252)
    assert res.fun.shape == (wl.m,) and res.jac.shape == (wl.m, wl.n)
    assert res.success == (res.status > 0)
    return s


def tall_factor(lib, J, f, shards=1, sstride=1):
    """Preconditioned Cholesky QR of [J | f] through the C ABI (CholeskyQR2
    when sstride == 1); `shards` > 1 splits the rows into rank-like pieces
    whose records are summed by blsq_tall_factor."""
    m, n = J.shape
    dev = J.device
    lay = lib.tall_layout(n)
    f64 = torch.float64
    GS = lay["record"]
    work = torch.empty(max(lay["gram_work"], 1), dtype=f64, device=dev)
    fac = torch.zeros(lay["fac_size"], dtype=f64, device=dev)
    recs = torch.empty((shards, GS), dtype=f64, device=dev)
    st = lib.stream(J)
    cut = [(m * r // shards) // 2 * 2 for r in range(shards)] + [m]

    def gram(p):
        for r in range(shards):
            a, b = cut[r], cut[r + 1]
            lib.call("blsq_tall_gram", p, b - a, n, J[a:b].data_ptr(),
                     f[a:b].data_ptr(), fac[lay["rinvp"]:].data_ptr(),
                     sstride if p == 1 else 1, work.data_ptr(),
                     recs[r].data_ptr(), st)

    def factor(p):
        lib.call("blsq_tall_factor", p, n, shards, GS, recs.data_ptr(),
                 fac.data_ptr(), st)

    gram(1); factor(1); gram(2); factor(2)
    refined = 0
    while sstride > 1 and float(fac[lay["refine"]]) != 0.0 and refined < 2:
        factor(3); gram(2); factor(2)
        refined += 1
    R = fac[lay["R"]:lay["R"] + n * n].view(n, n)
    return dict(R=R, qtf=fac[lay["qtf"]:lay["qtf"] + n],
                g=fac[lay["g"]:lay["g"] + n], obj=float(fac[lay["fobj"]]),
                info=float(fac[lay["info"]]), refined=refined)


def check_tall_factor(lib, dev):
    gen = torch.Generator(device="cpu").manual_seed(5)
    rel = lambda a, b: float((a - b).norm() / b.norm())        # noqa: E731
    for (m, n, shards) in ((1000, 10, 1), (4099, 16, 2), (20001, 64, 3),
                           (7777, 24, 1), (5000, 100, 2), (3000, 130, 1),
                           (901, 9, 1), (6005, 33, 2), (2047, 67, 1)):
        J = torch.randn((m, n), dtype=torch.float64, generator=gen).to(dev)
        f = torch.randn(m, dtype=torch.float64, generator=gen).to(dev)
        out = tall_factor(lib, J, f, shards)
        assert out["info"] == 0.0
        Q, R = torch.linalg.qr(J)
        sg = torch.sign(torch.diagonal(R))
        assert rel(out["R"], R * sg[:, None]) < 1e-13, (m, n)
        assert rel(out["qtf"], (Q * sg[None, :]).T @ f) < 1e-12, (m, n)
        assert rel(out["g"], J.T @ f) < 1e-13, (m, n)
        assert abs(out["obj"] - float(f @ f)) < 1e-13 * float(f @ f)
        assert float(out["R"].tril(-1).abs().max()) == 0.0
    # sampled preconditioner: pass 1 on one 64-row tile out of 4.  Homogeneous
    # rows -> accepted as is; ten huge rows in a tile the sample misses -> the
    # verification asks for another pass; both end at the same accuracy
    def sampled_tiles(ntiles, sstride):
        jobs = np.arange(ntiles // sstride, dtype=np.uint32)
        h = jobs * np.uint32(2654435761)
        h ^= h >> np.uint32(15)
        return set((jobs.astype(np.int64) * sstride + (h % sstride)).tolist())

    for spike in (False, True):
        J = torch.randn((40000, 16), dtype=torch.float64, generator=gen).to(dev)
        if spike:
            miss = [t for t in range(16, 40) if t not in sampled_tiles(40000 // 64, 4)][0]
            J[miss * 64 + 5:miss * 64 + 15] *= 1e3
        f = torch.randn(40000, dtype=torch.float64, generator=gen).to(dev)
        out = tall_factor(lib, J, f, shards=1, sstride=4)
        assert out["info"] == 0.0 and out["refined"] == (1 if spike else 0), out["refined"]
        Q, R = torch.linalg.qr(J)
        sg = torch.sign(torch.diagonal(R))
        assert rel(out["R"], R * sg[:, None]) < 1e-13
        assert rel(out["qtf"], (Q * sg[None, :]).T @ f) < 1e-12
        assert rel(out["g"], J.T @ f) < 1e-13
    # exactly rank-deficient Jacobian (two identical columns): the shifted
    # Cholesky must still deliver R^T R = J^T J to rounding
    J = torch.randn((5000, 16), dtype=torch.float64, generator=gen).to(dev)
    J[:, 9] = J[:, 3]
    f = torch.randn(5000, dtype=torch.float64, generator=gen).to(dev)
    out = tall_factor(lib, J, f)
    assert out["info"] == 0.0
    G = J.T @ J
    assert float((out["R"].T @ out["R"] - G).abs().max() / G.abs().max()) < 1e-12
    assert rel(out["R"].T @ out["qtf"], J.T @ f) < 1e-6


def check_tall_large(lib, dev, m=1 << 22, n=64):
    from bounded_lsq_b200.synthetic import TallLinExp
    wl = TallLinExp(m, n, seed=1, x0_tail=(0.8, 1.5, 0.3, 4.0)).to_device(dev)
    x0 = T(wl.x0, dev)
    J = wl.jac_t(x0).clone()
    f = wl.fun_t(x0)
    out = tall_factor(lib, J, f)
    G = J.T @ J
    assert float((out["R"].T @ out["R"] - G).abs().max() / G.abs().max()) < 1e-13
    g = J.T @ f
    assert float((out["R"].T @ out["qtf"] - g).norm() / g.norm()) < 1e-12
    assert float((out["g"] - g).norm() / g.norm()) < 1e-13
    del J
    obj0 = float(f @ f)
    objs = []
    for method in ("trf", "dogbox"):
        res = least_squares(wl.fun_t, x0, jac=wl.jac_t,
                            bounds=(T(wl.lb, dev), T(wl.ub, dev)), method=method,
                            _lib=lib)
        assert res.status > 0, (method, res.status)
        assert bool(((res.x >= T(wl.lb, dev)) & (res.x <= T(wl.ub, dev))).all())
        assert res.obj_value < obj0
        # the returned cost is the cost at the returned point
        fx = wl.fun_t(res.x)
        assert abs(float(fx @ fx) - res.obj_value) <= 1e-12 * res.obj_value
        assert res.nfev >= res.njev >= 2
        objs.append(res.obj_value)
    # both methods reach the same bounded minimum (ftol = sqrt(eps))
    assert abs(objs[0] - objs[1]) <= 1e-6 * objs[1], objs


def check_tall_options_vs_oracle(lib, dev, m=3000, n=12):
    """Tall mode with scaling='jac', a scaling vector and jac='2-point',
    side by side with the oracle (bit-identical to the reference on the golden
    files) on the same small C4-like problem: status, counters and active set
    equal, x and cost to the north-star 1e-8."""
    from oracle import blsq_oracle as orc
    from bounded_lsq_b200.synthetic import TallLinExp
    wl = TallLinExp(m, n, seed=11, x0_tail=(0.8, 1.5, 0.3, 4.0)).to_device(dev)
    rng = np.random.default_rng(4)
    svec = rng.uniform(0.5, 2.0, n)
    out = {}
    for method in ("trf", "dogbox"):
        for label, kw_o, kw_g in (
                ("jac", dict(scaling="jac"), dict(scaling="jac")),
                ("vec", dict(scaling=svec), dict(scaling=T(svec, dev))),
                ("fd", dict(jac="2-point"), dict(jac="2-point")),
                ("fd3", dict(jac="3-point"), dict(jac="3-point"))):
            ko = dict(jac=wl.jac_np)
            ko.update(kw_o)
            kg = dict(jac=wl.jac_t)
            kg.update(kw_g)
            ref = orc.least_squares(wl.fun_np, wl.x0, bounds=(wl.lb, wl.ub),
                                    method=method, **ko)
            res = least_squares(wl.fun_t, T(wl.x0, dev),
                                bounds=(T(wl.lb, dev), T(wl.ub, dev)),
                                method=method, _lib=lib, **kg)
            x = res.x.cpu().numpy()
            s = dict(status=(res.status, ref.status), nfev=(res.nfev, ref.nfev),
                     njev=(res.njev, ref.njev),
                     x_rel=float(np.abs(x - ref.x).max() / np.abs(ref.x).max()),
                     obj_rel=abs(res.obj_value - ref.obj_value) / ref.obj_value,
                     mask_eq=bits(res.active_mask.cpu().numpy(),
                                  np.asarray(ref.active_mask, dtype=np.int64)))
            out[(method, label)] = s
            assert s["status"][0] == s["status"][1], (method, label, s)
            assert s["mask_eq"], (method, label, s)
            assert s["obj_rel"] < 1e-8, (method, label, s)
            if not label.startswith("fd"):
                assert s["x_rel"] < 1e-8, (method, label, s)
                assert s["nfev"][0] == s["nfev"][1], (method, label, s)
            else:
                # torch's exp / gemv differ from NumPy's by an ulp; the forward
                # difference amplifies that by 1/h ~ 7e7 into J (1e-8 relative),
                # and cond(J) ~ 1e3 turns it into ~1e-5 in the weakly determined
                # exponents, while the cost agrees to 1e-12.  No implementation
                # that is not bit-identical in f can do better here.
                # (3-point: h ~ 6e-6, amplification 10x smaller)
                assert s["x_rel"] < (1e-4 if label == "fd" else 1e-6), \
                    (method, label, s)
            assert res.jac.shape == (m, n)
    return out


# ------------------------------------------------ benchmark driver (8f #3) --

def check_benchmark_table(lib, dev, out_path, max_n=None):
    """benchmarks/run_benchmarks.py (the reference's table from this path):
    every row must carry the reference's nfev / status / value / number of
    active bounds (golden corpus), except the runs the reference does not
    reproduce itself under 1-ulp noise (self_sensitive)."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location(
        "blsq_run_benchmarks", os.path.join(root, "benchmarks", "run_benchmarks.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rows = mod.main([str(out_path)], lib=lib, dev=dev, max_n=max_n)   # unbounded + bounded
    z = np.load(os.path.join(GOLDEN, "corpus.npz"))
    checked = unsupported = waived = 0
    for name, meth, r in rows:
        if r is None:
            unsupported += 1
            continue
        solver, sc = (meth[:-2], "jac") if meth.endswith("-s") else (meth, "1")
        key = f"{name}|{solver}|exact|{sc}|"
        if key + "scalars" not in z.files:
            continue
        if self_sensitive(z, key)[0]:
            waived += 1
            continue
        obj, status, nfev, njev, opt, ntr = z[key + "scalars"]
        mask = z[key + "mask"]
        assert r[4] == int(status) and r[0] == int(nfev), (name, meth, r)
        assert abs(r[2] - obj) <= 1e-8 * obj + 1e-18, (name, meth, r, obj)
        assert r[3] == int(np.count_nonzero(mask)), (name, meth, r)
        checked += 1
    text = open(out_path).read()
    assert "Bounded problems" in text and "Unbounded problems" in text
    assert "g norm" in text
    assert unsupported == 0
    return dict(checked=checked, unsupported=unsupported, waived=waived,
                instances=len({n for n, _, _ in rows}))


# --------------------------------------------- device-side compaction ABI --

def check_compact_batched(lib, dev, seed=9):
    """blsq_compact_batched against NumPy: survivors keep their order, ids and
    trial points move together; with and without an input index list and Xjac,
    sizes around the block boundaries of the kernel."""
    rng = np.random.default_rng(seed)
    for A, n, with_idx, with_j in ((1, 3, False, False), (1023, 4, False, True),
                                   (1024, 4, True, False), (1025, 6, True, True),
                                   (40000, 2, True, True), (5000, 8, False, False)):
        Btot = A * 2 if with_idx else A
        status = np.where(rng.random(Btot) < 0.6, -1, 2).astype(np.int32)
        istate = np.zeros((Btot, 8), np.int32)
        istate[:, 0] = status
        idx = np.sort(rng.choice(Btot, A, replace=False)).astype(np.int32) if with_idx else None
        X = rng.standard_normal((A, n))
        Xj = rng.standard_normal((A, n)) if with_j else None
        ti = torch.as_tensor(istate, device=dev)
        tx, tj = T(X, dev), (T(Xj, dev) if with_j else None)
        tidx = torch.as_tensor(idx, device=dev) if with_idx else None
        o32 = torch.full((A,), -7, dtype=torch.int32, device=dev)
        o64 = torch.full((A,), -7, dtype=torch.int64, device=dev)
        ox = torch.zeros((A, n), dtype=torch.float64, device=dev)
        oj = torch.zeros((A, n), dtype=torch.float64, device=dev) if with_j else None
        work = torch.empty(int(lib._dll.blsq_compact_work_size(A)), dtype=torch.int32,
                           device=dev)
        lib.call("blsq_compact_batched", A, None if tidx is None else tidx.data_ptr(),
                 ti.data_ptr(), n, tx.data_ptr(), None if tj is None else tj.data_ptr(),
                 o32.data_ptr(), o64.data_ptr(), ox.data_ptr(),
                 None if oj is None else oj.data_ptr(), work.data_ptr(), lib.stream(tx))
        pid = idx.astype(np.int64) if with_idx else np.arange(A)
        keep = status[pid] == -1
        k = int(keep.sum())
        assert np.array_equal(o32.cpu().numpy()[:k], pid[keep].astype(np.int32)), (A, n)
        assert np.array_equal(o64.cpu().numpy()[:k], pid[keep]), (A, n)
        assert bits(ox.cpu().numpy()[:k], X[keep]), (A, n)
        if with_j:
            assert bits(oj.cpu().numpy()[:k], Xj[keep]), (A, n)
        assert (o32.cpu().numpy()[k:] == -7).all()


# ------------------------------------- random small problems vs the oracle --

def check_random_small_vs_oracle(lib, dev, B=20, seed=42):
    """Random bounded nonlinear problems for every n = 1..8, both methods,
    fixed and 'jac' scaling, with bounds that are active at many solutions:
    the batched path against the oracle.  Gates: every solution feasible and
    its cost within the north-star 1e-8; status, nfev, x (1e-8) and the active
    set identical for >= 99 % (the rest are evaluations where two termination
    tests are met within an ulp of each other, SURVEY 7 hard part 1)."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    total = exact = 0
    for n in range(1, 9):
        for method in ("trf", "dogbox"):
            for scaling in (1.0, "jac"):
                m = int(rng.integers(n, 3 * n + 6))
                A = rng.standard_normal((m, n))
                Bm = rng.standard_normal((m, n)) * 0.5
                xt = rng.uniform(-1, 1, (B, n))

                def model(x):
                    return A @ x + 0.3 * np.sin(Bm @ x)
                y = np.array([model(xt[b]) for b in range(B)]) + \
                    0.01 * rng.standard_normal((B, m))
                lb, ub, x0 = np.full(n, -0.6), np.full(n, 0.7), np.zeros(n)
                At, Bt = T(A, dev), T(Bm, dev)

                def fun_t(X, Y):
                    return X @ At.T + 0.3 * torch.sin(X @ Bt.T) - Y

                def jac_t(X, Y):
                    return At[None] + 0.3 * torch.cos(X @ Bt.T)[:, :, None] * Bt[None]
                res = least_squares_batched(
                    fun_t, T(np.tile(x0, (B, 1)), dev), jac=jac_t,
                    bounds=(T(lb, dev), T(ub, dev)), method=method, scaling=scaling,
                    args=(PerProblem(T(y, dev)),), _lib=lib)
                X = res.x.cpu().numpy()
                assert np.all(X >= lb) and np.all(X <= ub)
                st, nf = res.status.cpu().numpy(), res.nfev.cpu().numpy()
                ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
                for b in range(B):
                    r = orc.least_squares(
                        lambda x, yb: model(x) - yb, x0,
                        jac=lambda x, yb: A + 0.3 * np.cos(Bm @ x)[:, None] * Bm,
                        bounds=(lb, ub), method=method, scaling=scaling, args=(y[b],))
                    total += 1
                    assert abs(ob[b] - r.obj_value) <= 1e-8 * r.obj_value + 1e-18, \
                        (n, method, scaling, b)
                    exact += (st[b] == r.status and nf[b] == r.nfev and
                              np.allclose(X[b], r.x, rtol=1e-8, atol=1e-9) and
                              np.array_equal(mk[b], np.asarray(r.active_mask)))
    assert exact >= 0.99 * total, (exact, total)
    return dict(total=total, exact=exact)


def check_random_tall_vs_oracle(lib, dev, seed=7):
    """Tall mode (n > 8, odd and even) on random bounded nonlinear problems
    against the oracle: status, counters, active set equal, x / cost 1e-8."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(seed)
    out = {}
    for n in (9, 13, 20, 33):
        for method in ("trf", "dogbox"):
            m = int(rng.integers(3 * n, 6 * n))
            A = rng.standard_normal((m, n))
            Bm = rng.standard_normal((m, n)) * 0.3
            xt = rng.uniform(-1, 1, n)

            def model(x):
                return A @ x + 0.3 * np.sin(Bm @ x)
            y = model(xt) + 0.01 * rng.standard_normal(m)
            lb, ub, x0 = np.full(n, -0.6), np.full(n, 0.7), np.full(n, 0.05)
            At, Bt, yt = T(A, dev), T(Bm, dev), T(y, dev)
            ref = orc.least_squares(lambda x: model(x) - y, x0,
                                    jac=lambda x: A + 0.3 * np.cos(Bm @ x)[:, None] * Bm,
                                    bounds=(lb, ub), method=method)
            res = least_squares(lambda x: At @ x + 0.3 * torch.sin(Bt @ x) - yt, T(x0, dev),
                                jac=lambda x: At + 0.3 * torch.cos(Bt @ x)[:, None] * Bt,
                                bounds=(T(lb, dev), T(ub, dev)), method=method, _lib=lib)
            x = res.x.cpu().numpy()
            key = (n, method)
            out[key] = (res.status, res.nfev, int(np.count_nonzero(ref.active_mask)))
            assert res.status == ref.status and res.nfev == ref.nfev, (key, res.nfev, ref.nfev)
            assert np.allclose(x, ref.x, rtol=1e-8, atol=1e-9), key
            assert abs(res.obj_value - ref.obj_value) <= 1e-8 * ref.obj_value, key
            assert bits(res.active_mask.cpu().numpy(),
                        np.asarray(ref.active_mask, dtype=np.int64)), key
    return out


# ------------------------- edge cases the reference's loops have (SURVEY 5) --

def check_edge_cases_vs_oracle(lib, dev):
    """m < n (trust_region.py:108-112: full_rank = False, the LM iteration
    starts from alpha_lower = 0), NaN residuals at a trial point (trf.py:283,
    314-331 / dogbox.py:202: `NaN <= 0` is False, nothing is accepted, Delta is
    untouched, the loop spins to max_nfev -> status 0) and an exactly rank
    deficient Jacobian (duplicate columns), batched and tall, both methods,
    against the oracle."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(11)
    out = {}
    # ---- m < n, batched (n <= 8) ----
    for n, m in ((4, 2), (6, 3), (3, 1), (8, 5)):
        B = 12
        A = rng.standard_normal((m, n))
        Bm = rng.standard_normal((m, n)) * 0.5
        y = rng.standard_normal((B, m))
        lb, ub, x0 = np.full(n, -0.6), np.full(n, 0.7), np.zeros(n)
        At, Bt = T(A, dev), T(Bm, dev)
        for method in ("trf", "dogbox"):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                res = least_squares_batched(
                    lambda X, Y: X @ At.T + 0.3 * torch.sin(X @ Bt.T) - Y,
                    T(np.tile(x0, (B, 1)), dev),
                    jac=lambda X, Y: At[None] + 0.3 * torch.cos(X @ Bt.T)[:, :, None] * Bt[None],
                    bounds=(T(lb, dev), T(ub, dev)), method=method,
                    args=(PerProblem(T(y, dev)),), _lib=lib)
            ok = 0
            st = res.status.cpu().numpy()
            for b in range(B):
                try:
                    r = orc.least_squares(
                        lambda x, yb: A @ x + 0.3 * np.sin(Bm @ x) - yb, x0,
                        jac=lambda x, yb: A + 0.3 * np.cos(Bm @ x)[:, None] * Bm,
                        bounds=(lb, ub), method=method, args=(y[b],))
                except ValueError as e:
                    # trust_region.py:28-35: with m < n the LM step may end up
                    # to 1 % outside Delta, which the reflective branch rejects
                    # with ValueError -- per-problem status -102 in a batch
                    assert "not within the trust region" in str(e)
                    ok += st[b] == -102
                    continue
                X = res.x[b].cpu().numpy()
                assert np.all(X >= lb) and np.all(X <= ub)
                # the cost is what an underdetermined fit defines; x moves along
                # the null space with the rounding of the rank-deficient SVD
                # (slowly converging underdetermined fits accumulate the noise
                # of the null directions: 1e-6, measured 4e-8)
                if st[b] >= 0:
                    assert abs(float(res.obj_value[b]) - r.obj_value) <= \
                        1e-6 * r.obj_value + 1e-18, (n, m, method, b)
                ok += (int(st[b]) == r.status and int(res.nfev[b]) == r.nfev)
            out[("m<n", n, m, method)] = (ok, B)
            assert ok >= B - 2, (n, m, method, ok)
    # ---- NaN residual at the first trial point: spin to max_nfev ----
    for method in ("trf", "dogbox"):
        fun_np = lambda x: np.array([10.0 * (x[0] - 3.0), np.sqrt(2.0 - x[0])])      # noqa: E731
        jac_np = lambda x: np.array([[10.0], [-0.5 / np.sqrt(2.0 - x[0])]])          # noqa: E731
        with np.errstate(invalid="ignore"):
            r = orc.least_squares(fun_np, np.array([0.0]), jac=jac_np, method=method,
                                  max_nfev=17)
        res = least_squares(
            lambda x: torch.stack([10.0 * (x[0] - 3.0), torch.sqrt(2.0 - x[0])]),
            T([0.0], dev),
            jac=lambda x: torch.stack([torch.full_like(x[0], 10.0),
                                       -0.5 / torch.sqrt(2.0 - x[0])]).reshape(2, 1),
            method=method, max_nfev=17, _lib=lib)
        out[("nan", method)] = (res.status, res.nfev, r.status, r.nfev)
        assert r.status == 0 and r.nfev == 17, (r.status, r.nfev)
        assert res.status == r.status and res.nfev == r.nfev and res.njev == r.njev
        assert bits(res.x.cpu().numpy(), r.x), (res.x, r.x)
        assert res.success is False or res.success == False       # noqa: E712
    # ---- exactly rank-deficient Jacobian (duplicate columns), n = 3 ----
    A = np.array([[1.0, 1, 0], [2, 2, 1], [3, 3, 0], [4, 4, 2]])
    yv = np.array([1.0, 2.0, -1.0, 0.5])
    At, yt = T(A, dev), T(yv, dev)
    for method in ("trf", "dogbox"):
        r = orc.least_squares(lambda x: A @ x - yv, np.zeros(3), jac=lambda x: A,
                              method=method)
        res = least_squares(lambda x: At @ x - yt, T(np.zeros(3), dev),
                            jac=lambda x: At, method=method, _lib=lib)
        out[("rankdef", method)] = (res.status, res.nfev, r.status, r.nfev,
                                    res.obj_value, r.obj_value)
        assert res.status == r.status and res.nfev == r.nfev, out[("rankdef", method)]
        assert abs(res.obj_value - r.obj_value) <= 1e-8 * r.obj_value
    return out


def check_tall_edge_cases_vs_oracle(lib, dev):
    """The same edge cases through the tall kernels (n > 8): m < n, NaN
    residuals, and the kappa sweep: full-rank Jacobians with cond(J) = 1e6 ...
    1e12.  The reference's SVD (trf.py:272) and min-norm lstsq (dogbox.py:197)
    never fail on those; the shifted CholeskyQR3 of tall mode must not either,
    and TRF must reproduce status, nfev, the active set and the cost (1e-8; x
    to 10 kappa eps: J's own rounding is all that x is defined to -- measured
    1e-11 ... 3e-6 at kappa = 1e10).
    Dogbox on this family is ulp-chaotic IN THE REFERENCE (hundreds of
    iterations along an ill-conditioned valley: 1-ulp noise on f changes its
    nfev 318 -> 324 / 969 at kappa = 1e6 and x by 16 %), so for dogbox the
    gates are: no failure, feasible, and a cost no worse than the reference's
    by more than its own self-sensitivity; at kappa = 1e6 the reference
    ends with status 2 after 976 evaluations, with status 0 (budget of
    2400 exhausted, at a 6 - 7 % LOWER cost) in 13 of 16 runs with 1-ulp noise
    on f, and with status 2 after 195 - 306 evaluations at an 8 - 12 % HIGHER
    cost in 11 of 40 runs with 1-ulp noise on f and J
    (tests/golden/kappa_dogbox_sensitivity.json)."""
    from oracle import blsq_oracle as orc
    rng = np.random.default_rng(12)
    out = {}
    # ---- m < n ----
    n, m = 12, 7
    A = rng.standard_normal((m, n))
    Bm = rng.standard_normal((m, n)) * 0.3
    y = rng.standard_normal(m)
    lb, ub, x0 = np.full(n, -0.6), np.full(n, 0.7), np.full(n, 0.05)
    At, Bt, yt = T(A, dev), T(Bm, dev), T(y, dev)
    for method in ("trf", "dogbox"):
        def solve_ours():
            return least_squares(
                lambda x: At @ x + 0.3 * torch.sin(Bt @ x) - yt, T(x0, dev),
                jac=lambda x: At + 0.3 * torch.cos(Bt @ x)[:, None] * Bt,
                bounds=(T(lb, dev), T(ub, dev)), method=method, _lib=lib)
        try:
            r = orc.least_squares(lambda x: A @ x + 0.3 * np.sin(Bm @ x) - y, x0,
                                  jac=lambda x: A + 0.3 * np.cos(Bm @ x)[:, None] * Bm,
                                  bounds=(lb, ub), method=method)
        except ValueError as e:
            # trust_region.py:28-35 (see check_edge_cases_vs_oracle): the same
            # exception must come out of the tall driver
            try:
                solve_ours()
                raise AssertionError("reference raises %r, tall mode did not" % (e,))
            except ValueError as e2:
                assert str(e2) == str(e), (e, e2)
            out[("m<n", method)] = "ValueError: " + str(e)
            continue
        res = solve_ours()
        out[("m<n", method)] = (res.status, res.nfev, r.status, r.nfev,
                                res.obj_value, r.obj_value)
        X = res.x.cpu().numpy()
        assert np.all(X >= lb) and np.all(X <= ub)
        assert res.status > 0 and r.status > 0
        assert res.obj_value <= r.obj_value * (1 + 1e-6) + 1e-12, out[("m<n", method)]
    # ---- NaN residuals at the first trial ----
    n, m = 10, 30
    A = rng.standard_normal((m, n))
    yv = A @ np.full(n, 3.0)
    At, yt = T(A, dev), T(yv, dev)
    for method in ("trf", "dogbox"):
        with np.errstate(invalid="ignore"):
            r = orc.least_squares(
                lambda x: np.concatenate([A @ x - yv, [np.sqrt(2.0 - x[0])]]), np.zeros(n),
                jac=lambda x: np.vstack([A, np.r_[-0.5 / np.sqrt(2.0 - x[0]), np.zeros(n - 1)]]),
                method=method, max_nfev=9)

        def jac_t(x):
            last = torch.zeros(1, n, dtype=torch.float64, device=x.device)
            last[0, 0] = -0.5 / torch.sqrt(2.0 - x[0])
            return torch.cat([At, last], 0)
        res = least_squares(
            lambda x: torch.cat([At @ x - yt, torch.sqrt(2.0 - x[0]).reshape(1)]),
            T(np.zeros(n), dev), jac=jac_t, method=method, max_nfev=9, _lib=lib)
        out[("nan", method)] = (res.status, res.nfev, r.status, r.nfev)
        assert r.status == 0 and r.nfev == 9
        assert res.status == 0 and res.nfev == 9 and res.njev == r.njev
        assert np.allclose(res.x.cpu().numpy(), r.x, rtol=1e-8, atol=0)
        assert abs(res.obj_value - r.obj_value) <= 1e-8 * r.obj_value
    # ---- kappa sweep ----
    with open(os.path.join(GOLDEN, "kappa_dogbox_sensitivity.json")) as fh:
        sens = json.load(fh)
    m, n = 3000, 24
    for kappa in (1e6, 1e8, 1e10, 1e12):
        U, _ = np.linalg.qr(rng.standard_normal((m, n)))
        V, _ = np.linalg.qr(rng.standard_normal((n, n)))
        A = (U * np.logspace(0, -np.log10(kappa), n)) @ V.T
        xt = rng.uniform(-1, 1, n)
        y = A @ xt + 0.1 * np.sin(A @ xt) + 1e-3 * rng.standard_normal(m)
        lb, ub, x0 = np.full(n, -0.6), np.full(n, 0.7), np.full(n, 0.05)
        At, yt = T(A, dev), T(y, dev)
        for method in ("trf", "dogbox"):
            r = orc.least_squares(lambda x: A @ x + 0.1 * np.sin(A @ x) - y, x0,
                                  jac=lambda x: (1 + 0.1 * np.cos(A @ x))[:, None] * A,
                                  bounds=(lb, ub), method=method)
            res = least_squares(lambda x: At @ x + 0.1 * torch.sin(At @ x) - yt, T(x0, dev),
                                jac=lambda x: (1 + 0.1 * torch.cos(At @ x))[:, None] * At,
                                bounds=(T(lb, dev), T(ub, dev)), method=method, _lib=lib)
            X = res.x.cpu().numpy()
            s = dict(status=(res.status, r.status), nfev=(res.nfev, r.nfev),
                     x_rel=float(np.abs(X - r.x).max() / np.abs(r.x).max()),
                     obj_rel=abs(res.obj_value - r.obj_value) / r.obj_value,
                     mask_eq=bits(res.active_mask.cpu().numpy(),
                                  np.asarray(r.active_mask, dtype=np.int64)))
            out[(kappa, method)] = s
            assert np.all(X >= lb) and np.all(X <= ub)
            if method == "trf":
                assert s["status"][0] == s["status"][1] and s["nfev"][0] == s["nfev"][1], s
                assert s["mask_eq"] and s["obj_rel"] < 1e-8, (kappa, s)
                assert s["x_rel"] < max(1e-8, 10 * kappa * 2.2e-16), (kappa, s)
            else:
                assert res.status >= 0, (kappa, s)
                # kappa = 1e6: the worst of 56 runs of the reference algorithm
                # itself under 1-ulp noise (tests/golden/kappa_dogbox_sensitivity.py:
                # cost 0.93 ... 1.116 of the unperturbed run, 195 ... 2400
                # evaluations) with a 10 % margin; elsewhere 1 %
                gate = 1.1 * sens["cost_ratio_max"] if kappa == 1e6 else 1.01
                assert sens["unperturbed"]["nfev"] == 976 or kappa != 1e6
                assert res.obj_value <= r.obj_value * gate, (kappa, s)
    return out


def check_x_covariance(lib, dev):
    """options={'x_covariance': True}: (J^T J)^-1 at the solution (the meaning
    least_squares.py:248-252 documents) from the factor the solve holds,
    batched / single / tall; the default stays None as in the reference
    (trf.py:261,358)."""
    from bounded_lsq_b200.synthetic import TallLinExp
    model = ExpDecay2()
    B = 16
    _, y = model.make_data(B, seed=1)
    for method in ("trf", "dogbox"):
        r = least_squares_batched(model.fun_t, T(np.tile(model.x0, (B, 1)), dev),
                                  jac=model.jac_t, bounds=(model.lb, model.ub),
                                  method=method, args=(PerProblem(T(y, dev)),),
                                  options=dict(x_covariance=True), _lib=lib)
        X = r.x.cpu().numpy()
        C = r.x_covariance.cpu().numpy()
        for b in range(B):
            J = model.jac_np(X[b])
            if np.linalg.cond(J) > 1e4:
                continue                  # inv(J^T J) itself is not defined to 1e-7
            Rq = np.linalg.qr(J, mode="r")
            Ti = np.linalg.inv(Rq)
            ref = Ti @ Ti.T
            assert np.abs(C[b] - ref).max() <= 1e-8 * np.abs(ref).max(), (method, b)
    wl = TallLinExp(3000, 12, seed=1, x0_tail=(0.8, 1.5, 0.3, 4.0)).to_device(dev)
    rr = least_squares(wl.fun_t, T(wl.x0, dev), jac=wl.jac_t,
                       bounds=(T(wl.lb, dev), T(wl.ub, dev)),
                       options=dict(x_covariance=True), _lib=lib)
    J = wl.jac_np(rr.x.cpu().numpy())
    ref = np.linalg.inv(J.T @ J)
    assert np.abs(rr.x_covariance.cpu().numpy() - ref).max() <= 1e-8 * np.abs(ref).max()
    r1 = least_squares(lambda x: x - 1.0, T([3.0], dev), options=dict(x_covariance=True), _lib=lib)
    assert r1.x_covariance.shape == (1, 1) and float(r1.x_covariance[0, 0]) == 1.0
    assert least_squares(lambda x: x - 1.0, T([3.0], dev), _lib=lib).x_covariance is None
    # singular J^T J ("the inverse doesn't exist") -> None
    A = T(np.array([[1.0, 1.0], [2.0, 2.0], [3.0, 3.0]]), dev)
    r2 = least_squares(lambda x: A @ x - 1.0, T([0.0, 0.0], dev), jac=lambda x: A,
                       options=dict(x_covariance=True), _lib=lib)
    assert r2.x_covariance is None


def check_mode_routing(lib, dev):
    """A single problem with n <= 8 runs on the batched kernels unless it is
    tall: from least_squares.TALL_FROM_ROWS residuals on it goes to the tall
    kernels (n >= 2), as does options={'mode': 'tall'}; both routes agree with
    the oracle (status, nfev, active set; x and cost to 1e-8)."""
    from oracle import blsq_oracle as orc
    import importlib
    ls_mod = importlib.import_module("bounded_lsq_b200.least_squares")
    rng = np.random.default_rng(5)
    n = 4
    out = {}
    for m, jac_kind in ((ls_mod.TALL_FROM_ROWS + 37, "exact"), (600, "exact"),
                        (ls_mod.TALL_FROM_ROWS, "2-point")):
        t = np.linspace(0.0, 4.0, m)
        truth = np.array([2.0, 0.9, 1.2, 3.0])
        y = truth[0] * np.exp(-truth[1] * t) + truth[2] * np.exp(-truth[3] * t) \
            + 0.01 * rng.standard_normal(m)
        lb = np.array([0.0, 0.0, 0.0, 0.0])
        ub = np.array([10.0, 1.0, 1.1, 10.0])        # the third bound ends up active
        x0 = np.array([1.0, 0.5, 0.5, 2.0])
        tt, yt = T(t, dev), T(y, dev)
        calls = [0]

        def fun_t(x):
            calls[0] += 1
            return x[0] * torch.exp(-x[1] * tt) + x[2] * torch.exp(-x[3] * tt) - yt

        def jac_t(x):
            e1, e2 = torch.exp(-x[1] * tt), torch.exp(-x[3] * tt)
            return torch.stack([e1, -x[0] * tt * e1, e2, -x[2] * tt * e2], dim=1)

        def fun_n(x):
            return x[0] * np.exp(-x[1] * t) + x[2] * np.exp(-x[3] * t) - y

        def jac_n(x):
            e1, e2 = np.exp(-x[1] * t), np.exp(-x[3] * t)
            return np.stack([e1, -x[0] * t * e1, e2, -x[2] * t * e2], axis=1)
        for method in ("trf", "dogbox"):
            ref = orc.least_squares(fun_n, x0, jac=jac_n if jac_kind == "exact" else "2-point",
                                    bounds=(lb, ub), method=method)
            kw = dict(jac=jac_t if jac_kind == "exact" else "2-point",
                      bounds=(T(lb, dev), T(ub, dev)), method=method, _lib=lib)
            routes = {}
            for mode in (None, "batched", "tall"):
                if mode == "batched" and m > 4096:
                    continue                           # the slow route this replaces
                calls[0] = 0
                res = least_squares(fun_t, T(x0, dev), options=dict(mode=mode) if mode else {},
                                    **kw)
                routes[mode] = (res, calls[0])
                x = res.x.cpu().numpy()
                tol = 1e-8 if jac_kind == "exact" else 1e-6
                assert res.status == ref.status, (m, method, mode, res.status, ref.status)
                if jac_kind == "exact":
                    assert res.nfev == ref.nfev and res.njev == ref.njev, (m, method, mode)
                assert np.array_equal(res.active_mask.cpu().numpy(), ref.active_mask)
                assert np.abs(x - ref.x).max() <= tol * np.abs(ref.x).max(), (m, method, mode)
                assert abs(res.obj_value - ref.obj_value) <= tol * ref.obj_value
            # the automatic route is the tall one exactly when m is tall, and
            # costs one residual evaluation more than asking for it
            auto, tall = routes[None], routes["tall"]
            if m >= ls_mod.TALL_FROM_ROWS:
                assert bits(auto[0].x.cpu().numpy(), tall[0].x.cpu().numpy())
                assert auto[1] == tall[1] + 1, (auto[1], tall[1])
            else:
                assert bits(auto[0].x.cpu().numpy(), routes["batched"][0].x.cpu().numpy())
                assert auto[1] == routes["batched"][1]
            out[(m, jac_kind, method)] = (auto[0].status, auto[0].nfev)
    with pytest.raises(ValueError):
        least_squares(fun_t, T(x0, dev), options=dict(mode="wide"), _lib=lib)
    return out


def check_chunked_batch(lib, dev):
    """options={'chunk': K}: the batch solved K problems at a time gives the bits
    of the one-piece solve (per-problem arithmetic does not depend on the
    batch), with shared and with per-problem bounds, for device and (on the
    GPU) pinned host inputs."""
    model = ExpDecay2()
    B = 2500
    _, y = model.make_data(B, seed=33)
    X0 = np.tile(model.x0, (B, 1))
    lbB = np.tile(model.lb, (B, 1))
    ubB = np.tile(model.ub, (B, 1))
    ubB[::3, 2] = 1.2                                 # a per-problem bound that binds
    for method, jac in (("trf", model.jac_t), ("dogbox", "2-point")):
        for bounds in ((model.lb, model.ub), (T(lbB, dev), T(ubB, dev))):
            kw = dict(jac=jac, bounds=bounds, method=method, _lib=lib)
            one = least_squares_batched(model.fun_t, T(X0, dev), args=(PerProblem(T(y, dev)),), **kw)
            variants = [least_squares_batched(model.fun_t, T(X0, dev),
                                              args=(PerProblem(T(y, dev)),),
                                              options=dict(chunk=700), **kw)]
            if dev.type == "cuda":
                variants.append(least_squares_batched(
                    model.fun_t, torch.from_numpy(X0).pin_memory(),
                    args=(PerProblem(torch.from_numpy(y).pin_memory()),),
                    options=dict(chunk=1000, h2d_chunks=2, device=dev), **kw))
            for r in variants:
                assert r.x.shape == (B, model.n) and r.fun.shape == one.fun.shape
                for fld in ("x", "obj_value", "optimality", "status", "nfev", "njev",
                            "active_mask", "fun", "success"):
                    assert bits(r[fld].cpu().numpy(), one[fld].cpu().numpy()), (method, fld)
                assert r.rounds >= one.rounds
