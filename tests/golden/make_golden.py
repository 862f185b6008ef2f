"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

Run in the authoring container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference (nmayorov/bounded-lsq) is imported from /root/reference without
edits.  Under NumPy >= 2 its ``scaling == 'jac'`` test fails for ndarray
``scaling`` (trf.py:216,239; dogbox.py:141,165), so the public ``trf`` /
``dogbox`` entry points are called directly (least_squares.py:373-379 does the
same) with ``scaling`` an ndarray subclass whose ``== str`` is False -- exactly
what NumPy 1.9 returned.  Nothing else is touched.

While generating, every reference output is compared BIT-FOR-BIT with the
oracle (oracle/blsq_oracle.py) on this host; the outcome is stored in each
file's ``meta`` so tests and DESIGN.md can cite it.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, "/root/reference")

import importlib                           # noqa: E402
import bounded_lsq                         # noqa: E402,F401  (reference)
# the package __init__ rebinds `trf`/`dogbox` to functions; fetch the modules
rb = importlib.import_module("bounded_lsq.bounds")
rd = sys.modules["bounded_lsq.dogbox"]
rt = sys.modules["bounded_lsq.trf"]
rtr = importlib.import_module("bounded_lsq.trust_region")
from scipy.optimize._numdiff import approx_derivative  # noqa: E402

import packed_npz                          # noqa: E402
from oracle import blsq_oracle as orc      # noqa: E402
from problems import corpus                # noqa: E402
from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak, RatPoly5, TallLinExp  # noqa: E402

SQ = np.finfo(float).eps ** 0.5


class _Scal(np.ndarray):
    """ndarray whose comparison with a str is False (NumPy 1.9 semantics)."""

    def __eq__(self, other):
        if isinstance(other, str):
            return False
        return np.ndarray.__eq__(self, other)


def ref_solve(method, fun, jac, x0, lb, ub, scaling=None, ftol=SQ, xtol=SQ,
              gtol=SQ, max_nfev=None, fd=None, diff_step=None):
    """Run the reference trf/dogbox; record every trial point."""
    trials = []
    first = [True]

    def fun_w(x):
        if first[0]:
            first[0] = False
        else:
            trials.append(x.copy())
        return np.atleast_1d(fun(x))

    if fd is None:
        def jac_w(x, f):
            return np.atleast_2d(jac(x))
    else:
        def jac_w(x, f):
            return np.atleast_2d(approx_derivative(
                fun, x, rel_step=diff_step, method=fd, f0=f, bounds=(lb, ub)))

    if isinstance(scaling, str):
        sc = scaling          # 'jac': the str comparison works unmodified
    else:
        sc = (np.ones_like(x0) if scaling is None
              else np.asarray(scaling, float)).view(_Scal)
    solver = rt.trf if method == 'trf' else rd.dogbox
    res = solver(fun_w, jac_w, x0.copy(), lb, ub, ftol, xtol, gtol, max_nfev,
                 sc)
    return res, trials


def orc_solve(method, fun, jac, x0, lb, ub, scaling=None, ftol=SQ, xtol=SQ,
              gtol=SQ, max_nfev=None, fd=None, diff_step=None):
    trials = []
    first = [True]

    def fun_w(x):
        if first[0]:
            first[0] = False
        else:
            trials.append(x.copy())
        return np.atleast_1d(fun(x))

    if fd is None:
        def jac_w(x, f):
            return np.atleast_2d(jac(x))
    else:
        def jac_w(x, f):
            return np.atleast_2d(orc.fd_jacobian(fun, x, f, lb, ub, diff_step,
                                                 fd))
    sc = scaling if isinstance(scaling, str) else (
        np.ones_like(x0) if scaling is None else np.asarray(scaling, float))
    solver = orc.trf if method == 'trf' else orc.dogbox
    res = solver(fun_w, jac_w, x0.copy(), lb, ub, ftol, xtol, gtol, max_nfev,
                 sc)
    return res, trials


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def results_bitwise(r1, t1, r2, t2):
    ok = (r1.status == r2.status and r1.nfev == r2.nfev and
          r1.njev == r2.njev and same_bits(r1.x, r2.x) and
          same_bits(np.float64(r1.obj_value), np.float64(r2.obj_value)) and
          same_bits(np.asarray(r1.active_mask), np.asarray(r2.active_mask)) and
          len(t1) == len(t2) and all(same_bits(a, b) for a, b in zip(t1, t2)))
    return bool(ok)


def pack_result(res, trials, n, kmax):
    """Fixed-size record: first kmax trial points padded with NaN."""
    tp = np.full((kmax, n), np.nan)
    k = min(kmax, len(trials))
    if k:
        tp[:k] = np.array(trials[:k])
    return dict(x=np.asarray(res.x, float), obj=float(res.obj_value),
                status=int(res.status), nfev=int(res.nfev),
                njev=int(res.njev),
                mask=np.asarray(res.active_mask, dtype=np.int64),
                optimality=float(res.optimality), trials=tp,
                ntrials=len(trials))


# ------------------------------------------------------------------------
def gen_helpers(rng):
    """Elementwise bound passes (SURVEY 8a rows a15, a19-a23) + FD steps."""
    out = {}
    cases = []
    for n in (1, 2, 3, 4, 6, 8, 16, 64, 257):
        for rep in range(12):
            lb = rng.uniform(-3, 0, n)
            ub = lb + rng.uniform(0.1, 4, n)
            # infinities, some shared
            lb[rng.random(n) < 0.2] = -np.inf
            ub[rng.random(n) < 0.2] = np.inf
            fin_l, fin_u = np.isfinite(lb), np.isfinite(ub)
            x = np.where(fin_l & fin_u, lb + rng.random(n) * (ub - lb),
                         np.where(fin_l, lb + rng.random(n) * 3,
                                  np.where(fin_u, ub - rng.random(n) * 3,
                                           rng.standard_normal(n))))
            # put some coordinates exactly on / next to / past bounds
            k = rng.random(n)
            x = np.where((k < 0.1) & fin_l, lb, x)
            x = np.where((k > 0.9) & fin_u, ub, x)
            x = np.where((k > 0.1) & (k < 0.15) & fin_l,
                         np.nextafter(lb, np.inf), x)
            x = np.where((k > 0.85) & (k < 0.9) & fin_u,
                         np.nextafter(ub, -np.inf), x)
            d = rng.standard_normal(n)
            d[rng.random(n) < 0.15] = 0.0
            if rep % 3 == 0 and n > 1:      # force ties in the ratio test
                d[1] = d[0]
                x[1], lb[1], ub[1] = x[0], lb[0], ub[0]
            g = rng.standard_normal(n)
            g[rng.random(n) < 0.1] = 0.0
            tr = np.abs(rng.standard_normal(n)) + 0.01
            if rep % 4 == 0:                # trust-region bound == real bound
                j = rng.integers(n)
                if np.isfinite(ub[j]):
                    tr[j] = ub[j] - x[j]
            cases.append((x, d, g, tr, lb, ub))
    for i, (x, d, g, tr, lb, ub) in enumerate(cases):
        step, hits = rb.step_size_to_bound(x, d, lb, ub)
        o_step, o_hits = orc.step_size_to_bound(x, d, lb, ub)
        assert same_bits(step, o_step) and same_bits(hits, o_hits)
        act = rb.find_active_constraints(x, lb, ub, rtol=1e-3)
        assert same_bits(act, orc.find_active_constraints(x, lb, ub, 1e-3))
        act2 = rb.find_active_constraints(x, lb, ub, rtol=SQ)
        # strictly-feasible wants in-bounds input; clip first like callers do
        xc = np.clip(x, lb, ub)
        msf0 = rb.make_strictly_feasible(xc, lb, ub, rstep=0)
        msf1 = rb.make_strictly_feasible(xc, lb, ub, rstep=1e-10)
        assert same_bits(msf0, orc.make_strictly_feasible(xc, lb, ub, 0))
        assert same_bits(msf1, orc.make_strictly_feasible(xc, lb, ub, 1e-10))
        v, jv = rb.scaling_vector(xc, g, lb, ub)
        ov, ojv = orc.scaling_vector(xc, g, lb, ub)
        assert same_bits(v, ov) and same_bits(jv, ojv)
        inb = rb.in_bounds(x, lb, ub)
        assert bool(inb) == orc.in_bounds(x, lb, ub)
        fi = rd.find_intersection(xc, tr, lb, ub)
        ofi = orc.find_intersection(xc, tr, lb, ub)
        assert all(same_bits(a, b) for a, b in zip(fi, ofi))
        # FD steps via scipy internals (third-party arithmetic, restated)
        from scipy.optimize import _numdiff as nd
        h0 = nd._compute_absolute_step(None, xc, np.zeros(1), '2-point')
        h2, _ = nd._adjust_scheme_to_bounds(xc, h0, 1, '1-sided', lb, ub)
        oh2, _ = orc.fd_steps(xc, lb, ub, None, '2-point')
        assert same_bits(h2, oh2)
        hr = nd._compute_absolute_step(1e-2, xc, np.zeros(1), '2-point')
        hr2, _ = nd._adjust_scheme_to_bounds(xc, hr, 1, '1-sided', lb, ub)
        ohr2, _ = orc.fd_steps(xc, lb, ub, 1e-2, '2-point')
        assert same_bits(hr2, ohr2)
        h3 = nd._compute_absolute_step(None, xc, np.zeros(1), '3-point')
        h3a, os3 = nd._adjust_scheme_to_bounds(xc, h3, 1, '2-sided', lb, ub)
        oh3, oos3 = orc.fd_steps(xc, lb, ub, None, '3-point')
        assert same_bits(h3a, oh3) and same_bits(os3, oos3)
        p = f"c{i}_"
        out.update({p + "x": x, p + "xc": xc, p + "d": d, p + "g": g,
                    p + "tr": tr, p + "lb": lb, p + "ub": ub,
                    p + "step": np.float64(step), p + "hits": hits,
                    p + "act_1e3": act, p + "act_sq": act2,
                    p + "msf0": msf0, p + "msf1": msf1, p + "v": v,
                    p + "jv": jv, p + "inb": np.bool_(inb),
                    p + "fi_lo": fi[0], p + "fi_hi": fi[1],
                    p + "fi_ol": fi[2], p + "fi_ou": fi[3],
                    p + "fi_tl": fi[4], p + "fi_tu": fi[5],
                    p + "fd2": h2, p + "fd2_rel": hr2, p + "fd3": h3a,
                    p + "fd3_one": os3})
    out["ncases"] = np.int64(len(cases))
    out["meta"] = np.array(json.dumps(dict(
        source="reference bounds.py/dogbox.py + scipy _numdiff",
        oracle_bitwise_equal=True)))
    packed_npz.save(os.path.join(HERE, "helpers.npz"), out)
    print("helpers.npz:", len(cases), "cases; oracle bitwise equal")


def gen_tr_subproblem(rng):
    """solve_lsq_trust_region / intersect / minimize_quadratic / dogleg."""
    out = {}
    k = 0
    bit_ok = True
    for n in (1, 2, 3, 4, 6, 8, 12, 32, 64):
        for rep in range(16):
            m = n + int(rng.integers(0, 40))
            J = rng.standard_normal((m, n)) * np.exp(rng.uniform(-2, 2, n))
            if rep % 5 == 4 and n > 1:          # rank deficient
                J[:, -1] = J[:, 0]
            f = rng.standard_normal(m)
            U, s, Vt = np.linalg.svd(J, full_matrices=False)
            V = Vt.T
            uf = U.T.dot(f)
            gn = np.linalg.norm(V.dot(uf / np.maximum(s, 1e-300)))
            Delta = float(np.exp(rng.uniform(-4, 1))) * (gn if np.isfinite(gn)
                                                        else 1.0)
            a0 = [None, 0.0, float(np.exp(rng.uniform(-6, 2)))][rep % 3]
            p, alpha, nit = rtr.solve_lsq_trust_region(n, m, uf, s, V, Delta,
                                                       initial_alpha=a0)
            op, oalpha, onit = orc.solve_lsq_trust_region(n, m, uf, s, V,
                                                          Delta, a0)
            bit_ok &= same_bits(p, op) and alpha == oalpha and nit == onit
            pre = f"tr{k}_"
            out.update({pre + "uf": uf, pre + "s": s, pre + "V": V,
                        pre + "m": np.int64(m), pre + "Delta": np.float64(Delta),
                        pre + "alpha0": np.float64(np.nan if a0 is None else a0),
                        pre + "p": p, pre + "alpha": np.float64(alpha),
                        pre + "nit": np.int64(nit)})
            k += 1
    out["n_tr"] = np.int64(k)
    # line / sphere intersections
    k = 0
    for n in (1, 2, 4, 8, 33):
        for rep in range(10):
            s = rng.standard_normal(n)
            x = rng.standard_normal(n)
            Delta = np.linalg.norm(x) * (1.0 + rng.random())
            t1, t2 = rtr.intersect_trust_region(x, s, Delta)
            o1, o2 = orc.intersect_trust_region(x, s, Delta)
            bit_ok &= (t1 == o1 and t2 == o2)
            pre = f"it{k}_"
            out.update({pre + "x": x, pre + "s": s,
                        pre + "Delta": np.float64(Delta),
                        pre + "t": np.array([t1, t2])})
            k += 1
    out["n_it"] = np.int64(k)
    # 1-D quadratics
    abl = rng.standard_normal((200, 2))
    abl[::7, 0] = 0.0
    lo = -np.abs(rng.standard_normal(200))
    hi = lo + np.abs(rng.standard_normal(200)) * 2
    mq = np.array([rt.minimize_quadratic(a, b, l, u)
                   for (a, b), l, u in zip(abl, lo, hi)])
    omq = np.array([orc.minimize_quadratic(a, b, l, u)
                    for (a, b), l, u in zip(abl, lo, hi)])
    bit_ok &= same_bits(mq, omq)
    out.update(mq_ab=abl, mq_lo=lo, mq_hi=hi, mq_out=mq)
    # dogleg / constrained Cauchy
    k = 0
    for n in (1, 2, 3, 6, 8, 20):
        for rep in range(20):
            lb = -np.abs(rng.standard_normal(n)) - 0.1
            ub = np.abs(rng.standard_normal(n)) + 0.1
            lb[rng.random(n) < 0.2] = -np.inf
            ub[rng.random(n) < 0.2] = np.inf
            x = np.clip(rng.standard_normal(n) * 0.3, lb, ub)
            newton = rng.standard_normal(n) * np.exp(rng.uniform(-3, 1))
            cauchy = newton * rng.random() + 0.1 * rng.standard_normal(n) * \
                np.exp(rng.uniform(-3, 0))
            tr = np.exp(rng.uniform(-3, 1)) * np.ones(n) * \
                np.exp(rng.uniform(-0.5, 0.5, n))
            st, bh, th = rd.dogleg_step(x, cauchy.copy(), newton, tr, lb, ub)
            ost, obh, oth = orc.dogleg_step(x, cauchy.copy(), newton, tr, lb,
                                            ub)
            bit_ok &= same_bits(st, ost) and same_bits(bh, obh) and \
                bool(th) == bool(oth)
            cs, cb, ct = rd.constrained_cauchy_step(x, cauchy, tr, lb, ub)
            ocs, ocb, oct_ = orc.constrained_cauchy_step(x, cauchy, tr, lb, ub)
            bit_ok &= same_bits(cs, ocs) and same_bits(cb, ocb) and \
                bool(ct) == bool(oct_)
            pre = f"dl{k}_"
            out.update({pre + "x": x, pre + "cauchy": cauchy,
                        pre + "newton": newton, pre + "tr": tr,
                        pre + "lb": lb, pre + "ub": ub, pre + "step": st,
                        pre + "hits": bh, pre + "tr_hit": np.bool_(th),
                        pre + "cstep": cs, pre + "chits": cb,
                        pre + "ctr_hit": np.bool_(ct)})
            k += 1
    out["n_dl"] = np.int64(k)
    assert bit_ok
    out["meta"] = np.array(json.dumps(dict(
        source="reference trust_region.py / trf.py / dogbox.py",
        oracle_bitwise_equal=bool(bit_ok))))
    packed_npz.save(os.path.join(HERE, "tr_subproblem.npz"), out)
    print("tr_subproblem.npz: oracle bitwise equal =", bit_ok)


def check_corpus_against_reference_suite():
    """tests/problems.py restates the 58 instances of the reference's suite
    (benchmarks/lsq_problems.py:1003-1018) from the published formulae; here
    every instance is compared with the reference's own class: same name, x0
    and bounds exactly, fun / jac to rounding at x0 and at a random point.
    The MINPACK-2 data tables are written to problem_data.npz first."""
    sys.path.insert(0, "/root/reference/benchmarks")
    import lsq_problems as ref_suite
    np.savez_compressed(
        os.path.join(HERE, "problem_data.npz"),
        osborne1_y=ref_suite.ExponentialFitting().y,
        osborne2_y=ref_suite.GaussianFittingI().y,
        coating_xi=ref_suite.CoatingThickness().xi,
        coating_y=ref_suite.CoatingThickness().y)
    u, b = ref_suite.extract_lsq_problems()
    ref = dict(u + b)
    mine = {p.name: p for p in corpus()}
    assert set(ref) == set(mine), (set(ref) ^ set(mine))
    rng = np.random.default_rng(0)
    worst = 0.0
    for name, rp in ref.items():
        p = mine[name]
        assert np.array_equal(p.x0, np.asarray(rp.x0, float)), name
        lb = np.full(p.n, -np.inf) if rp.bounds[0] is None else \
            np.broadcast_to(np.asarray(rp.bounds[0], float), (p.n,))
        ub = np.full(p.n, np.inf) if rp.bounds[1] is None else \
            np.broadcast_to(np.asarray(rp.bounds[1], float), (p.n,))
        assert np.array_equal(p.lb, lb) and np.array_equal(p.ub, ub), name
        for x in (p.x0, p.x0 + 0.01 * rng.standard_normal(p.n)):
            f1, f2, j1, j2 = p.fun(x), rp.fun(x), p.jac(x), rp.jac(x)
            ef = np.abs(f1 - f2).max() / max(1.0, np.abs(f2).max())
            ej = np.abs(j1 - j2).max() / max(1.0, np.abs(j2).max())
            worst = max(worst, ef, ej)
            assert ef < 1e-12 and ej < 1e-12, (name, ef, ej)
    print(f"problems.py: {len(ref)} instances = the reference suite "
          f"(x0 / bounds exact, fun / jac within {worst:.1e})")
    return len(u), len(b)


def self_sensitivity(method, p, scaling, base, base_trials, nrep=12):
    """The reference against ITSELF with 1-ulp noise on the residuals
    (f * (1 + 2.2e-16 N(0, 1))): the best agreement any implementation that is
    not bit-identical can be asked for on this run (SURVEY 7, hard part 1).
    Returns [x_rel, obj_rel, runs with another nfev, runs with another status,
    first-step rel].  The first-step figure also takes 6 runs with 8-ulp noise:
    several instances start on an EXACT tie of a branch test (Watson at x0 = 0:
    the Gauss-Newton step is e_2, |p| = Delta = 1 exactly, and
    trust_region.py:116 `norm(p) <= Delta` is decided by the last bits of
    LAPACK's SVD), which a few ulps of a different summation order flip."""
    xr = orr = fs = 0.0
    dn = ds = 0
    for rep in range(nrep + 6):
        g = np.random.default_rng(rep)
        amp = 2.220446049250313e-16 * (1.0 if rep < nrep else 8.0)

        def fun(x):
            f = np.atleast_1d(p.fun(x))
            return f * (1.0 + amp * g.standard_normal(f.shape))
        try:
            r, t = ref_solve(method, fun, p.jac, p.x0, p.lb, p.ub, scaling=scaling)
        except Exception:                                     # noqa: BLE001
            if rep < nrep:
                ds += 1
            continue
        if t and base_trials:
            stepn = max(np.abs(base_trials[0] - p.x0).max(), 1e-300)
            fs = max(fs, float(np.abs(t[0] - base_trials[0]).max() / stepn))
        if rep >= nrep:
            continue
        xr = max(xr, float(np.abs(r.x - base.x).max() /
                           max(np.abs(base.x).max(), 1e-300)))
        orr = max(orr, abs(r.obj_value - base.obj_value) /
                  max(base.obj_value, 1e-300))
        dn += int(r.nfev != base.nfev)
        ds += int(r.status != base.status)
    return np.array([xr, orr, dn, ds, fs], dtype=np.float64)


def gen_corpus():
    """Config #1: all 58 instances x {trf, dogbox} x {exact, 2-point} plus
    'jac' scaling and 3-point on the exact/trf column, with the reference's
    self-sensitivity for the analytic runs."""
    nu, nb = check_corpus_against_reference_suite()
    KMAX = 8
    out = {}
    rows = []
    n_bit = 0
    variants = [("trf", None, None), ("dogbox", None, None),
                ("trf", "2-point", None), ("dogbox", "2-point", None),
                ("trf", None, "jac"), ("dogbox", None, "jac"),
                ("trf", "3-point", None)]
    for p in corpus():
        for method, fd, scaling in variants:
            key = f"{p.name}|{method}|{fd or 'exact'}|{scaling or '1'}"
            r, t = ref_solve(method, p.fun, p.jac, p.x0, p.lb, p.ub,
                             scaling=scaling, fd=fd)
            o, ot = orc_solve(method, p.fun, p.jac, p.x0, p.lb, p.ub,
                              scaling=scaling, fd=fd)
            bit = results_bitwise(r, t, o, ot)
            n_bit += bit
            rec = pack_result(r, t, p.n, KMAX)
            rows.append(dict(key=key, bitwise=bit, status=rec["status"],
                             nfev=rec["nfev"], njev=rec["njev"],
                             obj=rec["obj"]))
            for fld in ("x", "mask", "trials"):
                out[key + "|" + fld] = rec[fld]
            out[key + "|scalars"] = np.array(
                [rec["obj"], rec["status"], rec["nfev"], rec["njev"],
                 rec["optimality"], rec["ntrials"]], dtype=np.float64)
            if fd is None:
                out[key + "|sens"] = self_sensitivity(method, p, scaling, r, t)
        print(p.name, "done", flush=True)
    out["keys"] = np.array([r["key"] for r in rows])
    out["meta"] = np.array(json.dumps(dict(
        source="reference trf.py/dogbox.py run on tests/problems.py "
               "(= the reference suite, lsq_problems.py:1003-1018)",
        unbounded=nu, bounded=nb,
        runs=len(rows), oracle_bitwise_equal_runs=int(n_bit), kmax=KMAX,
        sens="x_rel, obj_rel, runs with another nfev, runs with another status "
             "of the reference under 1-ulp noise on f (12 runs); first-step rel "
             "(those + 6 runs with 8-ulp noise)")))
    np.savez_compressed(os.path.join(HERE, "corpus.npz"), **out)
    print(f"corpus.npz: {len(rows)} runs; oracle bitwise equal on {n_bit}")
    bad = [r["key"] for r in rows if not r["bitwise"]]
    if bad:
        print("  NOT bitwise:", bad)
    return rows


def gen_batched(name, wl, method, fd, B, seed):
    KMAX = 4
    truth, y = wl.make_data(B, seed=seed)
    X = np.empty((B, wl.n))
    obj = np.empty(B)
    opt = np.empty(B)
    status = np.empty(B, np.int64)
    nfev = np.empty(B, np.int64)
    njev = np.empty(B, np.int64)
    mask = np.empty((B, wl.n), np.int64)
    trials = np.full((B, KMAX, wl.n), np.nan)
    nbit = 0
    for b in range(B):
        fun = lambda x, yb=y[b]: wl.fun_np(x, yb)          # noqa: E731
        jac = (lambda x: wl.jac_np(x)) if fd is None else None
        r, t = ref_solve(method, fun, jac, wl.x0, wl.lb, wl.ub, fd=fd)
        o, ot = orc_solve(method, fun, jac, wl.x0, wl.lb, wl.ub, fd=fd)
        nbit += results_bitwise(r, t, o, ot)
        rec = pack_result(r, t, wl.n, KMAX)
        X[b], obj[b], opt[b] = rec["x"], rec["obj"], rec["optimality"]
        status[b], nfev[b], njev[b] = rec["status"], rec["nfev"], rec["njev"]
        mask[b], trials[b] = rec["mask"], rec["trials"]
    meta = dict(source=f"reference {method} on {type(wl).__name__}", B=B,
                seed=seed, m=wl.m, n=wl.n, jac=fd or "exact",
                oracle_bitwise_equal_runs=int(nbit))
    np.savez_compressed(os.path.join(HERE, name), y=y, truth=truth, x=X,
                        obj=obj, optimality=opt, status=status, nfev=nfev,
                        njev=njev, mask=mask, trials=trials,
                        meta=np.array(json.dumps(meta)))
    print(f"{name}: B={B} mean nfev={nfev.mean():.2f} statuses="
          f"{np.bincount(status).tolist()} oracle bitwise on {nbit}/{B}")


def gen_rat():
    """SURVEY 8a row a24 with bit-identical inputs: finite-difference solves
    of a transcendental-free model (only + - * /), so the device residuals are
    NumPy's to the last bit and every gate of the analytic configs applies."""
    for k, (method, fd) in enumerate((("trf", "2-point"), ("dogbox", "2-point"),
                                      ("trf", "3-point"), ("dogbox", "3-point"))):
        gen_batched(f"rat_{method}_{fd[0]}point.npz", RatPoly5(40), method, fd,
                    96, seed=10 + k)


ASYM_TAIL = (0.8, 1.5, 0.3, 4.0)


def gen_tall():
    """C4-like tall problems at sizes the CPU reference finishes quickly."""
    out = {}
    metas = []
    # a, b: the C4 start (symmetric exponentials, ulp-chaotic for TRF);
    # c, d: asymmetric start, well conditioned along the whole path
    for tag, m, n, seed, tail in (("a", 4096, 16, 3, None), ("b", 20000, 64, 0, None),
                                  ("c", 4096, 16, 3, ASYM_TAIL),
                                  ("d", 20000, 64, 0, ASYM_TAIL)):
        wl = TallLinExp(m, n, seed=seed) if tail is None else \
            TallLinExp(m, n, seed=seed, x0_tail=tail)
        for method in ("trf", "dogbox"):
            r, t = ref_solve(method, wl.fun_np, wl.jac_np, wl.x0, wl.lb, wl.ub)
            o, ot = orc_solve(method, wl.fun_np, wl.jac_np, wl.x0, wl.lb,
                              wl.ub)
            bit = results_bitwise(r, t, o, ot)
            rec = pack_result(r, t, n, 4)
            pre = f"{tag}_{method}_"
            for fld in ("x", "mask", "trials"):
                out[pre + fld] = rec[fld]
            out[pre + "scalars"] = np.array(
                [rec["obj"], rec["status"], rec["nfev"], rec["njev"],
                 rec["optimality"], rec["ntrials"]])
            metas.append(dict(tag=tag, m=m, n=n, seed=seed, method=method,
                              x0_tail=None if tail is None else list(tail),
                              bitwise=bit, status=rec["status"],
                              nfev=rec["nfev"], njev=rec["njev"],
                              nactive=int(np.count_nonzero(rec["mask"]))))
            print("tall", metas[-1])
        out[f"{tag}_y_checksum"] = np.float64(np.sum(wl.y))
        out[f"{tag}_A_checksum"] = np.float64(np.sum(wl.A))
    out["meta"] = np.array(json.dumps(metas))
    np.savez_compressed(os.path.join(HERE, "tall.npz"), **out)


def gen_c5():
    """Config C5 family (m x n linear + 2 exponentials, lb = 0 so that about
    half of the bounds are active at the solution) at sizes the CPU reference
    finishes in seconds: the parity evidence for the n > 64 tall kernels.
    e/f/g: asymmetric start (well conditioned path); h: the C5 benchmark
    start (identical exponentials, exactly rank-deficient Jacobian)."""
    out = {}
    metas = []
    for tag, m, n, seed, tail in (("e", 20000, 256, 5, ASYM_TAIL),
                                  ("f", 8000, 128, 5, ASYM_TAIL),
                                  ("g", 12000, 200, 5, ASYM_TAIL),
                                  ("h", 20000, 256, 5, None)):
        kw = {} if tail is None else dict(x0_tail=tail)
        wl = TallLinExp(m, n, seed=seed, lb=0.0, **kw)
        for method in ("trf", "dogbox"):
            r, t = ref_solve(method, wl.fun_np, wl.jac_np, wl.x0, wl.lb, wl.ub)
            o, ot = orc_solve(method, wl.fun_np, wl.jac_np, wl.x0, wl.lb,
                              wl.ub)
            bit = results_bitwise(r, t, o, ot)
            rec = pack_result(r, t, n, 4)
            pre = f"{tag}_{method}_"
            for fld in ("x", "mask", "trials"):
                out[pre + fld] = rec[fld]
            out[pre + "scalars"] = np.array(
                [rec["obj"], rec["status"], rec["nfev"], rec["njev"],
                 rec["optimality"], rec["ntrials"]])
            metas.append(dict(tag=tag, m=m, n=n, seed=seed, method=method,
                              lb=0.0,
                              x0_tail=None if tail is None else list(tail),
                              bitwise=bit, status=rec["status"],
                              nfev=rec["nfev"], njev=rec["njev"],
                              nactive=int(np.count_nonzero(rec["mask"]))))
            print("c5", metas[-1])
        out[f"{tag}_y_checksum"] = np.float64(np.sum(wl.y))
        out[f"{tag}_A_checksum"] = np.float64(np.sum(wl.A))
    out["meta"] = np.array(json.dumps(metas))
    np.savez_compressed(os.path.join(HERE, "c5.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "tall":
        gen_tall()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "c5":
        gen_c5()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "corpus":
        gen_corpus()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "rat":
        gen_rat()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "fd3":
        # SURVEY 8(f) rank 1: jac='3-point' on the C3 model, both methods
        gen_batched("c3_trf_3point.npz", GaussPeak(128), "trf", "3-point",
                    48, seed=2)
        gen_batched("c3_dogbox_3point.npz", GaussPeak(128), "dogbox",
                    "3-point", 48, seed=3)
        sys.exit(0)
    rng = np.random.default_rng(20261018)
    gen_helpers(rng)
    gen_tr_subproblem(rng)
    gen_corpus()
    gen_batched("c2_trf_exact.npz", ExpDecay2(64), "trf", None, 256, seed=0)
    gen_batched("c3_dogbox_2point.npz", GaussPeak(128), "dogbox", "2-point",
                256, seed=0)
    gen_batched("c2_dogbox_exact.npz", ExpDecay2(64), "dogbox", None, 64,
                seed=1)
    gen_batched("c3_trf_2point.npz", GaussPeak(128), "trf", "2-point", 64,
                seed=1)
    gen_batched("c3_trf_3point.npz", GaussPeak(128), "trf", "3-point", 48,
                seed=2)
    gen_batched("c3_dogbox_3point.npz", GaussPeak(128), "dogbox", "3-point",
                48, seed=3)
    gen_tall()
    gen_c5()
    gen_rat()
