"""The oracle (oracle/blsq_oracle.py) against the golden vectors produced by the
unmodified reference (tests/golden/make_golden.py).  CPU only.

Elementwise passes are compared bit-for-bit.  Anything that goes through a BLAS
reduction is compared bit-for-bit when possible and otherwise to 1e-12 (the
golden files were written on the authoring host; another CPU may pick another
OpenBLAS kernel and sum in another order)."""
import json
import os

import numpy as np
import pytest

import packed_npz
from oracle import blsq_oracle as orc
from problems import corpus
from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak, TallLinExp

SQ = np.finfo(float).eps ** 0.5


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _close(a, b, rtol=1e-12):
    return _bits(a, b) or np.allclose(a, b, rtol=rtol, atol=0, equal_nan=True)


def test_helpers_bit_exact(golden_dir):
    z = packed_npz.Packed(os.path.join(golden_dir, "helpers.npz"))
    assert json.loads(str(z["meta"]))["oracle_bitwise_equal"]
    for i in range(int(z["ncases"])):
        g = lambda k: z[f"c{i}_{k}"]            # noqa: E731
        x, xc, d, lb, ub = g("x"), g("xc"), g("d"), g("lb"), g("ub")
        step, hits = orc.step_size_to_bound(x, d, lb, ub)
        assert _bits(step, g("step")) and _bits(hits, g("hits"))
        assert _bits(orc.find_active_constraints(x, lb, ub, 1e-3), g("act_1e3"))
        assert _bits(orc.find_active_constraints(x, lb, ub, SQ), g("act_sq"))
        assert _bits(orc.make_strictly_feasible(xc, lb, ub, 0), g("msf0"))
        assert _bits(orc.make_strictly_feasible(xc, lb, ub, 1e-10), g("msf1"))
        v, jv = orc.scaling_vector(xc, g("g"), lb, ub)
        assert _bits(v, g("v")) and _bits(jv, g("jv"))
        assert orc.in_bounds(x, lb, ub) == bool(g("inb"))
        fi = orc.find_intersection(xc, g("tr"), lb, ub)
        for a, k in zip(fi, ("fi_lo", "fi_hi", "fi_ol", "fi_ou", "fi_tl", "fi_tu")):
            assert _bits(a, g(k))
        assert _bits(orc.fd_steps(xc, lb, ub, None, "2-point")[0], g("fd2"))
        assert _bits(orc.fd_steps(xc, lb, ub, 1e-2, "2-point")[0], g("fd2_rel"))
        h3, one3 = orc.fd_steps(xc, lb, ub, None, "3-point")
        assert _bits(h3, g("fd3")) and _bits(one3, g("fd3_one"))


def test_tr_subproblem(golden_dir):
    z = packed_npz.Packed(os.path.join(golden_dir, "tr_subproblem.npz"))
    for k in range(int(z["n_tr"])):
        g = lambda f: z[f"tr{k}_{f}"]           # noqa: E731
        a0 = float(g("alpha0"))
        a0 = None if np.isnan(a0) else a0
        s = g("s")
        p, alpha, nit = orc.solve_lsq_trust_region(
            s.size, int(g("m")), g("uf"), s, g("V"), float(g("Delta")), a0)
        assert nit == int(g("nit"))
        assert _close(p, g("p")) and _close(alpha, g("alpha"))
    for k in range(int(z["n_it"])):
        g = lambda f: z[f"it{k}_{f}"]           # noqa: E731
        t = orc.intersect_trust_region(g("x"), g("s"), float(g("Delta")))
        assert _close(np.array(t), g("t"))
    out = np.array([orc.minimize_quadratic(a, b, l, u) for (a, b), l, u in
                    zip(z["mq_ab"], z["mq_lo"], z["mq_hi"])])
    assert _bits(out, z["mq_out"])
    for k in range(int(z["n_dl"])):
        g = lambda f: z[f"dl{k}_{f}"]           # noqa: E731
        st, bh, th = orc.dogleg_step(g("x"), g("cauchy").copy(), g("newton"),
                                     g("tr"), g("lb"), g("ub"))
        assert _bits(st, g("step")) and _bits(bh, g("hits"))
        assert bool(th) == bool(g("tr_hit"))
        cs, cb, ct = orc.constrained_cauchy_step(g("x"), g("cauchy"), g("tr"),
                                                 g("lb"), g("ub"))
        assert _bits(cs, g("cstep")) and _bits(cb, g("chits"))
        assert bool(ct) == bool(g("ctr_hit"))


def test_intersect_raises():
    with pytest.raises(ValueError):
        orc.intersect_trust_region(np.ones(2), np.zeros(2), 5.0)
    with pytest.raises(ValueError):
        orc.intersect_trust_region(np.ones(2) * 9, np.ones(2), 1.0)


def _run_oracle(method, fun, jac, x0, lb, ub, fd=None, scaling=None):
    trials, first = [], [True]

    def fw(x):
        if first[0]:
            first[0] = False
        else:
            trials.append(x.copy())
        return np.atleast_1d(fun(x))

    if fd is None:
        jw = lambda x, f: np.atleast_2d(jac(x))                 # noqa: E731
    else:
        jw = lambda x, f: np.atleast_2d(                        # noqa: E731
            orc.fd_jacobian(fun, x, f, lb, ub, None, fd))
    sc = scaling if isinstance(scaling, str) else np.ones_like(x0)
    solver = orc.trf if method == "trf" else orc.dogbox
    return solver(fw, jw, x0.copy(), lb, ub, SQ, SQ, SQ, None, sc), trials


def _check_against(rec_x, rec_mask, rec_trials, scal, res, trials, name):
    obj, status, nfev, njev, opt, ntr = scal
    assert res.status == int(status), name
    assert res.nfev == int(nfev) and res.njev == int(njev), name
    assert _bits(np.asarray(res.active_mask, np.int64), rec_mask), name
    assert _close(res.x, rec_x, 1e-10), name
    assert _close(res.obj_value, obj, 1e-10), name
    k = min(len(trials), rec_trials.shape[0])
    if k:
        assert _close(np.array(trials[:k]), rec_trials[:k], 1e-10), name


def test_corpus_full_solves(golden_dir):
    z = _load(golden_dir, "corpus.npz")
    meta = json.loads(str(z["meta"]))
    assert meta["oracle_bitwise_equal_runs"] == meta["runs"]
    probs = {p.name: p for p in corpus()}
    for key in z["keys"]:
        key = str(key)
        name, method, jac, scaling = key.split("|")
        p = probs[name]
        res, trials = _run_oracle(method, p.fun, p.jac, p.x0, p.lb, p.ub,
                                  fd=None if jac == "exact" else jac,
                                  scaling="jac" if scaling == "jac" else None)
        _check_against(z[key + "|x"], z[key + "|mask"], z[key + "|trials"],
                       z[key + "|scalars"], res, trials, key)


@pytest.mark.parametrize("fname,wl,method,fd", [
    ("c2_trf_exact.npz", ExpDecay2(64), "trf", None),
    ("c2_dogbox_exact.npz", ExpDecay2(64), "dogbox", None),
    ("c3_dogbox_2point.npz", GaussPeak(128), "dogbox", "2-point"),
    ("c3_trf_2point.npz", GaussPeak(128), "trf", "2-point"),
])
def test_batched_samples(golden_dir, fname, wl, method, fd):
    z = _load(golden_dir, fname)
    meta = json.loads(str(z["meta"]))
    assert meta["oracle_bitwise_equal_runs"] == meta["B"]
    _, y = wl.make_data(meta["B"], seed=meta["seed"])
    assert _bits(y, z["y"]), "synthetic generator drifted from the golden data"
    for b in range(0, meta["B"], 4):      # every 4th problem keeps CPU time low
        fun = lambda x, yb=y[b]: wl.fun_np(x, yb)               # noqa: E731
        jac = (lambda x: wl.jac_np(x)) if fd is None else None
        res, trials = _run_oracle(method, fun, jac, wl.x0, wl.lb, wl.ub, fd=fd)
        scal = (z["obj"][b], z["status"][b], z["nfev"][b], z["njev"][b],
                z["optimality"][b], 0)
        _check_against(z["x"][b], z["mask"][b], z["trials"][b], scal, res,
                       trials, f"{fname}[{b}]")


def test_tall_small(golden_dir):
    z = _load(golden_dir, "tall.npz")
    for meta in json.loads(str(z["meta"])):
        tag = meta["tag"]
        if tag not in ("a", "c"):
            continue                 # b, d (m=20000, n=64) are host-emul / GPU cases
        kw = {} if meta.get("x0_tail") is None else dict(x0_tail=meta["x0_tail"])
        wl = TallLinExp(meta["m"], meta["n"], seed=meta["seed"], **kw)
        assert _bits(np.float64(np.sum(wl.y)), z[tag + "_y_checksum"])
        res, trials = _run_oracle(meta["method"], wl.fun_np, wl.jac_np, wl.x0,
                                  wl.lb, wl.ub)
        pre = f"{tag}_{meta['method']}_"
        _check_against(z[pre + "x"], z[pre + "mask"], z[pre + "trials"],
                       z[pre + "scalars"], res, trials, pre)


def test_front_end_validation():
    f = lambda x: x - 1.0                                       # noqa: E731
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], method="oops")
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], bounds=(0, 1, 2))
    with pytest.raises(ValueError):
        orc.least_squares(f, [[2.0]])
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], bounds=(3.0, 1.0))
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], bounds=(3.0, 4.0))
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], jac="oops")
    with pytest.raises(ValueError):
        orc.least_squares(f, [2.0], scaling=-1.0)
    with pytest.warns(UserWarning):
        orc.least_squares(f, [2.0], ftol=1e-30)
    r = orc.least_squares(f, [2.0], bounds=(1.5, 3.0))
    assert r.success and abs(r.x[0] - 1.5) < 1e-4 and r.active_mask[0] == -1
