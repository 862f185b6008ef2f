"""Compiled models whose Jacobian is derived from a templated residual
(csrc/blsq_dual.cuh, forward-mode dual numbers).

The unmarked tests need nvcc only: a host program built from blsq_dual.cuh
checks every operation and function against the double expression (value
bits) and mpmath (derivatives, 60 digits), with the documented conventions at
non-differentiable points; the templated reference models compile as
'autodiff', an unsupported function is a compile error in model.cu, and the
cache key covers blsq_dual.cuh.  The gpu tests check that 'inlined' gives the
bits of 'exact' for these models on every lane-group class, method and
active-set path, the accuracy of the derived J, solves against the oracle,
batch invariance, and the materialised kind with `rows` and `cols`."""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import mpmath as mp
import numpy as np
import pytest
import torch

import cases
import test_user_models as um
from bounded_lsq_b200 import BlsqError, PerProblem, least_squares_batched, models

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "bounded_lsq_b200", "csrc")

# the reference models of test_user_models.py, each written once as a template
EXPDECAY2 = r"""
struct Model {
    static constexpr int N = 4;
    template <class T>
    __device__ T residual(const T (&x)[4], int64_t pid, int r, const blsq_model_ctx& c) const {
        const double tr = c.data[1][r];
        const T e1 = exp(-x[1] * tr);
        const T e2 = exp(-x[3] * tr);
        return x[0] * e1 + x[2] * e2 - c.data[0][pid * c.m + r];
    }
};
"""

GAUSSPEAK = r"""
struct GaussPeak {
    static constexpr int N = 6;
    template <class T>
    __device__ T residual(const T (&x)[6], int64_t pid, int r, const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        const T z = (t - x[1]) / x[2];
        return x[0] * exp(-0.5 * z * z) + x[3] + x[4] * t + x[5] * t * t
               - c.data[0][pid * c.m + r];
    }
};
"""

RATPOLY5 = r"""
struct Model {
    static constexpr int N = 5;
    template <class T>
    __device__ T residual(const T (&x)[5], int64_t pid, int r, const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        const T num = x[0] + x[1] * t + x[2] * t * t;
        const T den = 1.0 + x[3] * t + x[4] * t * t;
        return num / den - c.data[0][pid * c.m + r];
    }
};
"""

THREEPEAK = r"""
struct Model {
    static constexpr int N = 11;
    template <class T>
    __device__ T residual(const T (&x)[11], int64_t pid, int r, const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        T f = x[9] + x[10] * t;
        for (int k = 0; k < 3; k++) {
            const T z = (t - x[3 * k + 1]) / x[3 * k + 2];
            f += x[3 * k] * exp(-0.5 * z * z);
        }
        return f - c.data[0][pid * c.m + r];
    }
};
"""

EXP1 = r"""
struct Model {
    static constexpr int N = 1;
    template <class T>
    __device__ T residual(const T (&x)[1], int64_t pid, int r, const blsq_model_ctx& c) const {
        return exp(-x[0] * c.data[1][r]) - c.data[0][pid * c.m + r];
    }
};
"""

# 16 parameters: two Chebyshev expansions u (coefficients x_0..x_15) and v
# (the same coefficients reversed) on s in [-1, 1], mixed nonlinearly
CHEB16 = r"""
struct Model {
    static constexpr int N = 16;
    template <class T>
    __device__ T residual(const T (&x)[16], int64_t pid, int r, const blsq_model_ctx& c) const {
        const double s = c.data[1][r];
        double p0 = 1.0, p1 = s;
        T u = x[0] * p0 + x[1] * p1;
        T v = x[15] * p0 + x[14] * p1;
        for (int k = 2; k < 16; k++) {
            const double p2 = 2.0 * s * p1 - p0;
            u += x[k] * p2;
            v += x[15 - k] * p2;
            p0 = p1;
            p1 = p2;
        }
        return u + 0.3 * sin(v) + 0.1 * tanh(u) + 0.02 * pow(v, 2) - c.data[0][pid * c.m + r];
    }
};
"""


def _cheb(t):
    p = [np.ones_like(t), t]
    for _ in range(2, 16):
        p.append(2.0 * t * p[-1] - p[-2])
    return p


def _cheb16_uv(X, t):
    p = _cheb(t)
    u = X[:, 0:1] * p[0] + X[:, 1:2] * p[1]
    v = X[:, 15:16] * p[0] + X[:, 14:15] * p[1]
    for k in range(2, 16):
        u = u + X[:, k:k + 1] * p[k]
        v = v + X[:, 15 - k:16 - k] * p[k]
    return u, v


def _cheb16_np(X, t):
    u, v = _cheb16_uv(X, t)
    return u + 0.3 * np.sin(v) + 0.1 * np.tanh(u) + 0.02 * v ** 2


# name: the templated source, then the fields of test_user_models.REF
AD = {name: (src,) + um.REF[name][1:] for name, src in (
    ("ExpDecay2", EXPDECAY2), ("GaussPeak", GAUSSPEAK), ("RatPoly5", RATPOLY5),
    ("ThreePeak", THREEPEAK), ("Exp1", EXP1))}
AD["Cheb16"] = (CHEB16, "Model", 16, (-1.0, 1.0), np.full(16, 0.05), np.full(16, -0.4),
                np.full(16, 0.5), [-0.5] * 16, [0.5] * 16, _cheb16_np)


def problem_data(name, m, B, seed):
    src, cls, n, (t0, t1), x0, lb, ub, lo, hi, f = AD[name]
    rng = np.random.default_rng(seed)
    t = np.linspace(t0, t1, m)
    truth = rng.uniform(lo, hi, (B, n))
    y = f(truth, t) + 0.01 * rng.standard_normal((B, m))
    return t, y, np.asarray(x0, dtype=float), np.asarray(lb, float), np.asarray(ub, float)


@pytest.fixture(scope="module")
def cache(tmp_path_factory):
    return str(tmp_path_factory.mktemp("blsq_ad_models"))


@pytest.fixture(scope="module")
def compiled(cache):
    """Every templated model and the hand-written reference models, compiled
    once, in parallel: {name: autodiff model}, {name: hand model}."""
    with ThreadPoolExecutor(8) as ex:
        ad = {k: ex.submit(models.compile_model, v[0], v[1], cache) for k, v in AD.items()}
        hand = {k: ex.submit(models.compile_model, v[0], v[1], cache) for k, v in um.REF.items()}
        return {k: f.result() for k, f in ad.items()}, {k: f.result() for k, f in hand.items()}


# ------------------------------------------------------------- no GPU ----

U = 2.0 ** -53
UNARY = ("neg", "pos", "lit", "powi", "exp", "expm1", "log", "log1p", "sqrt", "cbrt", "sin",
         "cos", "tan", "atan", "sinh", "cosh", "tanh", "erf", "fabs")
BINARY = ("add", "sub", "mul", "div", "pow", "atan2", "hypot", "fmin", "fmax", "iadd", "isub",
          "imul", "idiv")
COMPARE = ("eq", "ne", "lt", "le", "gt", "ge")

# d/da (unary) or (d/da, d/db) in mpmath
MP_D = {
    "neg": lambda a: -1, "pos": lambda a: 1, "lit": lambda a: mp.mpf(2) / 3 - 4,
    "powi": lambda a: 3 * a ** 2, "exp": mp.exp, "expm1": mp.exp, "log": lambda a: 1 / a,
    "log1p": lambda a: 1 / (1 + a), "sqrt": lambda a: 1 / (2 * mp.sqrt(a)),
    "cbrt": lambda a: 1 / (3 * mp.cbrt(abs(a)) ** 2), "sin": mp.cos, "cos": lambda a: -mp.sin(a),
    "tan": lambda a: mp.sec(a) ** 2, "atan": lambda a: 1 / (1 + a * a), "sinh": mp.cosh,
    "cosh": mp.sinh, "tanh": lambda a: mp.sech(a) ** 2,
    "erf": lambda a: 2 / mp.sqrt(mp.pi) * mp.exp(-a * a), "fabs": lambda a: mp.sign(a),
    "add": lambda a, b: (1, 1), "sub": lambda a, b: (1, -1), "mul": lambda a, b: (b, a),
    "div": lambda a, b: (1 / b, -a / b ** 2),
    "pow": lambda a, b: (b * mp.power(a, b - 1), mp.power(a, b) * mp.log(a)),
    "atan2": lambda a, b: (b / (a * a + b * b), -a / (a * a + b * b)),
    "hypot": lambda a, b: (a / mp.hypot(a, b), b / mp.hypot(a, b)),
}
for _op in ("add", "sub", "mul", "div"):
    MP_D["i" + _op] = MP_D[_op]

GRID1 = [0.0, -0.0, 5e-324, 1e-300, 1e-10, 0.1, 0.5, 0.75, 1.0, 1.5, 2.0, 3.5, 10.0, 27.0,
         100.0, 700.0, 1e10, 1e300, float("inf"), float("nan")]
GRID1 = GRID1 + [-x for x in GRID1 if x == x and x != 0.0] + [-1.0 + 2 ** -30, 1.5707963267948966]
GRID2 = [0.0, -0.0, 1e-300, 0.3, 1.0, 2.5, 7.0, 1e5, 1e300, -1e-300, -0.3, -1.0, -2.5, -7.0, 3.0,
         -3.0, float("inf")]


def _build_rules(tmp):
    exe = os.path.join(tmp, "dual_rules")
    subprocess.run([models._nvcc()[0], "-std=c++17", "-fmad=false", "-Xcompiler", "-ffp-contract=off",
                    "-Wno-deprecated-gpu-targets", "-I", CSRC, "-o", exe,
                    os.path.join(HERE, "dual_host", "dual_rules.cu")], check=True)
    return exe


def _run_rules(exe, lines):
    """[(value from the duals, value from doubles, d/da, d/db)] for `lines`
    of (op, form, a, b)."""
    inp = "".join(f"{op} {form} {float(a).hex()} {float(b).hex()}\n"
                  for op, form, a, b in lines)
    out = subprocess.run([exe], input=inp, capture_output=True, text=True, check=True).stdout
    return [tuple(float.fromhex(w) for w in ln.split()) for ln in out.splitlines()]


def _cond(g, args):
    """Condition number of g at args: sum_i |a_i dg/da_i / g|, by relative
    central differences at 60 digits."""
    g0, c = g(*args), mp.mpf(0)
    if g0 == 0:
        return mp.mpf(0)
    for i, a in enumerate(args):
        if a == 0:
            continue
        e = mp.mpf(10) ** -25
        hi = list(args)
        lo = list(args)
        hi[i], lo[i] = a * (1 + e), a * (1 - e)
        c += abs((g(*hi) - g(*lo)) / (2 * e * g0))
    return c


@pytest.fixture(scope="module")
def rules(tmp_path_factory):
    return _build_rules(str(tmp_path_factory.mktemp("dual_rules")))


def test_dual_value_channel_and_derivatives(rules):
    """Every operation and function on a grid with extreme, denormal, infinite
    and NaN arguments: the value of the dual evaluation has the bits of the
    double expression (also for the comparisons), and where the derivative
    exists and is a finite double it is within 8 u (1 + cond) of mpmath, cond
    the derivative's own condition number."""
    lines = [(op, "DD", a, 0.0) for op in UNARY for a in GRID1]
    lines += [(op, form, a, b) for op in BINARY + COMPARE for form in ("DD", "Dd", "dD")
              for a in GRID2 for b in GRID2 if not (op[0] == "i" and form == "dD")]
    out = _run_rules(rules, lines)
    assert len(out) == len(lines)
    checked = 0
    mp.mp.dps = 60
    for (op, form, a, b), (vd, vv, d0, d1) in zip(lines, out):
        assert np.float64(vd).tobytes() == np.float64(vv).tobytes(), (op, form, a, b, vd, vv)
        if op in COMPARE:
            assert d0 == 0.0 and d1 == 0.0
            continue
        if form == "Dd":
            assert d1 == 0.0
        if form == "dD":
            assert d0 == 0.0
        if op in ("fmin", "fmax") or not (np.isfinite(a) and np.isfinite(b) and np.isfinite(vd)):
            continue                                   # conventions: below
        if (op in ("sqrt", "cbrt", "fabs", "log", "hypot", "atan2") and a == 0.0) \
                or (op == "pow" and (a <= 0.0 or b == 0.0)) \
                or (op == "hypot" and a == 0.0 and b == 0.0) or (op == "atan2" and b == 0.0):
            continue
        A, Bm = mp.mpf(a), mp.mpf(b)
        unary = op in UNARY
        if not unary and form == "DD":
            refs = MP_D[op](A, Bm)
            if any(abs(mp.mpf(r)) > np.finfo(float).max for r in refs if mp.im(r) == 0):
                continue                               # an overflowing partial: inf * 0
        for k, got in ((0, d0), (1, d1)):
            if unary and k == 1:
                break
            if (k == 0 and form == "dD") or (k == 1 and form == "Dd"):
                continue
            g = (lambda x, y=None: mp.mpf(MP_D[op](x))) if unary else \
                (lambda x, y, k=k: mp.mpf(MP_D[op](x, y)[k]))
            args = (A,) if unary else (A, Bm)
            ref = g(*args)
            if abs(ref) > np.finfo(float).max or mp.im(ref) != 0:
                continue
            tol = 8 * U * (1 + _cond(g, args)) * abs(ref) + 4 * 2.0 ** -1074
            assert abs(mp.mpf(got) - ref) <= tol, (op, form, a, b, k, got, float(ref))
            checked += 1
    assert checked > 1500, checked


def test_dual_conventions(rules):
    """The derivatives at non-differentiable points documented in
    blsq_dual.cuh."""
    nan = float("nan")
    expect = [  # (op, form, a, b, d/da, d/db)
        ("fabs", "DD", 0.0, 0.0, 0.0, 0.0), ("fabs", "DD", -0.0, 0.0, 0.0, 0.0),
        ("fabs", "DD", -2.0, 0.0, -1.0, 0.0),
        ("sqrt", "DD", 0.0, 0.0, 0.0, 0.0), ("cbrt", "DD", 0.0, 0.0, 0.0, 0.0),
        ("pow", "Dd", 0.0, 0.5, 0.0, 0.0), ("pow", "Dd", 0.0, -1.0, 0.0, 0.0),
        ("pow", "Dd", 0.0, 0.0, 0.0, 0.0), ("pow", "Dd", 0.0, 1.0, 1.0, 0.0),
        ("pow", "Dd", 0.0, 2.0, 0.0, 0.0), ("pow", "DD", 0.0, 2.0, 0.0, 0.0),
        ("pow", "DD", -2.0, 3.0, 12.0, 0.0), ("pow", "dD", -2.0, 2.0, 0.0, 0.0),
        ("pow", "dD", 0.0, 2.0, 0.0, 0.0), ("powi", "DD", -2.0, 0.0, 12.0, 0.0),
        ("hypot", "DD", 0.0, 0.0, 0.0, 0.0), ("atan2", "DD", 0.0, 0.0, 0.0, 0.0),
        ("fmin", "DD", 1.0, 1.0, 0.5, 0.5), ("fmax", "DD", 1.0, 1.0, 0.5, 0.5),
        ("fmin", "DD", 1.0, 2.0, 1.0, 0.0), ("fmin", "DD", 3.0, 2.0, 0.0, 1.0),
        ("fmax", "DD", 1.0, 2.0, 0.0, 1.0), ("fmax", "DD", 3.0, 2.0, 1.0, 0.0),
        ("fmin", "DD", nan, 2.0, 0.0, 1.0), ("fmax", "DD", 2.0, nan, 1.0, 0.0),
        ("fmin", "Dd", 1.0, 1.0, 0.5, 0.0), ("fmax", "dD", 1.0, 1.0, 0.0, 0.5),
    ]
    out = _run_rules(rules, [e[:4] for e in expect])
    for e, (vd, vv, d0, d1) in zip(expect, out):
        assert np.float64(vd).tobytes() == np.float64(vv).tobytes(), e
        assert (d0, d1) == e[4:], (e, d0, d1)


def test_autodiff_models_compile(compiled):
    ad, hand = compiled
    for name, cm in ad.items():
        assert cm.n == AD[name][2] and cm.version == 1, name
        assert cm.jacobian == "autodiff" and cm.has_jacobian, name
    for name, cm in hand.items():
        assert cm.jacobian == "analytic", name


def test_no_jacobian_and_unsupported_function(compiled, cache):
    nj = models.compile_model(um.NOJAC, cache_dir=cache)
    assert nj.jacobian is None and not nj.has_jacobian
    for kind in ("exact", "inlined"):
        with pytest.raises(ValueError, match="jacobian_row.*template"):
            nj.callbacks(kind, m=8)
    with pytest.raises(ValueError, match="jac_kind"):
        compiled[0]["Exp1"].callbacks("inlined-3-point", m=8)
    bad = EXP1.replace("exp(-x[0]", "lgamma(-x[0]")
    with pytest.raises(BlsqError, match="model.cu.*error"):
        models.compile_model(bad, cache_dir=cache)
    # a jacobian_row wins over the templated residual
    row = um.EXP1.split("    __device__ void jacobian_row")[1].rsplit("};", 1)[0]
    both = EXP1.rsplit("};", 1)[0] + "    __device__ void jacobian_row" + row + "};\n"
    assert models.compile_model(both, cache_dir=cache).jacobian == "analytic"


def test_cache_key_covers_dual_header():
    assert any(p.endswith("blsq_dual.cuh") for p in models._HEADERS)
    assert all(os.path.exists(p) for p in models._HEADERS)


def test_cache_changes_with_dual_header(cache, tmp_path, monkeypatch):
    """A changed blsq_dual.cuh is a new key (a copy of the headers stands in
    for the package's)."""
    hdrs = []
    for p in models._HEADERS:
        q = tmp_path / os.path.basename(p)
        q.write_bytes(open(p, "rb").read())
        hdrs.append(str(q))
    monkeypatch.setattr(models, "_HEADERS", hdrs)
    dual = next(h for h in hdrs if h.endswith("blsq_dual.cuh"))
    with open(dual, "a") as f:
        f.write("// a\n")
    assert models.compile_model(EXP1, cache_dir=cache).built
    assert not models.compile_model(EXP1, cache_dir=cache).built
    with open(dual, "a") as f:
        f.write("// b\n")
    assert models.compile_model(EXP1, cache_dir=cache).built


# ---------------------------------------------------------------- GPU ----

DEV = torch.device("cuda:0")


def solve(cm, kind, method, t, y, x0, lb, ub, m, options=None, host=False):
    return um.solve(cm, kind, method, t, y, x0, lb, ub, m, options=options, host=host)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["trf", "dogbox"])
@pytest.mark.parametrize("name", list(AD))
def test_inlined_equals_exact(compiled, name, method):
    """For every lane-group class (m on both sides of each edge, m < n too):
    autodiff 'inlined' gives the bits of autodiff 'exact' (TRF: J and f from
    one dual evaluation against f from the double residual; dogbox: J at the
    Jacobian point), and the rounds went through the compiled hook."""
    cm = compiled[0][name]
    for m in um.lane_class_edges(cm.n):
        data = problem_data(name, m, 96, seed=m)
        r0, _ = solve(cm, "exact", method, *data, m)
        r1, served = solve(cm, "inlined", method, *data, m)
        um.same_bits(r0, r1)
        assert served[0] >= 2, m


@pytest.mark.gpu
@pytest.mark.parametrize("name,method", [("GaussPeak", "dogbox"), ("ExpDecay2", "trf")])
def test_inlined_active_set_paths(compiled, name, method):
    """The same bits after compaction, in the graph tail, with `chunk` and
    with staged host inputs."""
    cm = compiled[0][name]
    m = 64 if name == "ExpDecay2" else 128
    B = 140000
    t, y, x0, lb, ub = problem_data(name, m, 4096, seed=21)
    y = np.tile(y, (B // 4096 + 1, 1))[:B]
    r0, _ = solve(cm, "exact", method, t, y, x0, lb, ub, m)
    for opts, host in ((None, False), ({"chunk": 50000}, False),
                       ({"h2d_chunks": 2, "prologue_rounds": 3}, True)):
        r1, served = solve(cm, "inlined", method, t, y, x0, lb, ub, m, options=opts, host=host)
        um.same_bits(r0, r1)
        assert served[0] >= 10, opts
    assert int((r0.status > 0).sum()) >= 0.99 * B


# the models' residuals in mpmath, without the data term
MP_F = {
    "ExpDecay2": lambda x, t: x[0] * mp.exp(-x[1] * t) + x[2] * mp.exp(-x[3] * t),
    "GaussPeak": lambda x, t: x[0] * mp.exp(-((t - x[1]) / x[2]) ** 2 / 2) + x[3] + x[4] * t
    + x[5] * t * t,
    "RatPoly5": lambda x, t: (x[0] + x[1] * t + x[2] * t * t) / (1 + x[3] * t + x[4] * t * t),
    "ThreePeak": lambda x, t: x[9] + x[10] * t + sum(
        x[3 * k] * mp.exp(-((t - x[3 * k + 1]) / x[3 * k + 2]) ** 2 / 2) for k in range(3)),
    "Exp1": lambda x, t: mp.exp(-x[0] * t),
    "Cheb16": None,
}


def _cheb16_mp(x, t):
    p = [mp.mpf(1), t]
    for _ in range(2, 16):
        p.append(2 * t * p[-1] - p[-2])
    u = sum(x[k] * p[k] for k in range(16))
    v = sum(x[15 - k] * p[k] for k in range(16))
    return u + mp.mpf("0.3") * mp.sin(v) + mp.mpf("0.1") * mp.tanh(u) + mp.mpf("0.02") * v ** 2


MP_F["Cheb16"] = _cheb16_mp


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(AD))
def test_jacobian_accuracy(compiled, name):
    """The materialised autodiff J at random points against mpmath
    derivatives (40 digits) of the model: per element, the error is at most
    max(4 x the hand-written jacobian_row's error, 16 u ||row||_inf)."""
    ad, hand = compiled
    src, cls, n, (t0, t1), x0, lb, ub, lo, hi, f = AD[name]
    m, P = 16, 3
    rng = np.random.default_rng(11)
    t = np.linspace(t0, t1, m)
    X = rng.uniform(lo, hi, (P, n))
    y = np.zeros((P, m))
    args = (cases.T(y, DEV), cases.T(t, DEV))
    Xt = cases.T(X, DEV)
    Jad = ad[name].callbacks("exact", m=m)[1](Xt, None, *args).cpu().numpy()
    Jh = hand[name].callbacks("exact", m=m)[1](Xt, None, *args).cpu().numpy() \
        if name in hand else None
    mp.mp.dps = 40
    worst = 0.0
    for p in range(P):
        for r in range(m):
            tr = mp.mpf(t[r])
            xs = [mp.mpf(v) for v in X[p]]
            ref = []
            for k in range(n):
                def g(h, k=k):
                    xx = list(xs)
                    xx[k] = h
                    return MP_F[name](xx, tr)
                ref.append(mp.diff(g, xs[k]))
            ref = np.array([float(v) for v in ref])
            floor = 16 * U * np.abs(ref).max()
            err = np.abs(Jad[p, r] - ref)
            bound = np.full(n, floor)
            if Jh is not None:
                bound = np.maximum(bound, 4 * np.abs(Jh[p, r] - ref))
            assert np.all(err <= bound), (p, r, err, bound)
            worst = max(worst, float((err / np.maximum(floor, 1e-300)).max()))
    print(f"{name}: worst autodiff error {worst * 16:.2f} u ||row||")


def _jac_np(name, x, t):
    if name in ("GaussPeak", "ThreePeak"):
        return um._fd_free_jac(name, x, t)
    if name == "RatPoly5":
        num = x[0] + x[1] * t + x[2] * t * t
        den = 1.0 + x[3] * t + x[4] * t * t
        q = num / (den * den)
        return np.stack([1 / den, t / den, t * t / den, -q * t, -q * t * t], axis=1)
    u, v = _cheb16_uv(x[None], t)
    du = 1.0 + 0.1 / np.cosh(u[0]) ** 2
    dv = 0.3 * np.cos(v[0]) + 0.04 * v[0]
    p = _cheb(t)
    return np.stack([du * p[k] + dv * p[15 - k] for k in range(16)], axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["GaussPeak", "RatPoly5", "ThreePeak", "Cheb16"])
@pytest.mark.parametrize("method", ["trf", "dogbox"])
def test_against_oracle(compiled, name, method):
    """Autodiff 'inlined' solves of fresh problems against the oracle with
    the analytic Jacobian, with the gates of test_user_models' analytic
    kinds: every cost within 1e-8, status, nfev, x (1e-8) and the active set
    identical for >= 99 %."""
    from oracle import blsq_oracle as orc
    f = AD[name][9]
    m, B = 128, 100
    t, y, x0, lb, ub = problem_data(name, m, B, seed=1234)
    res, _ = solve(compiled[0][name], "inlined", method, t, y, x0, lb, ub, m)
    X, st, nf = res.x.cpu().numpy(), res.status.cpu().numpy(), res.nfev.cpu().numpy()
    ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
    assert np.all(X >= lb) and np.all(X <= ub)
    exact = 0
    for b in range(B):
        r = orc.least_squares(lambda x, yb: f(x[None], t)[0] - yb, x0,
                              jac=lambda x, yb: _jac_np(name, x, t), bounds=(lb, ub),
                              method=method, args=(y[b],))
        assert abs(ob[b] - r.obj_value) <= 1e-8 * r.obj_value + 1e-18, b
        exact += (st[b] == r.status and nf[b] == r.nfev and
                  np.allclose(X[b], r.x, rtol=1e-8, atol=1e-9) and
                  np.array_equal(mk[b], np.asarray(r.active_mask)))
    assert exact >= 0.99 * B, exact


@pytest.mark.gpu
@pytest.mark.parametrize("name,method", [("GaussPeak", "dogbox"), ("Cheb16", "trf")])
def test_batch_permutation_and_subset(compiled, name, method):
    """A permuted batch or a subset gives each problem the bits it gets in
    the whole batch."""
    m = 96
    t, y, x0, lb, ub = problem_data(name, m, 512, seed=77)
    cm = compiled[0][name]
    r0, _ = solve(cm, "inlined", method, t, y, x0, lb, ub, m)
    perm = np.random.default_rng(3).permutation(512)
    for sel in (perm, np.arange(1, 512, 3)):
        r1, _ = solve(cm, "inlined", method, t, y[sel], x0, lb, ub, m)
        for fld in um.FIELDS:
            a = getattr(r0, fld).cpu().numpy()[sel]
            assert cases.bits(getattr(r1, fld).cpu().numpy(), a), fld


@pytest.mark.gpu
def test_rows_and_cols_materialised(compiled):
    """Autodiff 'exact' with `rows` gives each problem the bits of the dense
    solve of its first rows[b] residuals, and with `cols` those of the dense
    solve of its first cols[b] parameters (the others held at x0)."""
    cm = compiled[0]["GaussPeak"]
    m, B, n = 64, 300, 6
    t, y, x0, lb, ub = problem_data("GaussPeak", m, B, seed=8)
    fun, jac = cm.callbacks("exact", m=m)
    Y, Tt = cases.T(y, DEV), cases.T(t, DEV)
    X0 = cases.T(np.tile(x0, (B, 1)), DEV)

    rows = np.where(np.arange(B) % 3 == 0, 40, m).astype(np.int32)
    r = least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method="trf",
                              args=(PerProblem(Y), Tt),
                              options={"rows": torch.as_tensor(rows, device=DEV)})
    for mr in (40, m):
        sel = np.nonzero(rows == mr)[0]
        rd, _ = solve(cm, "exact", "trf", t[:mr], np.ascontiguousarray(y[sel, :mr]), x0, lb, ub,
                      mr)
        for fld in um.FIELDS:
            assert cases.bits(getattr(r, fld).cpu().numpy()[sel],
                              getattr(rd, fld).cpu().numpy()), (mr, fld)

    cols = np.where(np.arange(B) % 2 == 0, 4, n).astype(np.int32)
    for method in ("trf", "dogbox"):
        r = least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method=method,
                                  args=(PerProblem(Y), Tt),
                                  options={"cols": torch.as_tensor(cols, device=DEV)})
        for N in (4, n):
            sel = np.nonzero(cols == N)[0]
            args = (PerProblem(Y[sel].contiguous()), Tt)
            if N == n:
                f, j = fun, jac
            else:
                def f(X, idx, Yb, T, P):
                    return fun(torch.cat([X, P if idx is None else P[idx]], 1), idx, Yb, T)

                def j(X, idx, Yb, T, P):
                    return jac(torch.cat([X, P if idx is None else P[idx]], 1), idx, Yb,
                               T)[:, :, :N]
                f.blsq_indexed = j.blsq_indexed = True
                args += (PerProblem(cases.T(np.tile(x0[N:], (len(sel), 1)), DEV)),)
            rd = least_squares_batched(f, X0[sel, :N].contiguous(), jac=j,
                                       bounds=(lb[:N], ub[:N]), method=method, args=args)
            for fld in um.FIELDS:
                a = getattr(r, fld).cpu().numpy()[sel]
                if fld in ("x", "active_mask"):
                    a = a[:, :N]
                assert cases.bits(getattr(rd, fld).cpu().numpy(), a), (method, N, fld)
