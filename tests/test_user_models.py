"""Residual models compiled from user source (models.compile_model).

The unmarked tests need nvcc only: every reference model compiles for sm_100a
and loads, compile errors and missing functions are reported, the cache
skips nvcc for an unchanged model and not for a changed one, and bad data
arguments are refused before any launch.  The gpu tests check that the
inlined kinds give the bits of the materialised ones for every lane-group
class, method and active-set path, and that the materialised kinds give the
bits of the library's own callbacks."""
import json
import os
import types
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import cases
from bounded_lsq_b200 import BlsqError, PerProblem, least_squares_batched, models
from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak, RatPoly5

# data: c.data[0] = y (PerProblem, (B, m)), c.data[1] = t (shared, (m,))
EXPDECAY2 = r"""
struct Model {   // same operation order as expdecay2_kernel
    static constexpr int N = 4;
    __device__ double residual(const double (&x)[4], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        const double tr = c.data[1][r];
        const double e1 = exp(-x[1] * tr);
        const double e2 = exp(-x[3] * tr);
        return x[0] * e1 + x[2] * e2 - c.data[0][pid * c.m + r];
    }
    __device__ void jacobian_row(const double (&x)[4], int64_t pid, int r,
                                 const blsq_model_ctx& c, double (&j)[4]) const {
        const double tr = c.data[1][r];
        const double e1 = exp(-x[1] * tr);
        const double e2 = exp(-x[3] * tr);
        j[0] = e1;
        j[1] = -x[0] * tr * e1;
        j[2] = e2;
        j[3] = -x[2] * tr * e2;
    }
};
"""

GAUSSPEAK = r"""
struct GaussPeak {
    static constexpr int N = 6;
    __device__ double residual(const double (&x)[6], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        const double z = (t - x[1]) / x[2];
        return x[0] * exp(-0.5 * z * z) + x[3] + x[4] * t + x[5] * t * t
               - c.data[0][pid * c.m + r];
    }
    __device__ void jacobian_row(const double (&x)[6], int64_t pid, int r,
                                 const blsq_model_ctx& c, double (&j)[6]) const {
        const double t = c.data[1][r];
        const double z = (t - x[1]) / x[2];
        const double e = exp(-0.5 * z * z);
        j[0] = e;
        j[1] = x[0] * e * z / x[2];
        j[2] = x[0] * e * z * z / x[2];
        j[3] = 1.0;
        j[4] = t;
        j[5] = t * t;
    }
};
"""

# + - * / only, in the operation order of synthetic.RatPoly5.fun_t
RATPOLY5 = r"""
struct Model {
    static constexpr int N = 5;
    __device__ double residual(const double (&x)[5], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        const double num = x[0] + x[1] * t + x[2] * t * t;
        const double den = 1.0 + x[3] * t + x[4] * t * t;
        return num / den - c.data[0][pid * c.m + r];
    }
    __device__ void jacobian_row(const double (&x)[5], int64_t pid, int r,
                                 const blsq_model_ctx& c, double (&j)[5]) const {
        const double t = c.data[1][r];
        const double num = x[0] + x[1] * t + x[2] * t * t;
        const double den = 1.0 + x[3] * t + x[4] * t * t;
        const double q = num / (den * den);
        j[0] = 1.0 / den;
        j[1] = t / den;
        j[2] = t * t / den;
        j[3] = -q * t;
        j[4] = -q * t * t;
    }
};
"""

# three Gaussian peaks on a linear background (a W11-like spectrum fit)
THREEPEAK = r"""
struct Model {
    static constexpr int N = 11;
    __device__ double residual(const double (&x)[11], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        const double t = c.data[1][r];
        double f = x[9] + x[10] * t;
        for (int k = 0; k < 3; k++) {
            const double z = (t - x[3 * k + 1]) / x[3 * k + 2];
            f += x[3 * k] * exp(-0.5 * z * z);
        }
        return f - c.data[0][pid * c.m + r];
    }
    __device__ void jacobian_row(const double (&x)[11], int64_t pid, int r,
                                 const blsq_model_ctx& c, double (&j)[11]) const {
        const double t = c.data[1][r];
        for (int k = 0; k < 3; k++) {
            const double s = x[3 * k + 2];
            const double z = (t - x[3 * k + 1]) / s;
            const double e = exp(-0.5 * z * z);
            j[3 * k] = e;
            j[3 * k + 1] = x[3 * k] * e * z / s;
            j[3 * k + 2] = x[3 * k] * e * z * z / s;
        }
        j[9] = 1.0;
        j[10] = t;
    }
};
"""

EXP1 = r"""
struct Model {
    static constexpr int N = 1;
    __device__ double residual(const double (&x)[1], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        return exp(-x[0] * c.data[1][r]) - c.data[0][pid * c.m + r];
    }
    __device__ void jacobian_row(const double (&x)[1], int64_t pid, int r,
                                 const blsq_model_ctx& c, double (&j)[1]) const {
        const double t = c.data[1][r];
        j[0] = -t * exp(-x[0] * t);
    }
};
"""

NOJAC = r"""
struct Model {
    static constexpr int N = 2;
    __device__ double residual(const double (&x)[2], int64_t pid, int r,
                               const blsq_model_ctx& c) const {
        return x[0] * c.data[1][r] + x[1] - c.data[0][pid * c.m + r];
    }
};
"""


def _threepeak_np(X, t):
    f = X[:, 9:10] + X[:, 10:11] * t
    for k in range(3):
        z = (t - X[:, 3 * k + 1:3 * k + 2]) / X[:, 3 * k + 2:3 * k + 3]
        f = f + X[:, 3 * k:3 * k + 1] * np.exp(-0.5 * z * z)
    return f


# name: (source, class name, n, t range, x0, lb, ub, truth low, truth high, f(X, t))
REF = {
    "ExpDecay2": (EXPDECAY2, "Model", 4, (0.0, 4.0), ExpDecay2.x0, ExpDecay2.lb, ExpDecay2.ub,
                  [1.0, 0.5, 0.5, 2.0], [3.0, 1.5, 2.0, 4.0],
                  lambda X, t: X[:, 0:1] * np.exp(-X[:, 1:2] * t)
                  + X[:, 2:3] * np.exp(-X[:, 3:4] * t)),
    "GaussPeak": (GAUSSPEAK, "GaussPeak", 6, (-5.0, 5.0), GaussPeak.x0, GaussPeak.lb,
                  GaussPeak.ub, [1.0, -1.0, 0.5, 0.0, -0.1, -0.01],
                  [3.0, 1.0, 1.5, 1.0, 0.1, 0.01],
                  lambda X, t: X[:, 0:1] * np.exp(-0.5 * ((t - X[:, 1:2]) / X[:, 2:3]) ** 2)
                  + X[:, 3:4] + X[:, 4:5] * t + X[:, 5:6] * t * t),
    "RatPoly5": (RATPOLY5, "Model", 5, (0.0, 3.0), RatPoly5.x0, RatPoly5.lb, RatPoly5.ub,
                 [0.5, -0.5, 0.0, 0.1, 0.05], [2.5, 1.5, 0.25, 0.8, 0.5],
                 lambda X, t: (X[:, 0:1] + X[:, 1:2] * t + X[:, 2:3] * t * t)
                 / (1.0 + X[:, 3:4] * t + X[:, 4:5] * t * t)),
    "ThreePeak": (THREEPEAK, "Model", 11, (0.0, 10.0),
                  np.array([1.5, 2.0, 0.6, 1.5, 5.0, 0.6, 1.5, 8.0, 0.6, 0.2, 0.0]),
                  np.array([0.0, 1.0, 0.2, 0.0, 4.0, 0.2, 0.0, 7.0, 0.2, -1.0, -1.0]),
                  np.array([4.0, 3.0, 1.5, 4.0, 6.0, 1.5, 4.0, 9.0, 1.5, 1.0, 1.0]),
                  [1.0, 1.7, 0.4, 1.0, 4.7, 0.4, 1.0, 7.7, 0.4, 0.0, -0.03],
                  [2.0, 2.3, 0.8, 2.0, 5.3, 0.8, 2.0, 8.3, 0.8, 0.4, 0.03], _threepeak_np),
    "Exp1": (EXP1, "Model", 1, (0.0, 4.0), np.array([1.0]), np.array([0.0]),
             np.array([5.0]), [0.3], [3.0], lambda X, t: np.exp(-X[:, 0:1] * t)),
}
FIELDS = ("x", "obj_value", "status", "nfev", "njev", "active_mask")


@pytest.fixture(scope="module")
def cache(tmp_path_factory):
    return str(tmp_path_factory.mktemp("blsq_models"))


@pytest.fixture(scope="module")
def compiled(cache):
    """Every reference model, compiled once, in parallel."""
    with ThreadPoolExecutor(len(REF)) as ex:
        fut = {k: ex.submit(models.compile_model, v[0], v[1], cache) for k, v in REF.items()}
        return {k: f.result() for k, f in fut.items()}


def lane_class_edges(n):
    """m at both sides of every lane-group class edge of lin_kernel for n
    parameters (blsq_lin.cuh LinCfg / lin_class), and one m < n."""
    rpl = 8 if n <= 6 else (4 if n <= 12 else 2)
    groups = (8, 16, 32) if n <= 8 else (16, 32)
    ms = {max(1, n - 1)}
    for g in groups:
        ms |= {g * rpl, g * rpl + 1}
    return sorted(ms)


# ------------------------------------------------------------- no GPU ----

def test_reference_models_compile(compiled):
    for name, cm in compiled.items():
        assert cm.n == REF[name][2], name
        assert cm.has_jacobian and cm.version == 1, name
        assert os.path.exists(cm.path)


def test_compile_errors(cache):
    with pytest.raises(BlsqError, match="model.cu.*error"):
        models.compile_model("struct Model { static constexpr int N = 2 }", cache_dir=cache)
    no_residual = EXP1.split("__device__ double residual")[0] + \
        "__device__ void jacobian_row" + EXP1.split("__device__ void jacobian_row")[1]
    with pytest.raises(BlsqError, match="residual"):
        models.compile_model(no_residual, cache_dir=cache)
    nj = models.compile_model(NOJAC, cache_dir=cache)
    assert nj.n == 2 and not nj.has_jacobian
    for kind in ("exact", "inlined"):
        with pytest.raises(ValueError, match="jacobian_row"):
            nj.callbacks(kind, m=8)
    with pytest.raises(ValueError, match="jac_kind"):
        nj.callbacks("inlined-3-point", m=8)
    # the host emulation of the library cannot run compiled kernels
    with pytest.raises(BlsqError, match="CUDA devices only"):
        nj.callbacks("2-point", m=8, lib=types.SimpleNamespace(requires_cuda=False))


def test_cache(compiled, cache, tmp_path, monkeypatch):
    again = models.compile_model(EXPDECAY2, cache_dir=cache)
    assert not again.built and again.path == compiled["ExpDecay2"].path
    changed = models.compile_model(EXPDECAY2 + "\n// changed\n", cache_dir=cache)
    assert changed.built and changed.path != again.path
    # a changed header is a new key too
    hdr = tmp_path / "extra.cuh"
    hdr.write_text("// one\n")
    monkeypatch.setattr(models, "_HEADERS", models._HEADERS + [str(hdr)])
    assert models.compile_model(EXP1, cache_dir=cache).built
    assert not models.compile_model(EXP1, cache_dir=cache).built
    hdr.write_text("// two\n")
    assert models.compile_model(EXP1, cache_dir=cache).built


def test_bad_data_arguments(compiled):
    fun, jac = compiled["Exp1"].callbacks("exact", m=4)
    X = torch.zeros((2, 1), dtype=torch.float64)
    ok = torch.zeros(4, dtype=torch.float64)
    with pytest.raises(ValueError, match="at most 8"):
        fun(X, None, *([ok] * 9))
    with pytest.raises(ValueError, match="float64"):
        fun(X, None, ok.float())
    with pytest.raises(ValueError, match="CUDA|cuda"):
        jac(X, None, ok)                    # a CPU tensor
    with pytest.raises(ValueError):
        fun(X, None, 1.0)                   # not a tensor


# ---------------------------------------------------------------- GPU ----

DEV = torch.device("cuda:0")


def problem_data(name, m, B, seed):
    src, cls, n, (t0, t1), x0, lb, ub, lo, hi, f = REF[name]
    rng = np.random.default_rng(seed)
    t = np.linspace(t0, t1, m)
    truth = rng.uniform(lo, hi, (B, n))
    y = f(truth, t) + 0.01 * rng.standard_normal((B, m))
    return t, y, np.asarray(x0, dtype=float), np.asarray(lb, float), np.asarray(ub, float)


def counted_hook(fun):
    """Wrap fun.blsq_linearise: served[0] counts the rounds it linearised."""
    served, inner = [0], fun.blsq_linearise

    def hook(*a, **k):
        r = inner(*a, **k)
        served[0] += r is not None
        return r
    fun.blsq_linearise = hook
    return served


def solve(cm, kind, method, t, y, x0, lb, ub, m, options=None, host=False):
    fun, jac = cm.callbacks(kind, m=m)
    served = counted_hook(fun) if hasattr(fun, "blsq_linearise") else None
    B = y.shape[0]
    X0 = cases.T(np.tile(x0, (B, 1)), DEV)
    Y, Tt = cases.T(y, DEV), cases.T(t, DEV)
    if host:
        X0, Y = X0.cpu().pin_memory(), Y.cpu().pin_memory()
    res = least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method=method,
                                args=(PerProblem(Y), Tt), options=options or {})
    return res, served


def same_bits(r0, r1):
    for fld in FIELDS:
        assert cases.bits(getattr(r1, fld).cpu().numpy(), getattr(r0, fld).cpu().numpy()), fld


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["trf", "dogbox"])
@pytest.mark.parametrize("name", list(REF))
def test_inlined_equals_materialised(compiled, name, method):
    """For every lane-group class (m on both sides of each edge, m < n too):
    'inlined' gives the bits of 'exact' and 'inlined-2-point' those of
    '2-point', and the rounds went through the compiled hook."""
    cm = compiled[name]
    for m in lane_class_edges(cm.n):
        data = problem_data(name, m, 96, seed=m)
        for mat, inl in (("exact", "inlined"), ("2-point", "inlined-2-point")):
            r0, _ = solve(cm, mat, method, *data, m)
            r1, served = solve(cm, inl, method, *data, m)
            same_bits(r0, r1)
            assert served[0] >= 2, (m, inl)


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind,method", [("ExpDecay2", "inlined", "trf"),
                                              ("GaussPeak", "inlined-2-point", "dogbox")])
def test_inlined_active_set_paths(compiled, name, kind, method):
    """The same bits after compaction, in the graph tail, with `chunk` and
    with staged host inputs (two copy chunks: the prologue runs the second
    at a problem offset)."""
    cm = compiled[name]
    m = 64 if name == "ExpDecay2" else 128
    B = 140000
    t, y, x0, lb, ub = problem_data(name, m, 4096, seed=21)
    y = np.tile(y, (B // 4096 + 1, 1))[:B]
    mat = "exact" if kind == "inlined" else "2-point"
    r0, _ = solve(cm, mat, method, t, y, x0, lb, ub, m)
    for opts, host in ((None, False), ({"chunk": 50000}, False),
                       ({"h2d_chunks": 2, "prologue_rounds": 3}, True)):
        r1, served = solve(cm, kind, method, t, y, x0, lb, ub, m, options=opts, host=host)
        same_bits(r0, r1)
        assert served[0] >= 10, opts
    assert int((r0.status > 0).sum()) >= 0.99 * B


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["trf", "dogbox"])
def test_expdecay2_equals_library_callbacks(compiled, method):
    """Compiled ExpDecay2 'exact' and 'inlined' give the bits of the
    library's fused callbacks models.callbacks('ExpDecay2', 'exact')."""
    model = ExpDecay2()
    B = 4096
    _, y = model.make_data(B, seed=5)
    Y, X0 = cases.T(y, DEV), cases.T(np.tile(model.x0, (B, 1)), DEV)
    f0, j0 = models.callbacks("ExpDecay2", "exact")
    r0 = least_squares_batched(f0, X0, jac=j0, bounds=(model.lb, model.ub), method=method,
                               args=(PerProblem(Y),))
    for kind in ("exact", "inlined"):
        r1, _ = solve(compiled["ExpDecay2"], kind, method, model.t, y, model.x0,
                      model.lb, model.ub, model.m)
        same_bits(r0, r1)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["trf", "dogbox"])
def test_ratpoly5_equals_torch_callbacks(compiled, method):
    """RatPoly5 (+ - * / only): '2-point' and 'inlined-2-point' give the bits
    of the torch callbacks synthetic.RatPoly5.fun_t on the golden problems,
    and so meet the gates of the golden 2-point tests."""
    name = f"rat_{method}_2point"
    r0, z, trials = cases.run_golden_batched(None, DEV, name)
    m = int(json.loads(str(z["meta"]))["m"])
    model = RatPoly5(m)
    for kind in ("2-point", "inlined-2-point"):
        r1, _ = solve(compiled["RatPoly5"], kind, method, model.t, z["y"], model.x0,
                      model.lb, model.ub, m)
        same_bits(r0, r1)
        s = cases.summarize(r1, z, trials)
        obj = r1.obj_value.cpu().numpy()
        assert s["mask_eq"] >= 0.95 and s["status_eq"] >= 0.95 and s["nfev_eq"] >= 0.95, s
        assert float((np.abs(obj - z["obj"]) <= 1e-8 * z["obj"]).mean()) >= 0.95, s


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind", [("GaussPeak", "inlined-2-point"),
                                       ("GaussPeak", "inlined"),
                                       ("ThreePeak", "inlined")])
@pytest.mark.parametrize("method", ["trf", "dogbox"])
def test_against_oracle(compiled, name, kind, method):
    """Fresh problems against the oracle, with the gates of
    cases.check_random_small_vs_oracle: every cost within 1e-8, status,
    nfev, x (1e-8) and the active set identical for >= 99 % (2-point: the
    gates of cases.check_golden_fd_jac, >= 95 %)."""
    from oracle import blsq_oracle as orc
    f = REF[name][9]
    m = 128
    B = 100
    t, y, x0, lb, ub = problem_data(name, m, B, seed=1234)
    res, _ = solve(compiled[name], kind, method, t, y, x0, lb, ub, m)
    X, st, nf = res.x.cpu().numpy(), res.status.cpu().numpy(), res.nfev.cpu().numpy()
    ob, mk = res.obj_value.cpu().numpy(), res.active_mask.cpu().numpy()
    assert np.all(X >= lb) and np.all(X <= ub)
    fd = kind.endswith("2-point")
    exact = 0
    for b in range(B):
        fb = (lambda x, yb: f(x[None], t)[0] - yb)
        jb = "2-point" if fd else (lambda x, yb: _fd_free_jac(name, x, t))
        r = orc.least_squares(fb, x0, jac=jb, bounds=(lb, ub), method=method, args=(y[b],))
        assert abs(ob[b] - r.obj_value) <= 1e-8 * r.obj_value + 1e-18, b
        exact += (st[b] == r.status and nf[b] == r.nfev and
                  np.allclose(X[b], r.x, rtol=1e-8, atol=1e-9) and
                  np.array_equal(mk[b], np.asarray(r.active_mask)))
    assert exact >= (0.95 if fd else 0.99) * B, exact


def _fd_free_jac(name, x, t):
    """The analytic Jacobian of the reference models, NumPy."""
    if name == "GaussPeak":
        z = (t - x[1]) / x[2]
        e = np.exp(-0.5 * z * z)
        return np.stack([e, x[0] * e * z / x[2], x[0] * e * z * z / x[2],
                         np.ones_like(t), t, t * t], axis=1)
    cols = []
    for k in range(3):
        s = x[3 * k + 2]
        z = (t - x[3 * k + 1]) / s
        e = np.exp(-0.5 * z * z)
        cols += [e, x[3 * k] * e * z / s, x[3 * k] * e * z * z / s]
    return np.stack(cols + [np.ones_like(t), t], axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind,method", [("ExpDecay2", "inlined", "trf"),
                                              ("GaussPeak", "inlined-2-point", "dogbox"),
                                              ("ThreePeak", "inlined", "dogbox")])
def test_batch_permutation_and_subset(compiled, name, kind, method):
    """PerProblem data is indexed by problem id: a permuted batch or a
    subset gives each problem the bits it gets in the whole batch."""
    m = 96
    t, y, x0, lb, ub = problem_data(name, m, 512, seed=77)
    cm = compiled[name]
    r0, _ = solve(cm, kind, method, t, y, x0, lb, ub, m)
    perm = np.random.default_rng(3).permutation(512)
    for sel in (perm, np.arange(1, 512, 3)):
        r1, _ = solve(cm, kind, method, t, y[sel], x0, lb, ub, m)
        for fld in FIELDS:
            a = getattr(r0, fld).cpu().numpy()[sel]
            assert cases.bits(getattr(r1, fld).cpu().numpy(), a), fld


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["exact", "2-point"])
def test_rows_materialised(compiled, kind):
    """The materialised kinds take `rows`: each problem gets the bits of the
    dense solve of its first rows[b] residuals (same lane-group class);
    `rows` and `cols` with an inlined kind raise."""
    cm = compiled["ExpDecay2"]
    m, B = 64, 300
    t, y, x0, lb, ub = problem_data("ExpDecay2", m, B, seed=8)
    rows = np.where(np.arange(B) % 3 == 0, 40, m).astype(np.int32)
    fun, jac = cm.callbacks(kind, m=m)
    X0 = cases.T(np.tile(x0, (B, 1)), DEV)
    r = least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method="trf",
                              args=(PerProblem(cases.T(y, DEV)), cases.T(t, DEV)),
                              options={"rows": torch.as_tensor(rows, device=DEV)})
    for mr in (40, m):
        sel = np.nonzero(rows == mr)[0]
        rd, _ = solve(cm, kind, "trf", t[:mr], np.ascontiguousarray(y[sel, :mr]), x0, lb, ub,
                      mr)
        for fld in FIELDS:
            assert cases.bits(getattr(r, fld).cpu().numpy()[sel],
                              getattr(rd, fld).cpu().numpy()), (mr, fld)
    fun, jac = cm.callbacks("inlined", m=m)
    for key, val in (("rows", torch.as_tensor(rows, device=DEV)),
                     ("cols", torch.full((B,), 4, dtype=torch.int32, device=DEV))):
        with pytest.raises(ValueError, match="compiled into the linearisation"):
            least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method="trf",
                                  args=(PerProblem(cases.T(y, DEV)), cases.T(t, DEV)),
                                  options={key: val})
