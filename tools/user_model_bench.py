"""Compiled user models (models.compile_model) against the library's routes.

C2 (1M ExpDecay2 fits, TRF, m = 64): the compiled 'inlined' kind against the
shipped models.callbacks('ExpDecay2', 'inlined'), the fused 'exact'
callbacks and the torch callbacks.  C3 (one 1M-problem chunk of GaussPeak,
dogbox, m = 128): compiled 'inlined-2-point' against the fused
models.callbacks('GaussPeak', '2-point') and the compiled '2-point'.  W11
(three Gaussian peaks, n = 11, m = 128, TRF): compiled 'inlined' against
'exact'.  Per route: ms per solve (device events over --steps solves after
--warmup, routes alternated), fits/s and the full-batch linearise time from a
separate timed solve.  Also the cold and warm compile times and the bit
identity of the routes that must agree.  The card's name and power limit are
read in the same run.

    python tools/user_model_bench.py --out user_model_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from bounded_lsq_b200 import PerProblem, least_squares_batched, models   # noqa: E402
from bounded_lsq_b200.batched import summarize_timers                     # noqa: E402
from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak                # noqa: E402
import test_user_models as ref                                             # noqa: E402

DEV = torch.device("cuda:0")
FIELDS = ("x", "obj_value", "status", "nfev", "njev", "active_mask")


def T(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device=DEV)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout
    return q.strip().splitlines()[0] if q.strip() else "unknown"


def run(route, method, x0, lb, ub, B, options=None):
    fun, jac, args = route
    X0 = T(np.tile(x0, (B, 1)))
    return least_squares_batched(fun, X0, jac=jac, bounds=(lb, ub), method=method,
                                 args=args, options=options or {})


def bench(routes, method, x0, lb, ub, B, steps, warmup):
    out = {}
    for name, r in routes.items():
        for _ in range(warmup):
            run(r, method, x0, lb, ub, B)
        out[name] = dict(ms=[])
    for _ in range(steps):                     # alternate the routes
        for name, r in routes.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = run(r, method, x0, lb, ub, B)
            e1.record()
            torch.cuda.synchronize()
            out[name]["ms"].append(e0.elapsed_time(e1))
            out[name]["res"] = res
    results = {}
    for name, r in routes.items():
        ms = out[name]["ms"]
        timers = {}
        run(r, method, x0, lb, ub, B, options={"timers": timers})
        torch.cuda.synchronize()
        lin = summarize_timers(timers).get("linearise", {})
        res = out[name]["res"]
        results[name] = dict(
            ms_per_solve=float(np.median(ms)), ms_all=[round(v, 3) for v in ms],
            fits_per_s=B / (np.median(ms) / 1e3),
            linearise_total_ms=lin.get("total_ms"),
            linearise_full_batch=lin.get("full_batch"),
            rounds=res.rounds, kernel_launches=res.kernel_launches,
            converged=int((res.status > 0).sum()))
    return results, {k: v["res"] for k, v in out.items()}


def same(r0, r1):
    return all(np.asarray(getattr(r0, f).cpu()).tobytes() ==
               np.asarray(getattr(r1, f).cpu()).tobytes() for f in FIELDS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rec = dict(card=card(), torch=torch.__version__)

    with tempfile.TemporaryDirectory() as cache:
        t0 = time.perf_counter()
        ed = models.compile_model(ref.EXPDECAY2, cache_dir=cache)
        t1 = time.perf_counter()
        models.compile_model(ref.EXPDECAY2, cache_dir=cache)
        t2 = time.perf_counter()
        gp = models.compile_model(ref.GAUSSPEAK, "GaussPeak", cache_dir=cache)
        t3 = time.perf_counter()
        w11 = models.compile_model(ref.THREEPEAK, cache_dir=cache)
        t4 = time.perf_counter()
    rec["compile_s"] = dict(expdecay2_cold=t1 - t0, expdecay2_warm=t2 - t1,
                            gausspeak_cold=t3 - t2, threepeak_cold=t4 - t3)

    # C2
    m2 = ExpDecay2()
    B = 1_000_000
    _, y = m2.make_data(B, seed=0)
    Y, t = T(y), T(m2.t)
    f_s, j_s = models.callbacks("ExpDecay2", "inlined")
    f_e, j_e = models.callbacks("ExpDecay2", "exact")
    f_c, j_c = ed.callbacks("inlined", m=m2.m)
    routes = {"compiled_inlined": (f_c, j_c, (PerProblem(Y), t)),
              "shipped_inlined": (f_s, j_s, (PerProblem(Y),)),
              "fused_exact": (f_e, j_e, (PerProblem(Y),)),
              "torch": (m2.fun_t, m2.jac_t, (PerProblem(Y),))}
    res, sol = bench(routes, "trf", m2.x0, m2.lb, m2.ub, B, a.steps, a.warmup)
    rec["c2"] = dict(B=B, m=m2.m, method="trf", routes=res, bits_compiled_eq_shipped=same(
        sol["compiled_inlined"], sol["shipped_inlined"]),
        bits_compiled_eq_fused_exact=same(sol["compiled_inlined"], sol["fused_exact"]))
    del Y, sol, routes
    torch.cuda.empty_cache()

    # C3: one 1M-problem chunk
    m3 = GaussPeak()
    _, y = m3.make_data(B, seed=1)
    Y, t = T(y), T(m3.t)
    f_g, j_g = models.callbacks("GaussPeak", "2-point")
    f_i, j_i = gp.callbacks("inlined-2-point", m=m3.m)
    f_m, j_m = gp.callbacks("2-point", m=m3.m)
    routes = {"compiled_inlined_2point": (f_i, j_i, (PerProblem(Y), t)),
              "fused_2point": (f_g, j_g, (PerProblem(Y),)),
              "compiled_2point": (f_m, j_m, (PerProblem(Y), t))}
    res, sol = bench(routes, "dogbox", m3.x0, m3.lb, m3.ub, B, a.steps, a.warmup)
    rec["c3"] = dict(B=B, m=m3.m, method="dogbox", routes=res,
                     bits_inlined_eq_materialised=same(sol["compiled_inlined_2point"],
                                                       sol["compiled_2point"]))
    del Y, sol, routes
    torch.cuda.empty_cache()

    # W11
    Bw, mw = 250_000, 128
    tw, yw, x0, lb, ub = ref.problem_data("ThreePeak", mw, Bw, seed=2)
    Y, t = T(yw), T(tw)
    f_i, j_i = w11.callbacks("inlined", m=mw)
    f_x, j_x = w11.callbacks("exact", m=mw)
    routes = {"compiled_inlined": (f_i, j_i, (PerProblem(Y), t)),
              "compiled_exact": (f_x, j_x, (PerProblem(Y), t))}
    res, sol = bench(routes, "trf", x0, lb, ub, Bw, a.steps, a.warmup)
    rec["w11"] = dict(B=Bw, m=mw, method="trf", routes=res,
                      bits_inlined_eq_exact=same(sol["compiled_inlined"], sol["compiled_exact"]))

    s = json.dumps(rec, indent=1, default=float)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
