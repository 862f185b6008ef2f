#!/usr/bin/env python
"""Ragged-parameter benchmark, workload "C2-mixed": 10^6 fits of 1 to 4
exponential terms, f(t) = sum_k a_k exp(-b_k t) - y on m = 64 samples, with
n = 2, 4, 6, 8 parameters in equal shares (a fixed seed decides which
problem has how many), TRF with the analytic Jacobian in torch.

Two routes to the same fits, timed alternately in the same process (host
clock around synchronised solves, median over --steps):
  one batch    all 10^6 problems padded to n = 8, options={'cols': cols}; the
               unused terms are held at amplitude 0, so they add 0.0
  four dense   the same problems as four dense batches, one per n, solved
               one after another with callbacks of their own width
The outputs of the two routes must be bit-identical (checked on every field
and reported).  A third, instrumented solve of the one-batch route reports
per-segment kernel times from the `timers` events (linearise and round
launches of each segment; the graph tail is off there), and the launch and
round counts of both routes.  The card name and power limit are read in the
same process.

    python tools/ragged_cols_bench.py [--B 1000000] [--steps 5] [--warmup 2] [--out f.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bounded_lsq_b200 import PerProblem, least_squares_batched       # noqa: E402
from ragged_bench import gpu_info                                   # noqa: E402

M = 64
NMAX = 8
T_GRID = np.linspace(0.0, 4.0, M)


def callbacks(dev):
    t = torch.as_tensor(T_GRID, dtype=torch.float64, device=dev)

    def terms(X):
        # a_k exp(-b_k t) for the X.shape[1] // 2 terms of this width, summed
        # in a fixed order: a padded term (a_k = 0) adds exactly 0.0
        return [(X[:, 2 * k, None], torch.exp(-X[:, 2 * k + 1, None] * t[None, :]))
                for k in range(X.shape[1] // 2)]

    def fun(X, Y):
        f = None
        for a, e in terms(X):
            f = a * e if f is None else f + a * e
        return f - Y

    def jac(X, Y):
        cols = []
        for a, e in terms(X):
            cols += [e, -a * t[None, :] * e]
        return torch.stack(cols, dim=2)
    return fun, jac


def make_problems(B, seed):
    rng = np.random.default_rng(seed)
    K = rng.permutation(np.repeat(np.arange(1, 5), -(-B // 4))[:B])    # terms per problem
    a = rng.uniform(0.5, 2.0, (B, 4))
    b = np.sort(rng.uniform(0.2, 3.0, (B, 4)), axis=1)
    y = np.zeros((B, M))
    for k in range(4):
        on = (k < K)[:, None]
        y += np.where(on, a[:, k, None] * np.exp(-b[:, k, None] * T_GRID[None, :]), 0.0)
    y += 0.01 * rng.standard_normal((B, M))
    x0 = np.zeros((B, NMAX))
    for k in range(4):
        on = k < K
        x0[:, 2 * k] = np.where(on, 1.0, 0.0)          # held terms: amplitude 0
        x0[:, 2 * k + 1] = 0.5 + k
    lb = np.tile([0.0, 0.01], 4)
    ub = np.tile([10.0, 10.0], 4)
    return 2 * K, y, x0, lb, ub


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2025)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    B = a.B
    cols, y, x0, lb, ub = make_problems(B, a.seed)
    fun, jac = callbacks(dev)
    Y = torch.as_tensor(y, device=dev)
    X0 = torch.as_tensor(x0, device=dev)
    LB, UB = torch.as_tensor(lb, device=dev), torch.as_tensor(ub, device=dev)
    C = torch.as_tensor(cols, dtype=torch.int32, device=dev)
    groups = [(N, np.nonzero(cols == N)[0]) for N in (2, 4, 6, 8)]
    dense = [(N, torch.as_tensor(sel, device=dev), Y[sel].contiguous(),
              X0[sel, :N].contiguous()) for N, sel in groups]

    def one_batch(**opts):
        return least_squares_batched(fun, X0, jac=jac, bounds=(LB, UB), method="trf",
                                     args=(PerProblem(Y),), options=dict(cols=C, **opts))

    def four_dense():
        return [(sel, least_squares_batched(fun, x0n, jac=jac, bounds=(LB[:N], UB[:N]),
                                            method="trf", args=(PerProblem(yn),)))
                for N, sel, yn, x0n in dense]

    routes = {"one_batch_cols": one_batch, "four_dense_batches": four_dense}
    for _ in range(a.warmup):
        for f in routes.values():
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in routes}
    res = {}
    for _ in range(a.steps):
        for k, f in routes.items():
            t0 = time.perf_counter()
            res[k] = f()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)

    # the outputs of the two routes, bit for bit
    r1 = res["one_batch_cols"]
    identical = {}
    for fld in ("x", "obj_value", "optimality", "status", "nfev", "njev", "active_mask"):
        ok = True
        for sel, r in res["four_dense_batches"]:
            N = r.x.shape[1] if r[fld].dim() == 2 else None
            v1 = r1[fld][sel] if N is None else r1[fld][sel, :N]
            ok = ok and torch.equal(v1, r[fld])
            if N is not None and fld == "x":
                ok = ok and torch.equal(r1.x[sel, N:], X0[sel, N:])
        identical[fld] = bool(ok)

    timers = {}
    one_batch(timers=timers)
    torch.cuda.synchronize()
    seg = {}
    for N, kinds in sorted(timers.get("segments", {}).items()):
        seg[str(N)] = {}
        for kind in ("linearise", "round"):
            ev = kinds.get(kind, [])
            ms = [s.elapsed_time(e) for s, e, _ in ev]
            rmax = max((r for _, _, r in ev), default=0)
            full = [t for t, (_, _, r) in zip(ms, ev) if r == rmax]
            seg[str(N)][kind] = {"launches": len(ms), "total_ms": sum(ms),
                                 "full_batch_running": rmax,
                                 "full_batch_avg_ms": sum(full) / len(full) if full else None}
    cb = timers.get("callbacks", [])
    ms = {k: float(np.median(v)) * 1e3 for k, v in times.items()}
    out = {
        "workload": "C2-mixed", "B": B, "m": M, "n_padded": NMAX,
        "cols": "2, 4, 6, 8 in equal shares", "method": "trf", "jac": "analytic (torch)",
        "seed": a.seed, "steps": a.steps, "warmup": a.warmup, "gpu": gpu_info(),
        "ms_per_solve": ms,
        "ms_per_solve_all": {k: [t * 1e3 for t in v] for k, v in times.items()},
        "fits_per_s": {k: B / (v * 1e-3) for k, v in ms.items()},
        "one_batch_over_four_dense": ms["one_batch_cols"] / ms["four_dense_batches"],
        "rounds": {"one_batch_cols": int(r1.rounds),
                   "four_dense_batches": [int(r.rounds) for _, r in res["four_dense_batches"]]},
        "kernel_launches": {"one_batch_cols": int(r1.kernel_launches),
                            "four_dense_batches": [int(r.kernel_launches)
                                                   for _, r in res["four_dense_batches"]]},
        "mean_nfev": float(r1.nfev.double().mean().item()),
        "success": float(r1.success.double().mean().item()),
        "bit_identical": identical,
        "instrumented_one_batch": {
            "note": "CUDA events around every launch; the graph tail is off",
            "callbacks_ms": sum(s.elapsed_time(e) for s, e, _ in cb),
            "segments": seg},
    }
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if not all(identical.values()):
        sys.exit("the two routes differ: " + json.dumps(identical))


if __name__ == "__main__":
    main()
