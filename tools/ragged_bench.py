#!/usr/bin/env python
"""Ragged-batch benchmark, workload "C2-ragged": 10^6 ExpDecay2 fits (TRF,
rows-aware fused callbacks, width 64) where problem b observes the first
rows[b] samples of the shared grid, rows[b] uniform in 24..64 from a fixed
seed.  In the same process the same problems are solved with rows = 64 for
all (through the same rows path) as the dense reference point.

Per arm: fits/s and ms per solve (host clock around synchronised solves),
mean nfev, the mean time of the full-batch `linearise` launches (CUDA events,
a separate instrumented solve) and their GB/s on the algorithmic bytes
sum_b 8 rows_b (n+1) + 8 LS, as a fraction of the HBM peak bench.py uses.

    python tools/ragged_bench.py [--B 1000000] [--steps 5] [--warmup 2] [--out f.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bounded_lsq_b200 import PerProblem, least_squares_batched, models   # noqa: E402
from bounded_lsq_b200 import _lib as L                                    # noqa: E402
from bounded_lsq_b200.synthetic import ExpDecay2                          # noqa: E402


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (as bench.py)"


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:                      # noqa: BLE001
        info["power_limit"] = f"unknown ({e!r})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = L.get_lib()
    model = ExpDecay2()
    B, n, W = a.B, model.n, model.m
    _, ypool = model.make_data(min(B, 65536), seed=1)
    y = np.tile(ypool, (-(-B // len(ypool)), 1))[:B].copy()
    rows = np.random.default_rng(a.seed).integers(24, W + 1, B)
    y_rag = y.copy()
    y_rag[np.arange(W)[None, :] >= rows[:, None]] = np.nan    # never read
    X0 = torch.as_tensor(np.tile(model.x0, (B, 1)), device=dev)
    fun, jac = models.callbacks("ExpDecay2", "exact", rows=True)
    LS = lib.lin_record_size(n)
    peak, peak_src = hbm_peak()
    arms = {"C2-ragged": (y_rag, rows), "C2-rows64": (y, np.full(B, W))}
    data = {k: (torch.as_tensor(yy, device=dev),
                torch.as_tensor(rr, dtype=torch.int32, device=dev)) for k, (yy, rr) in arms.items()}

    def solve(k, **opts):
        yt, rt = data[k]
        return least_squares_batched(fun, X0, jac=jac, bounds=(model.lb, model.ub),
                                     method="trf", args=(PerProblem(yt), PerProblem(rt)),
                                     options=dict(rows=rt, **opts))

    out = {"workload": "C2-ragged", "B": B, "n": n, "width": W, "rows": "uniform 24..64",
           "seed": a.seed, "steps": a.steps, "warmup": a.warmup, "gpu": gpu_info(),
           "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "arms": {}}
    for k in arms:
        for _ in range(a.warmup):
            solve(k)
    torch.cuda.synchronize()
    # alternate the arms step by step: both see the same state of the machine
    times = {k: [] for k in arms}
    res = {}
    for _ in range(a.steps):
        for k in arms:
            t0 = time.perf_counter()
            res[k] = solve(k)
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    for k in arms:
        rt = data[k][1]
        timers = {}
        solve(k, timers=timers)
        torch.cuda.synchronize()
        ev = timers["linearise"]
        rmax = max(r for _, _, r in ev)
        full = [s.elapsed_time(e) for s, e, r in ev if r == rmax]
        lin_ms = sum(full) / len(full)
        byts = 8.0 * float(rt.sum().item()) * (n + 1) + 8.0 * LS * B
        gbs = byts / (lin_ms * 1e-3) / 1e9
        ms = float(np.median(times[k])) * 1e3
        r = res[k]
        out["arms"][k] = {
            "fits_per_s": B / (ms * 1e-3), "ms_per_step": ms,
            "ms_per_step_all": [t * 1e3 for t in times[k]],
            "mean_rows": float(rt.double().mean().item()),
            "mean_nfev": float(r.nfev.double().mean().item()),
            "success": float(r.success.double().mean().item()),
            "linearise_full_batch": {"launches": len(full), "avg_ms": lin_ms,
                                     "algorithmic_bytes": byts, "gbs": gbs,
                                     "fraction_of_hbm_peak": gbs / peak}}
    rg, dn = out["arms"]["C2-ragged"], out["arms"]["C2-rows64"]
    out["ragged_over_rows64"] = {
        "sum_rows": rg["mean_rows"] / dn["mean_rows"],
        "linearise_full_batch_ms": rg["linearise_full_batch"]["avg_ms"] /
        dn["linearise_full_batch"]["avg_ms"],
        "ms_per_step": rg["ms_per_step"] / dn["ms_per_step"]}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
