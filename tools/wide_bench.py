#!/usr/bin/env python
"""Batched mode at 9 <= n <= 16: workloads W11 and W16.

W11: 10^6 fits of three Gaussian peaks on a linear baseline, n = 11,
t = linspace(-5, 5, 128), m = 128.  Parameters per peak (A, mu, sigma), then
c0, c1.  Truth: A ~ U(1, 3), mu = (-2.5, 0, 2.5) + U(-0.3, 0.3),
sigma ~ U(0.4, 0.9), c0 ~ U(0, 1), c1 ~ U(-0.1, 0.1), noise 0.01, seed 0.
x0: A = 2, mu nominal, sigma = 0.6, c0 = 0.5, c1 = 0.  Bounds: A in [0, 5],
mu within +-1.2 of nominal, sigma in [0.1, 2], c0 in [-1, 2], c1 in [-1, 1].
W16: five peaks plus a constant, n = 16, t = linspace(-5, 5, 256), m = 256,
2.5 10^5 fits: nominal centres (-4, -2, 0, 2, 4), mu within +-0.8 of them,
sigma ~ U(0.3, 0.6) (x0 0.45), otherwise as W11 with c1 dropped.

Records: TRF with the analytic Jacobian and dogbox with 2-point, per workload.
Per record: fits/s with the data resident in HBM (host clock around
synchronised solves, median of --steps after --warmup); the full-batch
`linearise` launches (CUDA events of the driver's timers) per 10^6 problems
against the algorithmic bytes 8 m (n+1) + 8 LS per problem; the round kernel
instances per 10^6 problems from a torch.profiler run of its own (TRF MODE 1
and MODE 2 separately); kernel launches per solve; parity of a --sample fit
sample against the oracle; the oracle on all host cores and a Python loop of
single-problem least_squares calls (tall route) on --loop-fits fits.

    python tools/wide_bench.py [--steps 3] [--warmup 1] [--sample 2048]
                               [--loop-fits 100] [--out f.json]
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bounded_lsq_b200 import PerProblem, least_squares, least_squares_batched  # noqa: E402
from bounded_lsq_b200 import _lib as L                                          # noqa: E402
from ragged_bench import gpu_info                                               # noqa: E402

HBM_MEASURED_GBS = 6535.0          # DESIGN §7, measured copy bandwidth of one B200


class Peaks:
    """K Gaussian peaks (A, mu, sigma) plus a polynomial baseline of `nb`
    coefficients on t = linspace(-5, 5, m)."""

    def __init__(self, name, K, nb, m, B, centres, dmu, sig, sig0, seed=0):
        self.name, self.K, self.nb, self.m, self.B = name, K, nb, m, B
        self.n = 3 * K + nb
        self.t = np.linspace(-5.0, 5.0, m)
        c = np.asarray(centres, dtype=float)
        rng = np.random.default_rng(seed)
        xt = np.empty((B, self.n))
        xt[:, 0:3 * K:3] = rng.uniform(1, 3, (B, K))
        xt[:, 1:3 * K:3] = c + rng.uniform(-0.3, 0.3, (B, K))
        xt[:, 2:3 * K:3] = rng.uniform(*sig, (B, K))
        xt[:, 3 * K] = rng.uniform(0, 1, B)
        if nb > 1:
            xt[:, 3 * K + 1] = rng.uniform(-0.1, 0.1, B)
        self.xt = xt
        self.y = np.empty((B, m))
        for s in range(0, B, 65536):
            self.y[s:s + 65536] = self.fun_np_batch(xt[s:s + 65536])
        self.y += 0.01 * rng.standard_normal((B, m))
        x0 = np.zeros(self.n)
        x0[0:3 * K:3], x0[1:3 * K:3], x0[2:3 * K:3] = 2.0, c, sig0
        x0[3 * K] = 0.5
        lb, ub = np.empty(self.n), np.empty(self.n)
        lb[0:3 * K:3], ub[0:3 * K:3] = 0.0, 5.0
        lb[1:3 * K:3], ub[1:3 * K:3] = c - dmu, c + dmu
        lb[2:3 * K:3], ub[2:3 * K:3] = 0.1, 2.0
        lb[3 * K], ub[3 * K] = -1.0, 2.0
        if nb > 1:
            lb[3 * K + 1], ub[3 * K + 1] = -1.0, 1.0
        self.x0, self.lb, self.ub = x0, lb, ub

    def fun_np_batch(self, X):
        K, t = self.K, self.t
        out = X[:, 3 * K:3 * K + 1] + (X[:, 3 * K + 1:3 * K + 2] * t if self.nb > 1 else 0.0)
        for k in range(K):
            A, mu, s = X[:, 3 * k:3 * k + 1], X[:, 3 * k + 1:3 * k + 2], X[:, 3 * k + 2:3 * k + 3]
            out = out + A * np.exp(-0.5 * ((t - mu) / s) ** 2)
        return out

    def fun_np(self, x, yb):
        return self.fun_np_batch(x[None])[0] - yb

    def jac_np(self, x, yb):
        return self._jac(x[None], np, self.t)[0]

    def _jac(self, X, xp, t):
        K = self.K
        cols = []
        for k in range(K):
            A, mu, s = X[:, 3 * k:3 * k + 1], X[:, 3 * k + 1:3 * k + 2], X[:, 3 * k + 2:3 * k + 3]
            u = (t - mu) / s
            e = xp.exp(-0.5 * u * u)
            cols += [e, A * e * u / s, A * e * u * u / s]
        cols.append(xp.ones_like(cols[0]))
        if self.nb > 1:
            cols.append(xp.ones_like(cols[0]) * t)
        return xp.stack(cols, axis=-1) if xp is np else xp.stack(cols, dim=-1)

    def torch_callbacks(self, dev):
        K = self.K
        t = torch.as_tensor(self.t, device=dev)

        def fun(X, Y):
            out = X[:, 3 * K:3 * K + 1] + (X[:, 3 * K + 1:3 * K + 2] * t if self.nb > 1 else 0.0)
            for k in range(K):
                A, mu, s = X[:, 3 * k:3 * k + 1], X[:, 3 * k + 1:3 * k + 2], X[:, 3 * k + 2:3 * k + 3]
                out = out + A * torch.exp(-0.5 * ((t - mu) / s) ** 2)
            return out - Y

        def jac(X, Y):
            return self._jac(X, torch, t)
        return fun, jac


def W11(B):
    return Peaks("W11", 3, 2, 128, B, (-2.5, 0.0, 2.5), 1.2, (0.4, 0.9), 0.6)


def W16(B):
    return Peaks("W16", 5, 1, 256, B, (-4.0, -2.0, 0.0, 2.0, 4.0), 0.8, (0.3, 0.6), 0.45)


_W = None


def _oracle_one(args):
    from oracle import blsq_oracle as orc
    b, method, jac = args
    w = _W
    r = orc.least_squares(w.fun_np, w.x0, jac=w.jac_np if jac == "exact" else jac,
                          bounds=(w.lb, w.ub), method=method, args=(w.y[b],))
    return b, r.status, r.nfev, r.x, r.obj_value


def _pool_init(w):
    global _W
    _W = w


def kernel_profile(solve):
    """Device time per kernel family over one solve (torch.profiler, a run of
    its own): total ms and launches, and the time of the first launch."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        solve()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
    fam = {}
    for e in ev:
        nm = e.name
        if "lin_kernel" in nm:
            k = "lin_kernel"
        elif "round_kernel" in nm:
            # round_kernel<N, METHOD, MODE, ROWS>
            args = nm.split("round_kernel<")[1].split(">")[0].split(",")
            k = f"round_kernel METHOD {args[1].strip()} MODE {args[2].strip()}"
        else:
            continue
        d = e.time_range.elapsed_us() / 1e3
        f = fam.setdefault(k, {"launches": 0, "total_ms": 0.0, "first_ms": None})
        f["launches"] += 1
        f["total_ms"] += d
        if f["first_ms"] is None:
            f["first_ms"] = d
    return fam


def run_record(w, method, jac, a, dev):
    B, n, m = w.B, w.n, w.m
    lib = L.get_lib()
    fun, jacf = w.torch_callbacks(dev)
    X0 = torch.as_tensor(np.tile(w.x0, (B, 1)), device=dev)
    Y = torch.as_tensor(w.y, device=dev)
    lb, ub = torch.as_tensor(w.lb, device=dev), torch.as_tensor(w.ub, device=dev)

    def solve(**opts):
        return least_squares_batched(fun, X0, jac=jacf if jac == "exact" else jac,
                                     bounds=(lb, ub), method=method,
                                     args=(PerProblem(Y),), options=opts)
    for _ in range(a.warmup):
        solve()
    torch.cuda.synchronize()
    times = []
    for _ in range(a.steps):
        t0 = time.perf_counter()
        res = solve()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    ms = float(np.median(times)) * 1e3
    timers = {}
    solve(timers=timers)
    torch.cuda.synchronize()
    LS = lib.lin_record_size(n)
    lin = [(s.elapsed_time(e), r) for s, e, r in timers["linearise"]]
    full = [t for t, r in lin if r == B]
    lin_ms = float(np.mean(full))
    byts = B * (8.0 * m * (n + 1) + 8.0 * LS)
    rnd = [(s.elapsed_time(e), r) for s, e, r in timers["round"]]
    rfull = [t for t, r in rnd if r == B]
    prof = kernel_profile(solve)
    for f in prof.values():
        f["first_ms_per_1e6"] = f["first_ms"] * 1e6 / B
    rec = {
        "workload": w.name, "method": method, "jac": jac, "B": B, "n": n, "m": m,
        "fits_per_s": B / (ms * 1e-3), "ms_per_solve": ms,
        "ms_per_solve_all": [t * 1e3 for t in times],
        "rounds": int(res.rounds), "kernel_launches_per_solve": int(res.kernel_launches),
        "mean_nfev": float(res.nfev.double().mean().item()),
        "success": float(res.success.double().mean().item()),
        "linearise_full_batch": {
            "launches": len(full), "ms_per_1e6": lin_ms * 1e6 / B,
            "algorithmic_bytes_per_problem": byts / B,
            "gbs": byts / (lin_ms * 1e-3) / 1e9,
            "fraction_of_measured_6535_gbs": byts / (lin_ms * 1e-3) / 1e9 / HBM_MEASURED_GBS},
        "round_full_batch_events": {"launches": len(rfull),
                                    "ms_per_1e6": float(np.mean(rfull)) * 1e6 / B
                                    if rfull else None},
        "kernels_profiled": prof,
    }
    # the round kernel's share of the device time of the kernels above
    lin_tot = prof.get("lin_kernel", {}).get("total_ms", 0.0)
    rnd_tot = sum(v["total_ms"] for k, v in prof.items() if k.startswith("round_kernel"))
    rec["round_share_of_lin_plus_round"] = rnd_tot / max(lin_tot + rnd_tot, 1e-12)
    # parity on a sample against the oracle, which also times the oracle on
    # all host cores
    S = min(a.sample, B)
    idx = np.random.default_rng(1).choice(B, S, replace=False)
    ncpu = os.cpu_count() or 1
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(ncpu, initializer=_pool_init, initargs=(w,)) as pool:
        refs = pool.map(_oracle_one, [(int(b), method, jac) for b in idx], chunksize=8)
    t_or = time.perf_counter() - t0
    st, nf = res.status.cpu().numpy(), res.nfev.cpu().numpy()
    X, ob = res.x.cpu().numpy(), res.obj_value.cpu().numpy()
    eq_st = eq_nf = 0
    xr = cr = 0.0
    for b, rs, rn, rx, ro in refs:
        eq_st += int(st[b] == rs)
        eq_nf += int(nf[b] == rn)
        xr = max(xr, float(np.abs(X[b] - rx).max() / max(np.abs(rx).max(), 1e-300)))
        cr = max(cr, abs(float(ob[b]) - ro) / max(ro, 1e-300))
    rec["parity"] = {"sample": S, "status_equal_pct": 100.0 * eq_st / S,
                     "nfev_equal_pct": 100.0 * eq_nf / S, "max_rel_x": xr, "max_rel_cost": cr}
    rec["oracle_all_host_cores"] = {"cores": ncpu, "fits": S, "fits_per_s": S / t_or}
    # a Python loop of least_squares calls: the route a user has today
    f1, j1 = w.torch_callbacks(dev)
    done = 0
    t0 = time.perf_counter()
    for b in idx[:a.loop_fits]:
        yb = Y[int(b)]
        least_squares(lambda x: f1(x[None], yb[None])[0], torch.as_tensor(w.x0, device=dev),
                      jac=(lambda x: j1(x[None], yb[None])[0]) if jac == "exact" else jac,
                      bounds=(lb, ub), method=method)
        done += 1
        if time.perf_counter() - t0 > a.loop_budget_s:
            break
    torch.cuda.synchronize()
    rec["python_loop_tall"] = {"fits": done, "fits_per_s": done / (time.perf_counter() - t0)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B11", type=int, default=1_000_000)
    ap.add_argument("--B16", type=int, default=250_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sample", type=int, default=2048)
    ap.add_argument("--loop-fits", type=int, default=100)
    ap.add_argument("--loop-budget-s", type=float, default=60.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info(), "records": []}
    for w in (W11(a.B11), W16(a.B16)):
        for method, jac in (("trf", "exact"), ("dogbox", "2-point")):
            rec = run_record(w, method, jac, a, dev)
            print(json.dumps(rec), flush=True)
            out["records"].append(rec)
    out["gpu_after"] = gpu_info()
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
            fh.write("\n")


if __name__ == "__main__":
    main()
