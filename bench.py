#!/usr/bin/env python
"""Headline benchmark: bounded fits solved per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4]
    python bench.py --impl reference ...     # CPU arm (oracle port, all cores)
    python bench.py ... --dump-outputs DIR    # also write the results as .npy

BASELINE.json's metric has two halves.  The line's own metric/value is the
first (batched fits/s, workload c2 = configs[1]); the default run also measures
the second (TRF iterations/s of ONE tall problem, m=16M, n=64 = configs[3],
rows sharded over the GPUs) and attaches that complete record as "tall".
`--workload c4` makes the tall workload the line itself.

A *step* is one complete batched solve of the workload: every problem is taken
from x0 to termination by the lock-step driver (user callbacks in PyTorch +
the two CUDA kernels per round behind include/blsq.h).

  value  fits/s with the data (y, x0, bounds) already resident in HBM
  e2e    fits/s through the public API with HOST buffers: pinned y/x0 are
         copied to the device and x/status/cost copied back inside the timing
  roofline  the HBM-bound linearisation kernel (QR of [J | f] per problem):
         algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json
  cpu_baseline  the oracle (NumPy port of the reference) on the host cores,
         bounded sample of the same workload; parity_vs_gpu = the same fits
         solved on the GPU and compared with the oracle's results

With N > 1 (torchrun) the problems are split by index, no collective on the
data path ("weak": per-GPU batch fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION; this script's
# stdout is ONE JSON line
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"      # (also overrides an /etc/nccl.conf setting)

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(desc="batched TRF: 1M bounded 4-param exponential-decay fits, "
                    "m=64, analytic Jacobian", model="ExpDecay2", B=1_000_000,
               method="trf", jac="exact", n=4, m=64, prologue_rounds=7),
    # BASELINE.json configs[2] (10M problems; 61 GB of residual evaluations
    # per FD sweep, so the per-GPU batch is processed in chunks)
    "c3": dict(desc="batched dogbox: 10M bounded 6-param Gaussian-peak fits, "
                    "m=128, 2-point Jacobian", model="GaussPeak", B=10_000_000,
               method="dogbox", jac="2-point", n=6, m=128, chunk=1_000_000,
               prologue_rounds=2),
    # BASELINE.json configs[3]: one tall problem, rows sharded over the GPUs
    "c4": dict(desc="tall single problem: m=16M rows, n=64, bounded "
                    "linear+exponential model, TRF, row-sharded Cholesky QR on "
                    "FP64 tensor cores", kind="tall", m=1 << 24, n=64, method="trf"),
    # BASELINE.json configs[4]: 8-GPU configuration (12.5M rows = 51 GB per
    # GPU); lb = 0 puts half of the U(-1, 1) truth values outside the bounds
    "c5": dict(desc="tall single problem: m=100M rows, n=256, half the bounds "
                    "active, row-sharded across the GPUs", kind="tall",
               m=100_000_000, n=256, method="trf", lb=0.0, no_e2e=True),
}


def _model(name):
    from bounded_lsq_b200 import synthetic
    return getattr(synthetic, name)()


# ------------------------------------------------------------ CPU arm -----

def _cpu_worker(job):
    name, method, jac, seed, count = job
    from oracle import blsq_oracle as orc
    model = _model(name)
    _, y = model.make_data(count, seed=seed)
    t0 = time.perf_counter()
    nfev = 0
    res = []
    for b in range(count):
        if jac == "exact":
            r = orc.least_squares(model.fun_np, model.x0, jac=model.jac_np,
                                  bounds=(model.lb, model.ub), method=method,
                                  args=(y[b],))
        else:
            r = orc.least_squares(model.fun_np, model.x0, jac="2-point",
                                  bounds=(model.lb, model.ub), method=method,
                                  args=(y[b],))
        nfev += r.nfev
        res.append((r.x, r.status, r.nfev, r.obj_value))
    return count, nfev, time.perf_counter() - t0, res


def _cpu_worker_init():
    # one BLAS thread per worker process: the fits are tiny (68 x 4 SVDs) and
    # the parallelism is over problems.  (Environment variables would have to
    # be set before numpy is imported; threadpoolctl works at any time.)
    try:
        from threadpoolctl import threadpool_limits
        _cpu_worker_init.limit = threadpool_limits(limits=1)
    except Exception:
        pass
    from oracle import blsq_oracle  # noqa: F401


_CPU_POOL = {}


def _close_cpu_pools():
    for pool in _CPU_POOL.values():
        pool.terminate()
        pool.join()
    _CPU_POOL.clear()


import atexit  # noqa: E402
atexit.register(_close_cpu_pools)


def _cpu_pool(cores):
    """ONE worker pool per process, created and warmed outside every timed
    region.  The parent imports the model module (and with it torch) before
    the fork, so no worker pays an import inside a measurement."""
    import multiprocessing as mp
    pool = _CPU_POOL.get(cores)
    if pool is None:
        from oracle import blsq_oracle  # noqa: F401
        from bounded_lsq_b200 import synthetic  # noqa: F401
        pool = mp.get_context("fork").Pool(cores, initializer=_cpu_worker_init)
        _CPU_POOL[cores] = pool
        # warm-up: every worker solves a few fits
        pool.map(_cpu_worker, [("ExpDecay2", "trf", "exact", 1, 2)] * (2 * cores))
    return pool


def cpu_fits_per_second(w, per_core, cores=None, seed0=1000):
    """Oracle (NumPy port of the reference) over all host cores; the timed
    region is the pool.map over the jobs and nothing else."""
    cores = cores or os.cpu_count() or 1
    pool = _cpu_pool(cores)
    # two jobs per core: a core that finishes early picks up another one
    half = max(1, per_core // 2)
    jobs = [(w["model"], w["method"], w["jac"], seed0 + c, half)
            for c in range(2 * cores)]
    t0 = time.perf_counter()
    out = pool.map(_cpu_worker, jobs, chunksize=1)
    wall = time.perf_counter() - t0
    fits = sum(o[0] for o in out)
    cpu_fits_per_second.last = dict(
        seeds=[j[3] for j in jobs], per_core=half,
        results=[r for o in out for r in o[3]])
    return fits / wall, cores, fits, sum(o[1] for o in out) / fits


def gpu_parity_of_cpu_sample(w, fun, jac, lb, ub, dev):
    """SURVEY 8(d) "parity gates run with every measurement": the fits the
    cpu_baseline leg just solved with the oracle, solved again on the GPU."""
    import torch
    from bounded_lsq_b200 import least_squares_batched, PerProblem
    last = getattr(cpu_fits_per_second, "last", None)
    if not last:
        return None
    model = _model(w["model"])
    y = np.concatenate([model.make_data(last["per_core"], seed=sd)[1]
                        for sd in last["seeds"]])
    B = y.shape[0]
    res = least_squares_batched(
        fun, torch.as_tensor(np.tile(model.x0, (B, 1)), device=dev), jac=jac,
        bounds=(lb, ub), method=w["method"],
        args=(PerProblem(torch.as_tensor(y, device=dev)),))
    xr = np.array([r[0] for r in last["results"]])
    st = np.array([r[1] for r in last["results"]])
    nf = np.array([r[2] for r in last["results"]])
    ob = np.array([r[3] for r in last["results"]])
    x = res.x.cpu().numpy()
    return {
        "fits": int(B),
        "status_equal": float((res.status.cpu().numpy() == st).mean()),
        "nfev_equal": float((res.nfev.cpu().numpy() == nf).mean()),
        "x_rel_max": float((np.abs(x - xr).max(1) / np.abs(xr).max(1)).max()),
        "obj_rel_max": float((np.abs(res.obj_value.cpu().numpy() - ob) / ob).max()),
        "note": "GPU path vs the oracle on the cpu_baseline sample; the gates "
                "(1e-8 on x / cost, equal status) are enforced in tests/",
    }


# ------------------------------------------------------------ outputs -----

# --dump-outputs keeps under 64 MB for every workload: at most this many
# batched problems and tall rows, a fixed seeded sample of the larger outputs
DUMP_PROBLEMS = 32768
DUMP_ROWS = 8192


def _sample(total, k):
    """Sorted seeded sample of k of range(total); all of it when total <= k."""
    if total <= k:
        return np.arange(total)
    return np.sort(np.random.default_rng(0).choice(total, k, replace=False))


def write_outputs(out_dir, prefix, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if hasattr(a, "cpu"):
            a = a.cpu().numpy()
        np.save(os.path.join(out_dir, prefix + name + ".npy"),
                np.asarray(a, dtype=np.float64))


def dump_batched(out_dir, prefix, outs, chunk, B):
    """Every per-problem field least_squares_batched returned in the last
    timed step, for a seeded sample of the problems."""
    import torch
    idx = _sample(B, DUMP_PROBLEMS)
    arrays = {"problem_index": idx}
    for key in ("x", "obj_value", "optimality", "active_mask", "status",
                "nfev", "njev", "fun"):
        parts = []
        for c, o in enumerate(outs):
            c0 = c * chunk
            sel = idx[(idx >= c0) & (idx < c0 + o.x.shape[0])] - c0
            parts.append(o[key][torch.as_tensor(sel, device=o.x.device)].cpu())
        arrays[key] = torch.cat(parts)
    write_outputs(out_dir, prefix, arrays)


def dump_tall(out_dir, prefix, res):
    """The result of the last timed tall solve: x and the scalars whole, the
    residual and the Jacobian on a seeded sample of the rows."""
    import torch
    rows = _sample(res.fun.shape[0], DUMP_ROWS)
    r = torch.as_tensor(rows, device=res.fun.device)
    write_outputs(out_dir, prefix, {
        "x": res.x, "active_mask": res.active_mask, "obj_value": res.obj_value,
        "optimality": res.optimality, "status": res.status, "nfev": res.nfev,
        "njev": res.njev, "row_index": rows, "fun": res.fun[r], "jac": res.jac[r]})


def static_config(w, B, chunk, callbacks=None):
    """The workload description both arms print (run-dependent values are
    added to it by the arm that measured them)."""
    c = {"workload": w["desc"], "problems_per_gpu": B, "chunk": chunk,
         "method": w["method"], "jac": w["jac"], "n": w["n"], "m": w["m"]}
    if callbacks is not None:
        c["callbacks"] = callbacks
    return c


def run_reference_arm(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # a step is a bounded sample: ~1 s of CPU work per core (C2: 360 fits/s/
    # core, SURVEY section 6), the whole --steps K run a few minutes at most
    per_core = 256 if w["jac"] == "exact" else 96
    _cpu_pool(cores)
    for _ in range(min(args.warmup, 2)):
        cpu_fits_per_second(w, 16, cores)
    fits = 0
    nfev = 0.0
    wall = 0.0
    for k in range(args.steps):
        v, c, f, nf = cpu_fits_per_second(w, per_core, cores, seed0=2000 + 97 * k)
        fits += f
        nfev += nf * f
        wall += f / v
    value = fits / wall
    B = args.batch or w["B"]
    line = {
        "impl": "reference", "metric": "bounded fits solved/sec (batched)",
        "value": value, "unit": "fits/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": dict(static_config(w, B, min(B, w.get("chunk", B))),
                       sample_fits_per_step=fits // max(args.steps, 1),
                       fits_per_second_per_core=value / cores),
        "cpu_baseline": {"value": value, "unit": "fits/s", "cores": cores,
                         "kind": "port",
                         "sample": f"{fits // max(args.steps, 1)} fits per step "
                                   f"over {cores} worker processes (pool created "
                                   f"and warmed before the timed region), "
                                   f"oracle/blsq_oracle.py (NumPy/SciPy restatement "
                                   f"of the reference, bit-identical to it on the "
                                   f"golden files), mean nfev {nfev / fits:.1f}"},
        "e2e": {"value": value, "unit": "fits/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    if args.workload == "c2" and not args.no_tall and args.batch is None:
        line["tall"] = run_tall_reference_arm(args, WORKLOADS["c4"], standalone=False)
        line["config"]["tall_value"] = line["tall"]["value"]
    print(json.dumps(line))


# ------------------------------------------------------------ affinity ----

def pin_rank_to_gpu_cpus(local):
    """N > 1: the driver thread of this rank runs on the host cores NVML names
    as local to its GPU (torchrun does not bind ranks).  BLSQ_BENCH_PIN=0
    turns it off.  Returns what was done, for the JSON line."""
    if os.environ.get("BLSQ_BENCH_PIN", "1") == "0":
        return "off"
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        if not uuid.startswith("GPU-"):
            uuid = "GPU-" + uuid
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        near = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = sorted(os.sched_getaffinity(0))
        cpus = [c for c in near if c in allowed]
        if not cpus or len(cpus) == len(allowed):
            return "all %d allowed cores are local to the GPU" % len(allowed)
        os.sched_setaffinity(0, cpus)
        return "cores %d-%d of %d" % (cpus[0], cpus[-1], len(allowed))
    except Exception as e:                      # reporting only
        return "unavailable (%r)" % (e,)


# ------------------------------------------------------------ clocks ------

class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: in
    process through NVML (a few tens of microseconds per sample; spawning
    nvidia-smi inside a 100 ms region stalls the launch path for milliseconds
    and was visible in the number), nvidia-smi only as a fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReason bits
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40),
            ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4),
            ("hw_power_brake_slowdown", 0x80))

    def __init__(self, index, world=1, rank=0):
        """N > 1: ONE sampler for the job -- rank 0's thread reads the clocks of
        all `world` GPUs of the box; the other ranks make no NVML call at all
        (eight processes polling NVML were the one thing the 8-GPU bench did
        that tools/diag_first_step.py, which has no slow first step, did not)."""
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        self._hs = []
        self.active = rank == 0
        self.gpus = list(range(world)) if world > 1 else [index]
        if not self.active:
            return
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            for i in self.gpus:
                uuid = str(torch.cuda.get_device_properties(i).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                self._hs.append(pynvml.nvmlDeviceGetHandleByUUID(uuid))
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(
                self._hs[0], pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        nv = self._nvml
        for h in self._hs:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            row = [str(float(sm)), str(self._max)]
            row += ["Active" if mask & bit else "Not Active" for _, bit in self.BITS]
            self.rows.append(row)

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(
                        ["nvidia-smi", "-i", str(self.index),
                         "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                        capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.02 if self._nvml is not None else 0.2)

    def __enter__(self):
        if not self.active:
            return self
        # the first NVML queries of a process are the slow ones (they take the
        # driver's lock for 10-100 ms and stall a concurrent launch path): make
        # them here, before anything is timed
        if self._nvml is not None:
            for _ in range(8):
                try:
                    self._sample_nvml()
                except Exception:
                    break
                time.sleep(0.005)
            self.rows.clear()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                 "sw_power_cap", "hw_power_brake_slowdown"]
        reasons = [n for i, n in enumerate(names)
                   if any(len(r) > 2 + i and r[2 + i].lower().startswith("active")
                          for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "gpus_sampled": len(self.gpus),
                "source": "nvml" if self._nvml is not None else "nvidia-smi"}



# ------------------------------------------------------------ tall mode ---

TALL_METRIC = "TRF iterations/sec at m=16M, n=64 (tall)"


def _ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu
    capture (profiles/ncu_traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return json.load(fh).get(workload)
    except Exception:
        return None


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _fp64_peak():
    """Measured FP64 DMMA/DFMA peak of this pool's B200 (tools/fp64_peak.cu)."""
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles",
                                                 "FP64_PEAK.json")))["fp64_tflops"]), \
            "profiles/FP64_PEAK.json (tools/fp64_peak.cu measured on this pool's B200)"
    except Exception:
        return 37.0, "fallback 37.0 TFLOP/s (64 FMA/clk/SM x 148 SMs x 1965 MHz)"


def tall_cpu_iterations_per_second(n, m_cpu, max_nfev=4, seed=0):
    """The oracle's TRF (reference algorithm: LAPACK gesdd of the augmented
    Jacobian per iteration) on the host cores, BLAS threads = all cores, at a
    reduced m; returns (iterations/s at m_cpu, seconds, iterations)."""
    from oracle import blsq_oracle as orc
    from bounded_lsq_b200.synthetic import TallLinExp
    wl = TallLinExp(m_cpu, n, seed=seed)
    try:                                   # torchrun exports OMP_NUM_THREADS=1
        from threadpoolctl import threadpool_limits
        limit = threadpool_limits(limits=os.cpu_count())
    except Exception:
        limit = None
    t0 = time.perf_counter()
    r = orc.least_squares(wl.fun_np, wl.x0, jac=wl.jac_np, bounds=(wl.lb, wl.ub),
                          method="trf", max_nfev=max_nfev)
    dt = time.perf_counter() - t0
    if limit is not None:
        limit.restore_original_limits()
    return r.njev / dt, dt, r.njev


def run_tall_reference_arm(args, w, standalone=True):
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    cores = os.cpu_count() or 1
    n = w["n"]
    m_full = args.rows or w["m"]
    m_cpu = min(m_full, 1 << 19)
    for _ in range(min(args.warmup, 1)):
        tall_cpu_iterations_per_second(n, 1 << 14, 3)
    t0 = time.perf_counter()
    its = 0
    for k in range(args.steps):
        _, dt, it = tall_cpu_iterations_per_second(n, m_cpu, 4, seed=k)
        its += it
    wall = time.perf_counter() - t0
    # the reference's cost per iteration is linear in m (SURVEY section 6)
    value = its / wall * (m_cpu / m_full)
    sample = (f"oracle TRF (NumPy/SciPy restatement of the reference, LAPACK "
              f"gesdd per iteration) at m={m_cpu}, {its} iterations in "
              f"{wall:.1f} s, scaled linearly in m to m={m_full}")
    line = {
        "impl": "reference", "metric": TALL_METRIC, "value": value,
        "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["desc"], "rows": m_full, "n": n,
                   "cpu_rows": m_cpu, "extrapolated": m_cpu != m_full},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores,
                         "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    if standalone:
        print(json.dumps(line))
    return line


def run_tall(args, w, standalone=True, light=False, dump_prefix=None):
    """Tall workload.  standalone: own process-group set-up and JSON line;
    otherwise called from the batched main (default run) which attaches the
    returned dict to its line as "tall".  light: value only (no e2e, no CPU
    baseline) -- the asymmetric-start companion record.  dump_prefix: with
    --dump-outputs, the last timed solve's result goes to DIR/<prefix>*.npy."""
    import torch
    import torch.distributed as dist
    from bounded_lsq_b200 import least_squares
    from bounded_lsq_b200.synthetic import TallLinExpDevice

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and standalone:
        dist.init_process_group("nccl", device_id=dev)
    n = w["n"]
    m_total = args.rows or w["m"]
    rows = m_total // world                      # "strong": total rows fixed
    kw = dict(x0_tail=w["x0_tail"]) if w.get("x0_tail") else {}
    wl = TallLinExpDevice(rows, n, dev, seed=rank, lb=w.get("lb", -0.5), **kw)
    if args.method:
        w = dict(w, method=args.method)
    x0 = torch.as_tensor(wl.x0, device=dev)
    lb = torch.as_tensor(wl.lb, device=dev)
    ub = torch.as_tensor(wl.ub, device=dev)
    opts = {}
    fun, jac = wl.fun_t, wl.jac_t
    if args.callbacks == "fused":
        from bounded_lsq_b200 import models as fused
        fun, jac = fused.tall_callbacks(wl)

    def solve(timers=None):
        o = dict(opts)
        if timers is not None:
            o["timers"] = timers
        return least_squares(fun, x0, jac=jac, bounds=(lb, ub),
                             method=w["method"], options=o)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        res = solve()
    barrier()
    its = 0
    launches = 0
    nfev = 0
    with ClockSampler(local, world, rank) as clk:
        solve()                            # untimed, sampler thread running (see run_batched)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            res = solve()
            its += res.njev
            nfev += res.nfev
            launches += res.kernel_launches
        e1.record()
        barrier()
    dev_ms = reduce_max(e0.elapsed_time(e1))
    value = its / (dev_ms * 1e-3)
    if args.dump_outputs and dump_prefix is not None and rank == 0:
        dump_tall(args.dump_outputs, dump_prefix, res)

    # per-kernel timing (separate instrumented solve)
    collect = {}
    torch.cuda.synchronize()
    res_t = solve(collect)
    torch.cuda.synchronize()
    tsum = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in collect.items()}
    tcnt = {k: len(v) for k, v in collect.items()}
    gram_ms = tsum.get("gram1", 0.0) + tsum.get("gram2", 0.0)
    flops = 2.0 * rows * n * n * tcnt.get("gram1", 0)      # algorithmic QR flops
    peak, peak_src = _fp64_peak()
    ach = flops / (gram_ms * 1e-3) / 1e12 if gram_ms else None

    # end to end: the problem data comes from pinned host memory every step
    # (skipped for C5: 8 x 25 GB of pinned host memory)
    its_e2e, e2e_ms, h2d = 0, None, 0
    if not w.get("no_e2e") and not light:
        A_h = wl.A_t.cpu().pin_memory()
        t_h = wl.t_t.cpu().pin_memory()
        y_h = wl.y_t.cpu().pin_memory()
        x_out = torch.empty(n, dtype=torch.float64).pin_memory()
        # double-buffered input pipeline: every step's A, t, y come from pinned
        # host memory inside the timed region; the copy of step k + 1 runs on a
        # copy stream while step k is being solved (8.3 GB over PCIe is ~150 ms,
        # longer than a solve, so a serial copy would halve the rate)
        copy = torch.cuda.Stream(dev)
        bufs = [tuple(torch.empty_like(v) for v in (wl.A_t, wl.t_t, wl.y_t)) for _ in range(2)]
        copy.wait_stream(torch.cuda.current_stream(dev))

        def start_copy(k):
            with torch.cuda.stream(copy):
                for dst, src in zip(bufs[k % 2], (A_h, t_h, y_h)):
                    dst.copy_(src, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
            return ev

        barrier()
        e2 = torch.cuda.Event(enable_timing=True)
        e3 = torch.cuda.Event(enable_timing=True)
        e2.record()
        ev = start_copy(0)
        for k in range(args.steps):
            torch.cuda.current_stream(dev).wait_event(ev)
            if k + 1 < args.steps:
                ev = start_copy(k + 1)
            wl.load(*bufs[k % 2])
            r = solve()
            x_out.copy_(r.x, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()     # the result is on the host
            its_e2e += r.njev
        e3.record()
        barrier()
        e2e_ms = reduce_max(e2.elapsed_time(e3))
        h2d = (A_h.numel() + t_h.numel() + y_h.numel()) * 8
        del A_h, t_h, y_h, bufs
    if rank != 0:
        if world > 1 and standalone:
            dist.destroy_process_group()
        return None

    cpu = None
    if not args.no_cpu_baseline and not light:
        m_cpu = min(m_total, 1 << 19)
        v, dt, it = tall_cpu_iterations_per_second(n, m_cpu, 4)
        cpu = {"value": v * m_cpu / m_total, "unit": "iterations/s",
               "cores": os.cpu_count(), "kind": "port",
               "sample": f"oracle TRF (LAPACK gesdd per iteration, BLAS threads = "
                         f"all cores) at m={m_cpu}: {it} iterations in {dt:.1f} s "
                         f"= {v:.3f} it/s, scaled linearly in m to m={m_total} "
                         f"(extrapolated)"}
    line = {
        "metric": TALL_METRIC if n == 64 else
        "%s iterations/sec at m=%d, n=%d (tall)" % (w["method"].upper(), m_total, n),
        "value": value, "unit": "iterations/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": w["desc"], "rows_total": m_total,
                   "rows_per_gpu": rows, "n": n, "method": w["method"],
                   "callbacks": args.callbacks,
                   "x0_tail": list(w["x0_tail"]) if w.get("x0_tail") else
                   "SURVEY 8(d) start [.5, 1, .5, 1]: identical exponentials, "
                   "J(x0) exactly rank deficient, ulp-chaotic for TRF in the "
                   "reference itself; full parity is demonstrated on the "
                   "asymmetric start (tall_asymmetric_start)",
                   "step": "one complete TRF solve from x0; an iteration = one "
                           "accepted step (Jacobian + CholeskyQR2 + its trials)",
                   "iterations_per_step": its / args.steps,
                   "nfev_per_step": nfev / args.steps, "status": int(res.status),
                   "l2": "J (%.1f GB per GPU) exceeds the 126 MB L2"
                         % (rows * n * 8 / 1e9)},
        "e2e": ({"value": its_e2e / (e2e_ms * 1e-3), "unit": "iterations/s",
                 "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": n * 8,
                 "ms_per_step": e2e_ms / args.steps,
                 "pipeline": "inputs of step k+1 are copied (pinned host -> device, "
                             "copy stream, second buffer set) while step k is solved"}
                if e2e_ms else None),
        "gpu_launches": launches,
        "roofline": {
            "bound": "tensor", "kernel": "gram_kernel<%d,1> + gram_kernel<%d,2> " % ((n + 7) // 8, (n + 7) // 8) +
                                         "(Cholesky QR of [J | f], FP64 DMMA)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s",
            "frac": (ach / peak) if ach else None,
            "traffic": (_ncu_traffic("c4") or {}).get("bytes_per_launch"),
            "traffic_source": _ncu_traffic("c4"),
            "peak_source": peak_src,
            "algorithmic_flops_per_jacobian": 2.0 * rows * n * n,
            "route": "preconditioned Cholesky QR: pass 1 on a 1/8 row sample, "
                     "pass 2 (TRMM + SYRK on the upper 8x8 blocks) on every row: "
                     "~2.4 m n^2 flop executed for the 2 m n^2 quoted (ceiling "
                     "84% of peak); DESIGN.md section 2.2",
            "avg_launch_ms": {k: tsum[k] / tcnt[k] for k in tsum},
            "launches": tcnt,
            "share_of_solve_ms": {k: tsum[k] / sum(tsum.values()) for k in tsum},
        },
        "cpu_baseline": cpu,
        "clocks": clk.summary(),
    }
    if standalone:
        print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
    return line

# ------------------------------------------------------------ GPU arm -----

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=None,
                    help="problems per GPU (default: the workload's size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tall", action="store_true",
                    help="default (c2) run: skip the tall (C4) measurement that "
                         "is otherwise attached to the line as \"tall\"")
    ap.add_argument("--callbacks", default="fused", choices=["fused", "torch"],
                    help="residual/Jacobian callbacks: the fused CUDA model "
                         "op shipped for the synthetic workloads, or plain "
                         "torch elementwise ops")
    ap.add_argument("--rounds-log", default=None,
                    help="write the per-round CUDA-event timings of the "
                         "instrumented step (running problems, callbacks / "
                         "linearise / round ms) to this CSV file")
    ap.add_argument("--method", default=None, choices=["trf", "dogbox"],
                    help="tall workloads: override the method (C5: TRF vs dogbox)")
    ap.add_argument("--rows", type=int, default=None,
                    help="tall workload: total rows (default 2^24)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed "
                         "to DIR/<name>.npy (float64; a seeded sample of the "
                         "problems / rows, under 64 MB in all); the default run "
                         "adds the tall solve as DIR/tall_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results (--impl b200)")
    w = WORKLOADS[args.workload]
    if w.get("kind") == "tall":
        if args.impl == "reference":
            return run_tall_reference_arm(args, w)
        return run_tall(args, w, dump_prefix="")
    if args.impl == "reference":
        return run_reference_arm(args, w)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pinned = None
    if world > 1:
        pinned = pin_rank_to_gpu_cpus(local)
        dist.init_process_group("nccl", device_id=dev)

    line = run_batched(args, w, args.workload, args.steps, args.warmup,
                       args.batch or w["B"], cpu_baseline=not args.no_cpu_baseline,
                       dump_prefix="")
    if line is not None and pinned is not None:
        line["config"]["driver_thread_affinity"] = pinned

    # the other half of BASELINE.json's metric (TRF iterations/s at m=16M,
    # n=64) rides along on the default run as the "tall" object, and a run of
    # configs[2] (C3: dogbox, 2-point Jacobian; ONE 1M-problem chunk of the
    # 10M) as "c3".  Their headline numbers are repeated inside `config`.
    # Every record times --steps steps after --warmup warm-up solves: a record
    # of only two steps moved by 30% between runs whenever one host stall
    # landed in it.
    if args.workload == "c2" and not args.no_tall and args.batch is None:
        torch.cuda.empty_cache()
        tall_line = run_tall(args, WORKLOADS["c4"], standalone=False, dump_prefix="tall_")
        torch.cuda.empty_cache()
        tall_asym = run_tall(args, dict(WORKLOADS["c4"], x0_tail=(0.8, 1.5, 0.3, 4.0)),
                             standalone=False, light=True)
        torch.cuda.empty_cache()
        c3_line = run_batched(args, WORKLOADS["c3"], "c3", args.steps, args.warmup,
                              1_000_000, cpu_baseline=False)
        torch.cuda.empty_cache()
        # NOT the headline: the same C2 solve with the residual model compiled
        # into the linearisation kernel (J and f never touch HBM) -- what the
        # solver does when the callback is fusable (VERDICT r1, item 10)
        inl = run_batched(args, w, "c2", args.steps, args.warmup, w["B"],
                          cpu_baseline=False, inlined=True)
        if rank == 0:
            line["tall"] = tall_line
            line["tall_asymmetric_start"] = tall_asym
            line["c3"] = c3_line
            line["c2_inlined_model"] = {
                "note": "separate record, not the headline: ExpDecay2 compiled into "
                        "the linearisation kernel (models.callbacks(..., 'inlined')); "
                        "results bit-identical to the callback path",
                "value": inl["value"], "unit": inl["unit"], "steps": inl["steps"],
                "ms_per_step": inl["ms_per_step"], "e2e": inl["e2e"],
                "step_frac": inl["roofline"]["step_frac"],
                "gpu_launches": inl["gpu_launches"], "config": inl["config"]}
            cfg = line["config"]
            cfg["tall_value_it_per_s"] = tall_line["value"]
            cfg["tall_roofline_frac"] = tall_line["roofline"]["frac"]
            cfg["tall_e2e_it_per_s"] = (tall_line["e2e"] or {}).get("value")
            cfg["tall_asym_value_it_per_s"] = tall_asym["value"]
            cfg["c3_value_fits_per_s"] = c3_line["value"]
            cfg["c3_roofline_frac"] = c3_line["roofline"]["frac"]
            cfg["c3_e2e_fits_per_s"] = c3_line["e2e"]["value"]
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_batched(args, w, wname, steps, warmup, B, cpu_baseline=True, inlined=False,
                dump_prefix=None):
    """One batched workload on this rank's GPU (problems split by index over
    the ranks, no collective on the data path); returns the JSON record on
    rank 0, None elsewhere.  dump_prefix: with --dump-outputs, the last timed
    step's results go to DIR/<prefix>*.npy."""
    import torch
    import torch.distributed as dist
    from bounded_lsq_b200 import least_squares_batched, PerProblem
    from bounded_lsq_b200 import batched as drv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    model = _model(w["model"])
    chunk = min(B, w.get("chunk", B))
    n, m = w["n"], w["m"]
    method = w["method"]

    # synthetic data of the named shape, generated on the host once.  Every
    # GPU solves the SAME pool (weak scaling: per-GPU work exactly fixed).  With
    # a seed per rank the pools differ in their slowest problem -- C2: 113
    # evaluations for seed 10000, 254 for 10001 (oracle) -- and a solve runs as
    # many latency-sized tail rounds as its slowest problem needs: rank 1's
    # steps took 22.3 ms against rank 0's 19.0 for that reason alone.
    # BLSQ_BENCH_SEED_PER_RANK=1 restores the per-rank pools.
    t_gen = time.perf_counter()
    rng_seed = 10_000 + (rank if os.environ.get("BLSQ_BENCH_SEED_PER_RANK") == "1" else 0)
    ngen = min(B, 262_144)              # tile a 256k-problem pool up to B
    _, ypool = model.make_data(ngen, seed=rng_seed)
    reps = (B + ngen - 1) // ngen
    y_host = torch.from_numpy(np.tile(ypool, (reps, 1))[:B].copy()).pin_memory()
    x0_host = torch.from_numpy(np.tile(model.x0, (B, 1))).pin_memory()
    lb = torch.as_tensor(model.lb, device=dev)
    ub = torch.as_tensor(model.ub, device=dev)
    gen_s = time.perf_counter() - t_gen

    fun, jac = model.fun_t, (model.jac_t if w["jac"] == "exact" else "2-point")
    if args.callbacks == "fused" or inlined:
        try:
            from bounded_lsq_b200 import models as fused
            fun, jac = fused.callbacks(w["model"], "inlined" if inlined else w["jac"])
        except Exception as e:          # the fused op is optional sugar
            if rank == 0:
                print(f"# fused callbacks unavailable ({e!r}); using torch",
                      file=sys.stderr)
            args.callbacks = "torch"

    timers = {}

    def solve(y_any, x0_any, collect=None):
        """y / x0 on the device (value) or pinned on the host (e2e: the front
        end streams them in chunks and overlaps the copies with the first
        rounds, least_squares.py `_stage_host_inputs`)."""
        outs = []
        for c0 in range(0, B, chunk):
            yc = y_any[c0:c0 + chunk]
            opts = dict(timers=collect) if collect is not None else {}
            if not x0_any.is_cuda:
                opts.update(h2d_chunks=int(os.environ.get("BLSQ_BENCH_H2D_CHUNKS", "4")),
                            device=dev,
                            prologue_rounds=w.get("prologue_rounds", 6))
            res = least_squares_batched(
                fun, x0_any[c0:c0 + chunk], jac=jac, bounds=(lb, ub),
                method=method, args=(PerProblem(yc),), options=opts)
            outs.append(res)
        return outs

    y_dev = y_host.to(dev)
    x0_dev = x0_host.to(dev)
    x_out = torch.empty((B, n), dtype=torch.float64).pin_memory()
    st_out = torch.empty((B,), dtype=torch.int64).pin_memory()
    obj_out = torch.empty((B,), dtype=torch.float64).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing -----------------------------------------
    # the warm-up keeps the previous result alive while the next solve runs,
    # exactly as the timed loop does: with results dropped at once the second
    # TIMED step was the first to need a second set of result buffers and paid
    # the allocator's cudaMalloc for it (sporadic 20 - 150 ms on that step)
    outs = None
    for _ in range(max(warmup, 2)):
        outs = solve(y_dev, x0_dev)
    barrier()
    launches = 0
    rounds = 0
    with ClockSampler(local, world, rank) as clk:
        # one more untimed solve with the sampler thread already running: its
        # first NVML queries cost the launch path 10-100 ms once (seen as a
        # slow second step in 4 of 6 runs when the thread started with the
        # timed region)
        outs = solve(y_dev, x0_dev)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        marks = [e0]
        for _ in range(steps):
            outs = solve(y_dev, x0_dev)
            launches += sum(o.kernel_launches for o in outs)
            rounds += sum(o.rounds for o in outs)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append(ev)
        e1.record()
        barrier()
    dev_ms = reduce_max(e0.elapsed_time(e1))
    if args.dump_outputs and dump_prefix is not None and rank == 0:
        dump_batched(args.dump_outputs, dump_prefix, outs, chunk, B)
    per_step_ms = [a.elapsed_time(b) for a, b in zip(marks, marks[1:])]
    by_rank = None
    if world > 1:
        # every rank's own steps: the line's time is the MAX over ranks of the
        # whole region, so one slow rank (or one stalled step on any of them)
        # sets it
        mine = torch.tensor(per_step_ms, dtype=torch.float64, device=dev)
        allr = torch.empty((world, steps), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allr.view(-1), mine)
        by_rank = {"mean": [round(float(v), 3) for v in allr.mean(1)],
                   "max": [round(float(v), 3) for v in allr.max(1).values]}
    value = world * B * steps / (dev_ms * 1e-3)
    status = torch.cat([o.status for o in outs])
    nfev_mean = float(torch.cat([o.nfev for o in outs]).double().mean())
    njev_mean = float(torch.cat([o.njev for o in outs]).double().mean())
    converged = float((status > 0).double().mean())

    # ---- per-kernel timing for the roofline (separate instrumented step) --
    solve(y_dev, x0_dev, {})               # untimed: first eager-tail solve
    collect = {}
    torch.cuda.synchronize()
    solve(y_dev, x0_dev, collect)
    torch.cuda.synchronize()
    ksum = drv.summarize_timers(collect)
    if args.rounds_log and rank == 0:
        with open(args.rounds_log, "w") as fh:
            fh.write("round,running,callbacks_ms,linearise_ms,round_ms\n")
            cols = [collect.get(k, []) for k in ("callbacks", "linearise", "round")]
            for i, evs in enumerate(zip(*cols)):
                ms = [a.elapsed_time(b) for a, b, _ in evs]
                fh.write("%d,%d,%.5f,%.5f,%.5f\n" % (i, evs[0][2], *ms))

    # ---- end to end: host buffers in, host results out -------------------
    # Every step's x0 and y come from pinned host memory inside the timed
    # region through the public staging call (stage_host_inputs: chunked
    # copies on a copy stream, each chunk starts its first rounds as soon as
    # it has landed); the copies of step k + 1 are started before step k is
    # solved (second buffer set), as a serving loop would.
    from bounded_lsq_b200 import stage_host_inputs
    nch = int(os.environ.get("BLSQ_BENCH_H2D_CHUNKS", "4"))
    sets = [(torch.empty_like(x0_dev), torch.empty_like(y_dev)) for _ in range(2)]

    def stage(k):
        xb, yb = sets[k % 2]
        return stage_host_inputs(x0_host, (PerProblem(y_host),), {}, device=dev,
                                 h2d_chunks=nch, out=(xb, {id(y_host): yb}))

    def solve_staged(st):
        x0d, a, kw, plan = st
        outs = []
        for c0 in range(0, B, chunk):
            if chunk == B:
                opts = dict(prologue=plan, prologue_rounds=w.get("prologue_rounds", 6))
                xa, aa = x0d, a
            else:
                # chunked workloads (C3): the chunk's copies must have landed
                for p0, p1, ev in plan:
                    if p0 < c0 + chunk and p1 > c0:
                        torch.cuda.current_stream(dev).wait_event(ev)
                torch.cuda.current_stream(dev).wait_event(plan.x0_event)
                opts = {}
                xa = x0d[c0:c0 + chunk]
                aa = tuple(PerProblem(v.tensor[c0:c0 + chunk]) if isinstance(v, PerProblem)
                           else v for v in a)
            outs.append(least_squares_batched(fun, xa, jac=jac, bounds=(lb, ub),
                                              method=method, args=aa, options=opts))
        return outs

    # results go back on their own stream into one of two pinned sets: the
    # device-to-host copies of step k run under the solve of step k + 1, the
    # host has step k's results before step k + 1 ends
    back = torch.cuda.Stream(dev)
    outsets = [(x_out, st_out, obj_out),
               (torch.empty_like(x_out).pin_memory(), torch.empty_like(st_out).pin_memory(),
                torch.empty_like(obj_out).pin_memory())]

    def results_to_host(outs, k):
        xo, so, oo = outsets[k % 2]
        ev = torch.cuda.Event()
        back.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(back):
            for c, o in enumerate(outs):
                sl = slice(c * chunk, c * chunk + o.x.shape[0])
                xo[sl].copy_(o.x, non_blocking=True)
                so[sl].copy_(o.status, non_blocking=True)
                oo[sl].copy_(o.obj_value, non_blocking=True)
            ev.record(back)
        return ev, outs                    # `outs` stays referenced until the copies are done

    results_to_host(solve_staged(stage(0)), 0)[0].synchronize()   # untimed: streams, first capture
    barrier()
    e2 = torch.cuda.Event(enable_timing=True)
    e3 = torch.cuda.Event(enable_timing=True)
    e2.record()
    st = stage(0)
    pending = None
    marks = [e2]
    for k in range(steps):
        nxt = stage(k + 1) if k + 1 < steps else None
        outs = solve_staged(st)
        if pending is not None:
            pending[0].synchronize()       # step k - 1 is on the host
        pending = results_to_host(outs, k)
        st = nxt
        marks.append(torch.cuda.Event(enable_timing=True))
        marks[-1].record()
    pending[0].synchronize()               # the last step's results are on the host
    e3.record()
    torch.cuda.current_stream(dev).synchronize()
    barrier()
    e2e_ms = reduce_max(e2.elapsed_time(e3))
    e2e_steps = [round(a.elapsed_time(b), 3) for a, b in zip(marks, marks[1:])]
    e2e_value = world * B * steps / (e2e_ms * 1e-3)
    h2d = y_host.numel() * 8 + x0_host.numel() * 8
    d2h = x_out.numel() * 8 + st_out.numel() * 8 + obj_out.numel() * 8
    del sets

    del y_dev, x0_dev, outs, y_host, x0_host
    if rank != 0:
        return None

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else \
        "fallback 6650 GB/s (B200_PROFILING.md)"
    lin = ksum.get("linearise", {})
    rnd = ksum.get("round", {})
    roofline = {
        "bound": "hbm", "kernel": "lin_kernel (blsq_linearise_batched)",
        "achieved": lin.get("gbs"), "peak": peak, "unit": "GB/s",
        "frac": (lin.get("gbs") / peak) if lin.get("gbs") else None,
        "traffic": (_ncu_traffic(wname) or {}).get("bytes_per_launch"),
        "traffic_source": _ncu_traffic(wname), "peak_source": peak_src,
        "algorithmic_bytes_per_problem": lin.get("bytes_per_problem"),
        "avg_launch_ms": lin.get("avg_ms"), "launches": lin.get("launches"),
        "share_of_kernel_time": lin.get("share"),
        # the same kernel on the launches that still see the whole batch
        # (the average above includes ~100 latency-sized tail launches)
        "full_batch_launches": dict(
            lin.get("full_batch", {}),
            frac=(lin["full_batch"]["gbs"] / peak) if lin.get("full_batch") else None),
        "round_kernel": {"avg_launch_ms": rnd.get("avg_ms"),
                         "share_of_kernel_time": rnd.get("share"),
                         "gbs": rnd.get("gbs")},
        "callbacks_ms_per_step": ksum.get("callbacks_ms"),
        "kernels_ms_per_step": ksum.get("kernels_ms"),
    }
    # step level: SURVEY 8(d) algorithmic bytes of the WHOLE solve
    # (sum over problems of njev*8m(n+1) + nfev*(8m+32n)) over the device time
    # of a step -- callbacks, every kernel, launch gaps and host look-ups
    # included -- against the same HBM peak
    step_bytes = B * (njev_mean * 8 * m * (n + 1) + nfev_mean * (8 * m + 32 * n))
    roofline["step_algorithmic_bytes"] = step_bytes
    roofline["step_frac"] = step_bytes / (dev_ms / steps * 1e-3) / 1e9 / peak
    if ksum.get("kernels_ms"):
        roofline["step_frac_kernels_only"] = \
            step_bytes / (ksum["kernels_ms"] * 1e-3) / 1e9 / peak

    cpu = None
    if cpu_baseline:
        # the reference arm's own procedure (run_reference_arm): three steps of
        # 256 fits per core (96 for finite differences), total fits / total time
        per_core = 256 if w["jac"] == "exact" else 96
        cpu_fits_per_second(w, 16)                 # pool created and warmed untimed
        fits, wall, nfs = 0, 0.0, 0.0
        for k in range(3):
            vk, cores, fk, nfk = cpu_fits_per_second(w, per_core, seed0=2000 + 97 * k)
            fits += fk
            wall += fk / vk
            nfs += nfk * fk
        v, nf = fits / wall, nfs / fits
        cpu = {"value": v, "unit": "fits/s", "cores": cores, "kind": "port",
               "sample": f"{fits} fits (3 x {per_core}/core, as --impl reference), "
                         f"oracle/blsq_oracle.py NumPy/SciPy restatement, "
                         f"mean nfev {nf:.1f}"}
        try:
            cpu["parity_vs_gpu"] = gpu_parity_of_cpu_sample(w, fun, jac, lb, ub, dev)
        except Exception as e:                    # reporting only
            cpu["parity_vs_gpu"] = {"error": repr(e)}

    line = {
        "metric": "bounded fits solved/sec (batched)", "value": value,
        "unit": "fits/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": dev_ms / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": dict(
            static_config(w, B, chunk, "inlined" if inlined else args.callbacks),
            l2="inputs (J+f per round: %.1f GB) exceed the 126 MB L2"
               % (chunk * m * (n + 1) * 8 / 1e9),
            data_pool="%d distinct seeded problems tiled to %d (same traffic; host "
                      "generation time); the same pool on every GPU" % (ngen, B),
            mean_nfev=nfev_mean, mean_njev=njev_mean, converged_frac=converged,
            rounds_per_step=rounds / steps,
            per_step_ms=[round(v, 3) for v in per_step_ms],
            **({"per_step_ms_by_rank": by_rank} if by_rank else {})),
        "e2e": {"value": e2e_value, "unit": "fits/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / steps, "per_step_ms": e2e_steps,
                "pipeline": "stage_host_inputs: pinned x0 / y -> device in %d chunks on a "
                            "copy stream, each chunk starts its rounds when it lands; the "
                            "copies of step k+1 are started before step k is solved and the "
                            "results of step k return to pinned memory under step k+1 (own "
                            "stream, two buffer sets); the region ends when the last "
                            "results are on the host" % nch},
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clk.summary(),
    }
    return line




if __name__ == "__main__":
    main()
