"""bench.py's reference arm (`--impl reference`: the oracle on the host cores)
runs without a GPU; this checks that it prints ONE JSON line with the keys the
driver's contract names.  The GPU arm's line is checked on the B200
(tests/test_gpu_parity.py::test_bench_line_contract)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
             "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
             "e2e", "cpu_baseline")


def check_line(line, reference):
    for k in BASE_KEYS:
        assert k in line, k
    assert line["metric"] == "bounded fits solved/sec (batched)"
    assert line["unit"] == "fits/s" and line["higher_is_better"] is True
    assert line["dtype"] == "f64" and line["data"] == "synthetic"
    assert "workload" in line["config"] and "model" not in line["config"]
    assert line["vs_baseline"] is None            # BASELINE.md publishes no number
    cb = line["cpu_baseline"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in cb, k
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1
    e2e = line["e2e"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in e2e, k
    if reference:
        assert line["impl"] == "reference"
        assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
        assert e2e["value"] == line["value"] == cb["value"]
    else:
        assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
        assert line["gpu_launches"] > 0
        rf = line["roofline"]
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in rf, k
        assert rf["bound"] == "hbm" and 0 < rf["frac"] < 1
        assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
        ck = line["clocks"]
        assert "sm_mhz" in ck and "sm_max_mhz" in ck and "reasons" in ck


def run_bench(args, timeout):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args,
                         capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    line = run_bench(["--impl", "reference", "--steps", "1", "--warmup", "0"], 600)
    check_line(line, reference=True)
    tall = line["tall"]
    assert tall["impl"] == "reference" and tall["unit"] == "iterations/s"
    assert tall["config"]["extrapolated"] is True


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    line = run_bench(["--steps", "2", "--warmup", "3", "--no-tall",
                      "--dump-outputs", str(tmp_path)], 900)
    check_line(line, reference=False)
    assert line["steps"] == 2 and len(line["config"]["per_step_ms"]) == 2
    p = line["cpu_baseline"]["parity_vs_gpu"]
    assert p["status_equal"] == 1.0 and p["x_rel_max"] < 1e-8 and p["obj_rel_max"] < 1e-8
    # --dump-outputs: the last timed step's results on a seeded problem sample
    files = sorted(os.listdir(tmp_path))
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    out = {f[:-len(".npy")]: np.load(tmp_path / f) for f in files}
    assert all(a.dtype == np.float64 for a in out.values())
    idx = out["problem_index"]
    assert len(idx) == 32768 and (np.diff(idx) > 0).all()
    assert out["x"].shape == out["active_mask"].shape == (len(idx), 4)
    assert out["fun"].shape == (len(idx), 64)
    assert (out["status"] >= 0).all() and (out["status"] > 0).mean() > 0.99
    assert np.isfinite(out["obj_value"]).all()


@pytest.mark.gpu
def test_steps_set_every_record():
    """--steps K times K steps in every record of the default run, the
    attached tall, c3 and inlined-model records included."""
    line = run_bench(["--steps", "3", "--warmup", "1", "--no-cpu-baseline"], 900)
    for rec in (line, line["c3"], line["c2_inlined_model"]):
        assert rec["steps"] == 3 and len(rec["config"]["per_step_ms"]) == 3
    assert line["tall"]["steps"] == line["tall_asymmetric_start"]["steps"] == 3
