"""Where does a C2 step spend its time?  Device-resident solves under a few
driver variants, per-solve wall clock and CUDA-event time."""
import os, sys, time, json
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bounded_lsq_b200 import least_squares_batched, PerProblem, models
from bounded_lsq_b200.synthetic import ExpDecay2

dev = torch.device("cuda:0")
model = ExpDecay2()
B = int(os.environ.get("B", 1_000_000))
_, yp = model.make_data(262144, seed=10000)
y = torch.from_numpy(np.tile(yp, (4, 1))[:B].copy()).to(dev)
x0 = torch.from_numpy(np.tile(model.x0, (B, 1))).to(dev)
lb, ub = torch.as_tensor(model.lb, device=dev), torch.as_tensor(model.ub, device=dev)
fun, jac = models.callbacks("ExpDecay2", "exact")


def run(label, **opts):
    ts = []
    for i in range(8):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        r = least_squares_batched(fun, x0, jac=jac, bounds=(lb, ub), method="trf",
                                  args=(PerProblem(y),), options=dict(opts))
        e1.record()
        torch.cuda.synchronize()
        ts.append((round((time.perf_counter() - t0) * 1e3, 2), round(e0.elapsed_time(e1), 2)))
    print(json.dumps(dict(variant=label, wall_event_ms=ts, rounds=r.rounds,
                          launches=r.kernel_launches)), flush=True)


if os.environ.get("SWEEP"):
    # driver thresholds: where the CUDA-graph tail starts, rounds per replay,
    # compaction threshold
    run("default")
    for tb in (16384, 32768, 65536, 131072):
        run("tail_below=%d" % tb, tail_below=tb)
    for gr in (4, 16, 32):
        run("graph_tail_rounds=%d" % gr, graph_tail_rounds=gr)
    for tb, gr in ((32768, 16), (65536, 16)):
        run("tail_below=%d graph_tail_rounds=%d" % (tb, gr), tail_below=tb, graph_tail_rounds=gr)
    for cb in (0.5, 0.65, 0.85, 0.92):
        run("compact_below=%.2f" % cb, compact_below=cb)
    sys.exit(0)

run("default")
run("no graph tail", graph_tail_rounds=0)
run("prologue 7 rounds (no count, no host look)", prologue=[(0, B, None)], prologue_rounds=7)
run("check every 2 rounds", check_every=2)
run("no compaction", compact_below=0.0)
