"""Compiled models with Jacobians derived by forward-mode dual numbers
(csrc/blsq_dual.cuh) against the other routes of the same model.

C3 (one 1M-problem chunk of GaussPeak, dogbox, m = 128): autodiff
'inlined', 'inlined-2-point', autodiff 'exact' and the hand-written
jacobian_row's 'exact'.  C2 (1M ExpDecay2 fits, TRF, m = 64) and W11 (250k
three-peak fits, n = 11, m = 128, TRF): autodiff 'inlined' against the hand
'inlined'.  Per route: ms per solve (device events over --steps solves after
--warmup, the routes alternated), fits/s and the full-batch linearise time
from a separate timed solve; the bit identity of the routes that must agree.
Also the ptxas registers / stack / spills of every generated instance of the
templated models (N = 1, 4, 5, 6, 11, 16); `--ptxas-only` prints that table
without a GPU.  The card's name and power limit are read in the same run.

    python tools/autodiff_bench.py --out autodiff_bench.json
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(ROOT), os.path.join(os.path.dirname(ROOT), "tests"), ROOT]

from bounded_lsq_b200 import PerProblem, models      # noqa: E402
import test_autodiff_models as ad                     # noqa: E402
import test_user_models as hand                       # noqa: E402

PTXAS_MODELS = ("Exp1", "ExpDecay2", "RatPoly5", "GaussPeak", "ThreePeak", "Cheb16")


def ptxas_table(cms):
    """[(model, N, instance, class, registers, stack, spill stores, spill loads)]
    of every kernel in the models' ptxas logs."""
    rows = []
    for name, cm in cms.items():
        log = open(cm.path[:-3] + ".ptxas.log").read()
        for m in re.finditer(r"Compiling entry function '(\S+)' for 'sm_100a'\n((?:.*\n)*?)"
                             r"ptxas info\s+: Used (\d+) registers", log):
            dem = subprocess.run(["c++filt", m.group(1)], capture_output=True,
                                 text=True).stdout.strip()
            blk = m.group(2)
            stack = re.search(r"(\d+) bytes stack frame", blk)
            st = re.search(r"(\d+) bytes spill stores", blk)
            ld = re.search(r"(\d+) bytes spill loads", blk)
            k = re.search(r"lin_kernel<(\d+), (\d+), 3, (true|false), blsq_um::(\w+)<[^,>]+"
                          r"(?:, (true|false))?>", dem)
            if k:
                inst = {"Fd2Rows": "2-point", "AnalyticRows": "autodiff"}[k.group(4)]
                if k.group(5) == "true":
                    inst += " (dogbox J point)"
                cls = f"G={k.group(2)}" + (" MULTI" if k.group(3) == "true" else "")
            elif "fun_kernel" in dem or "jac_kernel" in dem:
                inst, cls = ("fun_kernel" if "fun_kernel" in dem else "jac_kernel"), "-"
            else:
                continue
            rows.append((name, cm.n, inst, cls, int(m.group(3)),
                         int(stack.group(1)) if stack else 0, int(st.group(1)) if st else 0,
                         int(ld.group(1)) if ld else 0))
    return sorted(rows, key=lambda r: (r[1], r[2], r[3]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    ap.add_argument("--ptxas-only", action="store_true")
    a = ap.parse_args()

    with tempfile.TemporaryDirectory() as cache:
        with ThreadPoolExecutor(8) as ex:
            fa = {k: ex.submit(models.compile_model, ad.AD[k][0], ad.AD[k][1], cache)
                  for k in PTXAS_MODELS}
            fh = {k: ex.submit(models.compile_model, hand.REF[k][0], hand.REF[k][1], cache)
                  for k in ("ExpDecay2", "GaussPeak", "ThreePeak")}
            cad = {k: f.result() for k, f in fa.items()}
            chand = {k: f.result() for k, f in fh.items()}
        table = ptxas_table(cad)
    rec = dict(ptxas=[dict(zip(("model", "N", "instance", "class", "registers", "stack",
                                "spill_stores", "spill_loads"), r)) for r in table])
    if a.ptxas_only:
        print("| model | N | instance | class | registers | stack (B) | spill stores (B) "
              "| spill loads (B) |\n|---|---|---|---|---|---|---|---|")
        for r in table:
            print("| " + " | ".join(str(v) for v in r) + " |")
        return

    import torch
    import user_model_bench as umb
    from bounded_lsq_b200.synthetic import ExpDecay2, GaussPeak
    rec.update(card=umb.card(), torch=torch.__version__)
    T = umb.T
    B = 1_000_000

    # C3: one 1M-problem chunk
    m3 = GaussPeak()
    _, y = m3.make_data(B, seed=1)
    args = (PerProblem(T(y)), T(m3.t))
    gp, gh = cad["GaussPeak"], chand["GaussPeak"]
    routes = {"autodiff_inlined": gp.callbacks("inlined", m=m3.m) + (args,),
              "inlined_2point": gp.callbacks("inlined-2-point", m=m3.m) + (args,),
              "autodiff_exact": gp.callbacks("exact", m=m3.m) + (args,),
              "hand_exact": gh.callbacks("exact", m=m3.m) + (args,)}
    res, sol = umb.bench(routes, "dogbox", m3.x0, m3.lb, m3.ub, B, a.steps, a.warmup)
    rec["c3"] = dict(B=B, m=m3.m, method="dogbox", routes=res,
                     bits_autodiff_inlined_eq_exact=umb.same(sol["autodiff_inlined"],
                                                             sol["autodiff_exact"]))
    del sol, routes, args
    torch.cuda.empty_cache()

    # C2
    m2 = ExpDecay2()
    _, y = m2.make_data(B, seed=0)
    args = (PerProblem(T(y)), T(m2.t))
    routes = {"autodiff_inlined": cad["ExpDecay2"].callbacks("inlined", m=m2.m) + (args,),
              "hand_inlined": chand["ExpDecay2"].callbacks("inlined", m=m2.m) + (args,)}
    res, sol = umb.bench(routes, "trf", m2.x0, m2.lb, m2.ub, B, a.steps, a.warmup)
    rec["c2"] = dict(B=B, m=m2.m, method="trf", routes=res)
    del sol, routes, args
    torch.cuda.empty_cache()

    # W11
    Bw, mw = 250_000, 128
    tw, yw, x0, lb, ub = hand.problem_data("ThreePeak", mw, Bw, seed=2)
    args = (PerProblem(T(yw)), T(tw))
    routes = {"autodiff_inlined": cad["ThreePeak"].callbacks("inlined", m=mw) + (args,),
              "hand_inlined": chand["ThreePeak"].callbacks("inlined", m=mw) + (args,)}
    res, sol = umb.bench(routes, "trf", x0, lb, ub, Bw, a.steps, a.warmup)
    rec["w11"] = dict(B=Bw, m=mw, method="trf", routes=res)

    s = json.dumps(rec, indent=1, default=float)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
