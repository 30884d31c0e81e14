"""Developer tool: a whole SLP solve on the GPU engine; prints per-iteration LP statistics and totals.
python tools/gpu_slp_run.py case118 LS [max_iter] [k=v lp options ...]"""
import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as g
g.build()
from helpers import problem
from activesetmethods_b200.slp import Model, Parameters, SlpLS, SlpTR
name = sys.argv[1]; alg = {"LS": "Line Search", "TR": "Trust Region"}[sys.argv[2]]
max_iter = int(sys.argv[3]) if len(sys.argv) > 3 else 40
opts = dict(eps_rel=1e-6, max_iter=4000000)
for kv in sys.argv[4:]:
    k, v = kv.split("=")
    opts[k] = float(v) if ("." in v or "e" in v) else int(v)
pr = problem(name)
mdl = Model.from_problem(pr, Parameters(algorithm=alg, max_iter=max_iter, lp_options=opts))
slp = (SlpLS if alg == "Line Search" else SlpTR)(mdl)
t0 = time.time()


def progress(b, d):
    """``b`` is the one-scenario batch driver behind ``slp``: its state is scenario 0 of each array."""
    if b.lp_log[0]:
        alpha = b.alpha[0] if hasattr(b, "alpha") else 1.0
        print(f"  [{time.time() - t0:7.1f}s] SLP it {b.iter[0]} last LP {b.lp_log[0][-1]} prim_infeas "
              f"{b.prim_infeas[0]:.3e} f {b.f[0]:.6f} alpha {alpha:.3g}", flush=True)


slp.record = progress
slp.run()
dt = time.time() - t0
its = [e[3] for e in slp.lp_log]
print(f"{name} {alg} {opts}: ret {slp.ret} SLP iterations {slp.iter} sub-LPs {len(its)} obj {slp.obj_val:.6f} "
      f"PDHG iterations total {sum(its)} (per LP: {its[:40]}) wall {dt:.1f}s -> {slp.iter / dt:.2f} SLP it/s")
