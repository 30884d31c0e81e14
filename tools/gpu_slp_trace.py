"""Developer tool: per-iteration trace of a GPU SLP solve.  python tools/gpu_slp_trace.py case9 TR [tight] [k=v ...]"""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as g
g.build()
from helpers import problem
from activesetmethods_b200.slp import Model, Parameters, SlpLS, SlpLSBatch, SlpTR, SlpTRBatch
name, a = sys.argv[1], sys.argv[2]
tight = len(sys.argv) > 3 and sys.argv[3] == "tight"
opts = {}
extra = {}
for kv in sys.argv[4:]:
    k, v = kv.split("=")
    if k in ("device_evaluator", "max_iter"):
        extra[k] = int(v)
        continue
    opts[k] = float(v) if ("." in v or "e" in v) else int(v)
tol = dict(tol_residual=1e-8, tol_infeas=1e-8) if tight else {}
mdl = Model.from_problem(problem(name), Parameters(algorithm={"LS": "Line Search", "TR": "Trust Region"}[a], lp_options=opts, **{'max_iter': 300, **extra}, **tol))


class Traced(SlpLSBatch if a == "LS" else SlpTRBatch):
    """The one-scenario batch behind ``slp``, printing scenario 0's state after each sub-LP solve."""

    def _solve_phase(self, fr, sel, delta):
        out = super()._solve_phase(fr, sel, delta)
        e = self.lp_log[0][-1]
        print(f"it {self.iter[0]:3d} fr {int(fr)} LP status {e[0]} obj {e[1]} newton {e[3]} |p| {np.abs(out[0][0]).max():.3e} "
              f"delta {getattr(self, 'delta', [0])[0]:.3e} prim {self.prim_infeas[0]:.3e} dual {self.dual_infeas[0]:.3e} "
              f"compl {self.compl[0]:.3e} f {self.f[0]:.9f}", flush=True)
        return out


slp = (SlpLS if a == "LS" else SlpTR)(mdl)
slp._batch = Traced
import time
t0 = time.time()
slp.run()
print("wall", time.time() - t0)
print("ret", slp.ret, "iter", slp.iter, "obj", slp.obj_val)
