"""Developer tool: B load scenarios of a case solved to the end by a lock-step batched SLP driver.
python tools/gpu_slp_batch.py case118 64 [max_iter] [dev] [--algorithm {ls,tr}]"""
import argparse, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g
g.build()
import bench
from activesetmethods_b200.examples import acopf
from activesetmethods_b200.slp import Parameters, SlpLSBatch, SlpTRBatch
ap = argparse.ArgumentParser()
ap.add_argument("case")
ap.add_argument("B", type=int)
ap.add_argument("max_iter", type=int, nargs="?", default=40)
ap.add_argument("dev", nargs="?", choices=["dev"], help="device-side ACOPF evaluator instead of the host callbacks")
ap.add_argument("--algorithm", choices=["ls", "tr"], default="ls", help="Line Search (default) or Trust Region")
a = ap.parse_args()
case, B, dev = a.case, a.B, a.dev == "dev"
tr = a.algorithm == "tr"
net = bench.network(case)
probs = [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(B)]
t0 = time.time()
cls = SlpTRBatch if tr else SlpLSBatch
b = cls(probs, Parameters(algorithm="Trust Region" if tr else "Line Search", max_iter=a.max_iter,
                          lp_options=dict(eps_rel=1e-6, max_iter=4000000)), device_evaluator=dev).run()
dt = time.time() - t0
solved = int(np.isin(b.ret, (0, 6)).sum())
print(f"{case} x {B} {cls.__name__} ({'device' if dev else 'host'} evaluator, max_iter {a.max_iter}): {b.rounds} lock-step "
      f"rounds ({b.two_phase_rounds} with two phase solves), statuses {dict(zip(*np.unique(b.ret, return_counts=True)))}, "
      f"SLP iterations min/mean/max {b.iter.min()}/{b.iter.mean():.1f}/{b.iter.max()}, sub-LP solves per scenario "
      f"min/mean/max {b.lp_solves.min()}/{b.lp_solves.mean():.1f}/{b.lp_solves.max()}, LP iterations {b.lp_iterations:.3g}, "
      f"wall {dt:.1f}s -> {B / dt:.2f} scenarios/s (full SLP solves), {solved} solved (status 0 or 6) -> "
      f"{solved / dt:.2f} solved scenarios/s, objective mean {b.obj_val.mean():.4f}")
if tr:
    print(f"final trust-region radius min/median/max {b.delta.min():.3e}/{np.median(b.delta):.3e}/{b.delta.max():.3e}")
