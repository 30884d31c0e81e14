"""Developer tool: all non-islanding N-1 branch outages of a case, solved to the end by the lock-step line-search driver
with the device-side evaluator, in two ways in one process:
  (a) one handle of `lanes` lanes, refilled from the queue of outages as runs end (continuous batching, `lanes=`);
  (b) consecutive lock-step batches of `lanes` outages, a new handle for each.
python tools/gpu_contingency_queue.py [case] [lanes] [max_iter]      (defaults: case1354pegase 1024 40)"""
import argparse, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g
g.build()
import bench
from activesetmethods_b200.examples import acopf
from activesetmethods_b200.slp import Parameters, SlpLSBatch


def card():
    """The card's name, power limit and top SM clock, printed beside the numbers they qualify."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True).stdout.strip()
    except FileNotFoundError:
        out = "nvidia-smi not found"
    print(out, flush=True)


ap = argparse.ArgumentParser()
ap.add_argument("case", nargs="?", default="case1354pegase")
ap.add_argument("lanes", type=int, nargs="?", default=1024)
ap.add_argument("max_iter", type=int, nargs="?", default=40)
a = ap.parse_args()
card()

net = bench.network(a.case)
t0 = time.time()
probs = [acopf.AcopfModel(n) for n in acopf.branch_contingencies(net)]
N = len(probs)
print(f"{a.case}: {net.nl} branches, {N} non-islanding outages, models built in {time.time() - t0:.1f}s; "
      f"{a.lanes} lanes, line search, device evaluator, max_iter {a.max_iter}", flush=True)
# round 6's LP options (tools/gpu_contingency_batch.py)
prm = lambda: Parameters(algorithm="Line Search", max_iter=a.max_iter,  # noqa: E731
                         lp_options=dict(eps_rel=1e-6, max_iter=4000000))


class Probe(SlpLSBatch):
    """Records how long building the handle (allocation + attach) took, and the wall time of the first sub-LP batch
    solve, which carries the barrier engine's host symbolic analysis and graph capture."""
    create_s = 0.0
    first_lp_time = None

    def _instantiate(self):
        t0 = time.time()
        opt = super()._instantiate()
        self.create_s = time.time() - t0
        return opt

    def _solve_phase(self, fr, sel, delta):
        out = super()._solve_phase(fr, sel, delta)
        if self.first_lp_time is None:
            self.first_lp_time = self.lp_time
        return out


def report(label, wall, create, first_solve, rounds, two_phase, ret, it):
    solved = int(np.isin(ret, (0, 6)).sum())
    print(f"{label}: wall {wall:.1f}s, handle creation {create:.2f}s + first sub-LP batch solve {first_solve:.2f}s "
          f"(symbolic analysis included), {rounds} rounds ({two_phase} with two phase solves), statuses "
          f"{dict(zip(*np.unique(ret, return_counts=True)))}, SLP iterations min/mean/max {it.min()}/{it.mean():.1f}/"
          f"{it.max()}, {solved} solved (status 0 or 6) -> {solved / wall:.2f} solved scenarios/s", flush=True)


# (a) one handle, refilled from the queue
t0 = time.time()
q = Probe(probs, prm(), device_evaluator=True, lanes=a.lanes).run()
wall_a = time.time() - t0
report(f"(a) queue, one handle of {a.lanes} lanes", wall_a, q.create_s, q.first_lp_time, q.rounds, q.two_phase_rounds,
       q.ret, q.iter)
print(f"    loads: {len(q.loads)} load_lanes calls, lanes per call min/mean/max "
      f"{min(len(l) for _, l in q.loads)}/{np.mean([len(l) for _, l in q.loads]):.1f}/"
      f"{max(len(l) for _, l in q.loads)}" if q.loads else "    loads: none", flush=True)
q.optimizer.close()

# (b) consecutive batches, a new handle each
t0 = time.time()
ret, it, rounds, two, create, first = [], [], 0, 0, 0.0, 0.0
for c0 in range(0, N, a.lanes):
    b = Probe(probs[c0:c0 + a.lanes], prm(), device_evaluator=True).run()
    ret.append(b.ret)
    it.append(b.iter)
    rounds += b.rounds
    two += b.two_phase_rounds
    create += b.create_s
    first += b.first_lp_time
    print(f"    chunk {c0}..{c0 + len(b.ret) - 1}: {b.rounds} rounds, {time.time() - t0:.1f}s so far", flush=True)
    b.optimizer.close()
wall_b = time.time() - t0
report(f"(b) {-(-N // a.lanes)} consecutive batches of <= {a.lanes}, a new handle each", wall_b, create, first, rounds,
       two, np.concatenate(ret), np.concatenate(it))
same = np.array_equal(q.ret, np.concatenate(ret)) and np.array_equal(q.iter, np.concatenate(it))
print(f"(a) vs (b): wall {wall_a:.1f}s vs {wall_b:.1f}s ({wall_b / wall_a:.2f}x); per-problem statuses and "
      f"iteration counts {'identical' if same else 'differ'}", flush=True)
card()
