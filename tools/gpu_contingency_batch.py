"""Developer tool: an N-1 contingency batch of ACOPF solved to the end by the lock-step line-search driver with the
device-side evaluator, next to the load batch of the same network and size, and the device time of one evaluation with
shared and with per-scenario branch coefficients.
python tools/gpu_contingency_batch.py [case] [B] [max_iter]      (defaults: case1354pegase 1024 40)"""
import argparse, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g
g.build()
import bench
import torch
from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf
from activesetmethods_b200.slp import Parameters, SlpLSBatch
from activesetmethods_b200.sublp import SubLp


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
ap.add_argument("B", type=int, nargs="?", default=1024)
ap.add_argument("max_iter", type=int, nargs="?", default=40)
ap.add_argument("--reps", type=int, default=20, help="timed evaluator calls per layout and pass")
a = ap.parse_args()
card()

net = bench.network(a.case)
t0 = time.time()
outages = acopf.branch_contingencies(net, a.B)
if len(outages) < a.B:
    sys.exit(f"{a.case} has only {len(outages)} non-islanding branch outages")
cont = [acopf.AcopfModel(n) for n in outages]
print(f"{a.case}: {net.nl} branches, first {a.B} non-islanding outages (last: branch "
      f"{int(np.argmin(outages[-1].br_status))}), models built in {time.time() - t0:.1f}s", flush=True)
loads = [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(a.B)]
prm = lambda: Parameters(algorithm="Line Search", max_iter=a.max_iter,  # noqa: E731
                         lp_options=dict(eps_rel=1e-6, max_iter=4000000))


def run(label, probs):
    t0 = time.time()
    b = SlpLSBatch(probs, prm(), device_evaluator=True).run()
    dt = time.time() - t0
    solved = int(np.isin(b.ret, (0, 6)).sum())
    print(f"{label}: {a.case} x {a.B} SlpLSBatch (device evaluator, max_iter {a.max_iter}): {b.rounds} lock-step rounds "
          f"({b.two_phase_rounds} with two phase solves), statuses {dict(zip(*np.unique(b.ret, return_counts=True)))}, "
          f"SLP iterations min/mean/max {b.iter.min()}/{b.iter.mean():.1f}/{b.iter.max()}, LP iterations "
          f"{b.lp_iterations:.3g}, wall {dt:.1f}s -> {a.B / dt:.2f} scenarios/s (full SLP solves), {solved} solved "
          f"(status 0 or 6) -> {solved / dt:.2f} solved scenarios/s, objective mean {b.obj_val.mean():.4f}", flush=True)
    b.optimizer.close()


run("N-1 branch outages", cont)
run("load scenarios", loads)

# one asm_slp_eval_acopf (x upload from pinned memory, the three evaluator kernels, the sub-LP data push) with the
# coefficients shared by the batch and per scenario, alternating, CUDA events on the handle's stream
m0 = cont[0]
arr = lambda k: np.array([getattr(m, k) for m in cont])  # noqa: E731
lp = SubLp(m0.n, m0.m, m0.j_str, arr("x_L"), arr("x_U"), arr("g_L"), arr("g_U"), batch=a.B)
x = torch.empty((a.B, m0.n), dtype=torch.float64, pin_memory=True).numpy()
x[:] = [np.clip(m.x0, m.x_L, m.x_U) for m in cont]
coef = np.ascontiguousarray(np.stack([lp._acopf_arrays(m)["coef"] for m in cont]))
print(f"per-scenario coefficients: {coef.nbytes / 1e6:.0f} MB (L2 126 MB: read from HBM)", flush=True)
times = {"shared": [], "per-scenario": []}
for _ in range(2):
    for mode in times:
        lp.attach_acopf(acopf.AcopfModel(net))
        if mode == "per-scenario":
            capi.check(lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(coef)))
        for _ in range(3):
            lp.eval_acopf(x, 1000.0, False)
        lp.timer_start()
        for _ in range(a.reps):
            lp.eval_acopf(x, 1000.0, False)
        times[mode].append(lp.timer_stop() / a.reps)
for mode, t in times.items():
    print(f"asm_slp_eval_acopf, {mode} coefficients: {' / '.join(f'{v:.3f}' for v in t)} ms per call "
          f"(two passes of {a.reps} calls)", flush=True)
lp.close()
card()
