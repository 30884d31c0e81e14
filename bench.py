#!/usr/bin/env python
"""Benchmark of the SLP sub-LP hot path (BASELINE.json: "scenarios/s batched", config 5: load-perturbed
case1354pegase scenarios split across the GPUs).

A *step* is one pass of the per-iteration hot path of the reference
(``sub_optimize!`` src/algorithms/subproblem.jl:229-542 + the merit reductions of src/algorithms/slp.jl:79-147)
over one batch of scenarios: Jacobian assembly + sub-LP bounds, the LP solve to ``--eps`` (1e-6, the parity bar),
the multiplier read-back with the reference's masking, the violation norm and the merit derivative.

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle's HiGHS simplex on all host cores

The job is fixed (``--scenarios``, default 1024 = BASELINE config 5) and split over the GPUs: strong scaling.  At
N = 1 the line also carries BASELINE's single-instance figures (sub-LP ms and SLP iterations/s on case13659pegase)
under ``single_instance``.  One JSON line is printed by rank 0.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes what the last timed step returned as ``DIR/<name>.npy`` (float64, at most 64 MB): the inputs depend
only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "sub-LP scenarios/s (SLP hot path: assembly + bounds + LP solve to 1e-6 objective accuracy + read-back + merit)"
UNIT = "scenarios/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--case", default="case1354pegase")
    ap.add_argument("--scenarios", type=int, default=1024,
                    help="scenarios of the whole job (BASELINE config 5: 1024), split over the GPUs")
    ap.add_argument("--single-case", default="case13659pegase",
                    help="instance of the single-instance metrics reported at N = 1 (sub-LP ms, SLP it/s); 'none' skips them")
    ap.add_argument("--single-slp-iters", type=int, default=60)
    ap.add_argument("--eps", type=float, default=5e-7,
                    help="relative KKT tolerance; 5e-7 keeps |pobj - dobj| / |obj| below the 1e-6 parity bar")
    ap.add_argument("--delta", type=float, default=1000.0, help="step bound (Line Search uses 1000, slp.jl:23)")
    ap.add_argument("--engine", type=int, default=0, help="0 / 4 barrier engine, 5 PDHG hybrid, 1 / 2 PDHG streaming / group")
    ap.add_argument("--max-iter", type=int, default=4_000_000)
    ap.add_argument("--cpu-sample", type=int, default=2, help="scenarios of the cpu_baseline sample")
    ap.add_argument("--ref-sample", type=int, default=0, help="scenarios per reference step (0 = one per core)")
    ap.add_argument("--workload", default="batch", choices=["batch", "single"],
                    help="batch: scenario batch per GPU (default, the driver's metric); single: one instance "
                         "(BASELINE config 4) -- group engine at N = 1, row-partitioned over NCCL at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0's "
                         "scenarios; full vectors for a fixed, seeded sample of them)")
    return ap.parse_args()


DUMP_LIMIT = 64 * 10**6


def dump_sample(n_scen, row_bytes, budget=32 << 20, cap=64):
    """Indices of a fixed, seeded sample of scenarios whose full output vectors together fit `budget` bytes."""
    k = max(1, min(n_scen, cap, budget // max(1, row_bytes)))
    return np.sort(np.random.default_rng(0).choice(n_scen, k, replace=False))


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy in float64 (integers and statuses are exact in it)."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


# ------------------------------------------------------------------------------------------------------------
# workload: first SLP linearisation (midpoint start, examples/acopf/init_opf.jl:25-29) of load scenarios
# ------------------------------------------------------------------------------------------------------------
def network(case):
    from activesetmethods_b200.examples import acopf
    if case == "case9":
        return acopf.case9()
    return acopf.synthetic_network(*acopf.PEGASE_SHAPES[case])


def linearise(net, scenario_ids):
    """Host NLP evaluation (the JuMP evaluator's role, MOI_wrapper.jl:1047-1069) of every scenario at x0."""
    from activesetmethods_b200.examples import acopf
    out = dict(x=[], f=[], df=[], E=[], dE=[], gL=[], gU=[], xL=[], xU=[])
    mdl0 = None
    for sid in scenario_ids:
        mdl = acopf.AcopfModel(acopf.perturb_loads(net, sid))
        mdl0 = mdl0 or mdl
        x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
        out["x"].append(x)
        out["f"].append(mdl.eval_f(x))
        out["df"].append(mdl.eval_grad_f(x, np.zeros(mdl.n)))
        out["E"].append(mdl.eval_g(x, np.zeros(mdl.m)))
        out["dE"].append(mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz)))
        out["gL"].append(mdl.g_L)
        out["gU"].append(mdl.g_U)
        out["xL"].append(mdl.x_L)
        out["xU"].append(mdl.x_U)
    return mdl0, {k: np.ascontiguousarray(np.array(v, dtype=np.float64)) for k, v in out.items()}


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# CPU arm (oracle: restated sub-LP build + HiGHS dual simplex) -- the checker used as the reported baseline
# ------------------------------------------------------------------------------------------------------------
_W = {}


def _cpu_init(case):
    from oracle import slp_oracle as so
    net = network(case)
    _W["net"], _W["so"] = net, so


def _cpu_solve(args):
    sid, delta = args
    so = _W["so"]
    mdl, d = linearise(_W["net"], [sid])
    pat = so.JacobianPattern(mdl.m, mdl.n, mdl.j_str)
    ref = so.SubLp(pat, d["gL"][0], d["gU"][0], d["xL"][0], d["xU"][0])
    t0 = time.perf_counter()
    out = ref.solve(pat.assemble(d["dE"][0]), d["df"][0], d["f"][0], d["E"][0], d["x"][0], delta, False)
    return time.perf_counter() - t0, int(out[5]), ref.last_objective


def cpu_baseline(case, delta, n_scen):
    _cpu_init(case)
    t0 = time.perf_counter()
    res = [_cpu_solve((1 + s, delta)) for s in range(n_scen)]
    dt = time.perf_counter() - t0
    solve_t = sum(r[0] for r in res)
    return {"value": n_scen / solve_t, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n_scen} scenarios of {case} (first SLP linearisation), oracle sub-LP build + HiGHS dual "
                      f"simplex, 1 thread, {solve_t:.1f} s of solve time ({dt:.1f} s wall incl. host NLP evaluation)",
            "objectives": [r[2] for r in res]}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_step = a.ref_sample or cores
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(a.case,)) as pool:
        def step(k):
            ids = [(1 + k * per_step + s, a.delta) for s in range(per_step)]
            t0 = time.perf_counter()
            res = pool.map(_cpu_solve, ids, chunksize=1)
            return time.perf_counter() - t0, res
        for k in range(a.warmup):
            step(k)
        t_total, n_ok = 0.0, 0
        for k in range(a.steps):
            dt, res = step(a.warmup + k)
            t_total += dt
            n_ok += sum(1 for r in res if r[1] == 0)
    if a.dump_outputs:
        last = a.warmup + a.steps - 1
        dump_outputs(a.dump_outputs, dict(
            scenario_id=[1 + last * per_step + s for s in range(per_step)], status=[r[1] for r in res],
            objective=[np.nan if r[2] is None else r[2] for r in res]))
    value = per_step * a.steps / t_total
    sample = (f"{per_step} scenarios of {a.case} per step over a {cores}-process pool (one HiGHS dual simplex per "
              f"core), host NLP evaluation included in the step")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * t_total / a.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{a.case} load scenarios, first SLP linearisation, sub-LP to simplex tolerance 1e-9",
                   "scenarios_per_step": per_step, "delta": a.delta, "optimal": n_ok},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def kkt_bytes(st, B):
    """Algorithmic bytes of one numeric factorisation and of one substitution pair of a batch of B LPs (DESIGN.md
    section 4.4).  A level's kernel must read every distinct f64 operand it uses once and read + write every target once;
    nothing survives in L2 from one level to the next when the batch working set (nnz(L) * B * 8 bytes) is much larger
    than L2.  Index lists are read once per warp, i.e. once per 32 scenarios.  Operands that several chunks of one
    level share are counted once -- the kernel re-reads them (from L1 / L2), so this is a lower bound of what it moves
    and `achieved` is conservative.  With supernodes a "level" is a step of the supernodal schedule and the panels are
    in the same two counters (every panel entry read and written once, the factorised diagonal block read once per row
    task): the symbolic analysis adds them, csrc/kkt_symbolic.hpp."""
    fr, ft = st["factor_distinct_reads"], st["factor_targets"]
    sr, stg = st["substitution_distinct_reads"], st["substitution_targets"]
    nnzL, N, terms = st["nnz_L"], st["kkt_dim"], st["terms"]
    per_lp_factor = 8 * fr + 16 * ft + 8 * nnzL + 8 * nnzL // 2 + 16 * N   # + clear W, scatter K, pivots in / out
    per_lp_pair = 8 * sr + 16 * stg + 24 * N                                # + the diagonal pass
    warps = max(1, B // 32)
    return B * per_lp_factor + warps * 16 * terms, B * per_lp_pair + warps * 32 * nnzL


def single_instance(a, local):
    """BASELINE's first metric on its own config: sub-LP ms and SLP iterations/s on case13659pegase (one GPU)."""
    from activesetmethods_b200.slp import Model, Parameters, SlpLS
    from activesetmethods_b200.sublp import SubLp
    from activesetmethods_b200.examples import acopf
    t0 = time.perf_counter()
    net = network(a.single_case)
    mdl = acopf.AcopfModel(net)
    t_model = time.perf_counter() - t0
    x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    args = (x, mdl.eval_f(x), mdl.eval_grad_f(x, np.zeros(mdl.n)), mdl.eval_g(x, np.zeros(mdl.m)),
            mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz)), a.delta, False)
    t0 = time.perf_counter()
    lp = SubLp(mdl.n, mdl.m, mdl.j_str, mdl.x_L, mdl.x_U, mdl.g_L, mdl.g_U, device=local, eps_rel=a.eps, engine=a.engine)
    lp.sub_optimize(*args)                                   # first call: symbolic analysis + graph capture
    t_first = time.perf_counter() - t0
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        out = lp.sub_optimize(*args)
        times.append(time.perf_counter() - t0)
    info = lp.last_info[0]
    loop_ms, its = lp.last_solve_timing()
    st = lp.ipm_info() if lp.engine_info()["engine"] == 4 else {}
    lp.close()
    # SLP line search (reference defaults: tolerances 1e-2, Delta = 1000) with the device-side NLP evaluator
    prm = Parameters(algorithm="Line Search", max_iter=a.single_slp_iters, device=local, device_evaluator=True,
                     lp_options=dict(eps_rel=a.eps, engine=a.engine))
    slp = SlpLS(Model.from_problem(mdl, prm))
    t0 = time.perf_counter()
    slp.run()
    t_slp = time.perf_counter() - t0
    n_lp = len(slp.lp_log)
    return {"case": a.single_case, "n": mdl.n, "m": mdl.m, "nnz_coo": mdl.nnz,
            "sub_lp_ms": 1e3 * float(np.median(times)), "sub_lp_device_ms": loop_ms, "sub_lp_status": int(out[5]),
            "sub_lp_objective": info["objective"], "sub_lp_newton_steps": int(info["iterations"]),
            "first_call_s": t_first, "symbolic_ms": st.get("symbolic_ms"), "kkt": st,
            "slp_iter_per_s": slp.iter / t_slp, "slp_iterations": int(slp.iter), "slp_sub_lps": n_lp,
            "slp_status": int(slp.ret), "slp_objective": float(slp.obj_val), "slp_violation": float(slp.prim_infeas),
            "slp_wall_s": t_slp, "slp_lp_statuses": sorted(set(int(e[0]) for e in slp.lp_log)),
            "note": f"Line Search, reference tolerances (1e-2), at most {a.single_slp_iters} SLP iterations, device-side "
                    f"ACOPF evaluator; host model build {t_model:.1f} s not included"}


def run_ours(a):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        g.build()
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    from activesetmethods_b200 import capi, shard
    from activesetmethods_b200.sublp import SubLp
    lib = capi.load()
    if lib.asm_device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)

    total_scen = a.scenarios
    net = network(a.case)
    ids = shard.split_scenarios(total_scen, world)[rank]     # strong scaling: contiguous blocks of scenario ids (= seeds)
    S = len(ids)
    t0 = time.perf_counter()
    mdl, d = linearise(net, ids)
    t_host_eval = time.perf_counter() - t0
    n, m, nnz = mdl.n, mdl.m, mdl.nnz
    lp = SubLp(n, m, mdl.j_str, d["xL"], d["xU"], d["gL"], d["gU"], batch=S, device=local, eps_rel=a.eps,
               engine=a.engine, max_iter=a.max_iter)
    nnz_csr = lp.nnz_csr

    def pinned(shape, dtype=torch.float64):
        return torch.empty(shape, dtype=dtype).pin_memory().numpy()

    hin = {k: pinned(d[k].shape) for k in ("x", "f", "df", "E", "dE")}
    for k in hin:
        hin[k][...] = d[k]
    hdelta = pinned((S,))
    hdelta[...] = a.delta
    hout = dict(p=pinned((S, n)), lam=pinned((S, m)), mu_u=pinned((S, n)), mu_l=pinned((S, n)),
                slack=pinned((S, m, 2)), viol=pinned((S,)), deriv=pinned((S,)), nu=pinned((S, m)))
    hstatus = torch.empty(S, dtype=torch.int32).pin_memory().numpy()
    info = (capi.LpInfo * S)()
    P = capi.dptr

    def e2e_step():
        """What a caller of the plugin does per SLP iteration: host buffers in, host results out."""
        capi.check(lib.asm_slp_sub_optimize(
            lp._h, P(hin["x"]), P(hin["f"]), P(hin["df"]), P(hin["E"]), P(hin["dE"]), P(hdelta), 0,
            C.byref(lp.params), P(hout["p"]), P(hout["lam"]), P(hout["mu_u"]), P(hout["mu_l"]), P(hout["slack"]),
            hstatus.ctypes.data_as(capi.c_int32_p), info))
        capi.check(lib.asm_slp_norm_violations(lp._h, None, None, 0, P(hout["viol"])))
        np.abs(hout["lam"], out=hout["nu"])                   # compute_nu!, slp_line_search.jl:251-261
        capi.check(lib.asm_slp_merit_derivative(lp._h, P(hout["nu"]), 0, P(hout["deriv"])))

    def resident_step():
        """Same work with x_k, df, E, dE already in HBM: device time from CUDA events on the handle's stream."""
        lp.timer_start()
        lp.reassemble(False)
        capi.check(lib.asm_slp_solve(lp._h, C.byref(lp.params), info))
        lp.extract_device()
        capi.check(lib.asm_slp_norm_violations(lp._h, None, None, 0, P(hout["viol"])))
        return lp.timer_stop()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        return shard.max_over_ranks(x, device="cuda" if world > 1 else None)

    def sum_over_ranks(x):
        return shard.sum_over_ranks(x, device="cuda" if world > 1 else None)

    # ---- warm-up: full steps (the first one runs the symbolic analysis and captures the CUDA graphs)
    lp.update(hin["x"], hin["f"], hin["df"], hin["E"], hin["dE"], hdelta, False)   # inputs resident
    t0 = time.perf_counter()
    resident_step()
    t_first = time.perf_counter() - t0
    for _ in range(max(0, a.warmup - 2)):
        resident_step()
    e2e_step()
    eng = lp.engine_info()
    kst = lp.ipm_info() if eng["engine"] == 4 else None      # sizes; the per-solve counters are refreshed below
    # timing rule: inputs larger than L2, or flush L2 between timed steps (outside the timed region)
    Bpad = 1 if S <= 1 else (32 if S <= 32 else ((S + 63) // 64) * 64)
    working_set = Bpad * (8 * (kst["nnz_L"] + 2 * kst["kkt_dim"]) if kst else (16 * nnz_csr + 64 * n + 48 * m))
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if working_set < 2 * (126 << 20) else None

    def flush_l2():
        if flush_buf is not None:
            flush_buf.zero_()
            torch.cuda.synchronize()

    # ---- timed, inputs resident in HBM: CUDA events on the handle's stream
    clocks = ClockSampler(local)
    sync_all()
    clocks.start()
    l0 = lp.launch_count()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(a.steps):
        flush_l2()
        dev_ms += resident_step()
    sync_all()
    wall_resident = time.perf_counter() - t0
    launches = lp.launch_count() - l0
    infos = [dict(status=int(i.status), iterations=int(i.iterations), objective=float(i.objective),
                  pres=float(i.primal_residual), dres=float(i.dual_residual), gap=float(i.gap)) for i in info[:S]]
    loop_ms, loop_its = lp.last_solve_timing()
    dumped = None
    if a.dump_outputs and rank == 0:
        # the last resident step left its results on the device: read them back outside the timed region; copies,
        # because the end-to-end steps below reuse the host buffers
        capi.check(lib.asm_slp_extract(lp._h, P(hout["p"]), P(hout["lam"]), P(hout["mu_u"]), P(hout["mu_l"]),
                                       P(hout["slack"]), hstatus.ctypes.data_as(capi.c_int32_p)))
        rows = dump_sample(S, 8 * (3 * n + 3 * m))
        dumped = {"scenario_id": np.array(ids), "status": hstatus.copy(), "objective": [i["objective"] for i in infos],
                  "violation": hout["viol"].copy(), "sample_scenario_id": np.array(ids)[rows], "p": hout["p"][rows],
                  "lambda": hout["lam"][rows], "mult_x_U": hout["mu_u"][rows], "mult_x_L": hout["mu_l"][rows],
                  "p_slack": hout["slack"][rows]}
    dev_s = max_over_ranks(dev_ms * 1e-3)
    # ---- timed, end to end through the C ABI with pinned host buffers (same number of steps)
    sync_all()
    e2e_wall = 0.0
    for _ in range(a.steps):
        flush_l2()
        sync_all()
        t0 = time.perf_counter()
        e2e_step()
        torch.cuda.synchronize()
        e2e_wall += time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_wall)
    clk = clocks.stop()
    n_opt = sum_over_ranks(float(sum(1 for i in infos if i["status"] == 0)))
    its_max = max_over_ranks(float(max(i["iterations"] for i in infos)))
    its_sum = sum_over_ranks(float(sum(i["iterations"] for i in infos)))
    value = total_scen * a.steps / dev_s
    e2e = total_scen * a.steps / e2e_s
    h2d = 8 * S * (2 * n + m + nnz + 2) + 8 * S * m          # sub_optimize inputs + nu
    d2h = 8 * S * (3 * n + m + 2 * m) + 4 * S + 8 * S * 2    # p, lambda, mu_U, mu_L, slacks, status, 2 merit scalars

    # ---- roofline of the dominant kernel, measured live with CUDA events on the handle's stream
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if kst is not None:
        kst = lp.ipm_info()
        fac_ms, pair_ms = lp.ipm_timing(10)
        by_fac, by_pair = kkt_bytes(kst, Bpad)
        newton = its_sum / total_scen
        if os.path.exists(tpath):
            try:
                sched = "levels" if os.environ.get("ASM_IPM_SUPERNODE") == "1" else "supernodal"
                traffic = json.load(open(tpath)).get(f"ldl_factor:{sched}:{a.case}:{S}")
            except (OSError, ValueError):
                traffic = None
        achieved = by_fac / (fac_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic,
                    "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s",
                    "kernel": "one numeric L D L' of the KKT matrices of the whole batch, replayed as one CUDA graph: per step "
                              "of the supernodal schedule k_sn_diag + k_sn_rows (dense panels of the supernodes) and "
                              "k_ldl_factor (chunked updates that leave them)",
                    "bytes_per_launch": by_fac, "factor_ms": fac_ms, "launches_per_factorisation": kst["launches_factor"],
                    "substitution_pair_ms": pair_ms, "substitution_pair_bytes": by_pair,
                    "substitution_pair_gbs": by_pair / (pair_ms * 1e-3) / 1e9,
                    "newton_steps_mean": newton, "kkt": kst,
                    "share_of_step": {"factor": kst["factorisations"] * fac_ms / (1e3 * dev_s / a.steps),
                                      "substitutions": kst["substitution_pairs"] * pair_ms / (1e3 * dev_s / a.steps)}}
    else:
        pm, dm = lp.kernel_timing(50)
        by_primal = Bpad * (8 * nnz_csr + 8 * m + 56 * n) + 4 * nnz_csr + 4 * (n + 1)
        by_dual = Bpad * (8 * nnz_csr + 8 * n + 40 * m) + 4 * nnz_csr + 4 * (m + 1)
        achieved = (by_primal + by_dual) / ((pm + dm) * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": None,
                    "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s",
                    "kernel": "k_primal2 + k_dual2 (one PDHG iteration of the whole batch)",
                    "bytes_per_launch_pair": by_primal + by_dual, "primal_ms": pm, "dual_ms": dm,
                    "loop_ms_per_iteration": loop_ms / max(loop_its, 1)}

    cpu = None
    single = None
    if rank == 0 and world == 1 and a.cpu_sample > 0:
        cpu = cpu_baseline(a.case, a.delta, a.cpu_sample)
        # the same scenarios on the GPU against the checker: relative objective difference (parity bar 1e-6)
        rels = [abs(infos[s]["objective"] - obj) / max(1.0, abs(obj))
                for s, obj in enumerate(cpu.pop("objectives")) if obj is not None and infos[s]["status"] == 0]
        cpu["gpu_objective_rel_diff_max"] = max(rels) if rels else None
        cpu["gpu_objective_parity_1e-6"] = bool(rels) and max(rels) <= 1e-6
    lp.close()
    if rank == 0 and world == 1 and a.single_case != "none":
        single = single_instance(a, local)
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * dev_s / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{total_scen} load-perturbed {a.case} scenarios (BASELINE config 5), split over the "
                                   f"GPUs ({S} on rank 0), first SLP linearisation, Line Search step bound {a.delta:g}",
                       "scenarios_total": total_scen, "scenarios_per_gpu": S,
                       "n": n, "m": m, "nnz_coo": nnz, "nnz_csr": nnz_csr, "eps_rel": a.eps,
                       "engine": eng, "optimal": int(n_opt), "lp_iterations_max": int(its_max),
                       "lp_iterations_mean": its_sum / total_scen,
                       "worst_relative_residuals": {
                           "primal": max(i["pres"] for i in infos), "dual": max(i["dres"] for i in infos),
                           "gap": max(i["gap"] / (1.0 + 2.0 * abs(i["objective"])) for i in infos)},
                       "warmup_steps": f"{a.warmup} full steps ({max(0, a.warmup - 1)} resident + 1 end-to-end); the first "
                                       f"one ({t_first:.2f} s) includes the symbolic analysis and the CUDA-graph capture",
                       "l2": ("no flush: the factorisation working set (%.0f MB) exceeds the 126 MB L2"
                              if flush_buf is None else
                              "working set %.0f MB: L2 flushed between timed steps by writing 256 MB")
                             % (working_set / 1e6),
                       "host_nlp_evaluation_s": t_host_eval, "wall_s_resident": wall_resident},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": a.steps, "ms_per_step": 1e3 * e2e_s / a.steps},
            "gpu_launches": int(launches), "roofline": roofline, "clocks": clk,
        }
        if cpu is not None:
            out["cpu_baseline"] = cpu
        if single is not None:
            out["single_instance"] = single
        if dumped is not None:
            dump_outputs(a.dump_outputs, dumped)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_single(a):
    """One sub-LP of one instance: `SubLp` (persistent group kernel) on one GPU, `B200RowPartitionedLP` on several."""
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        g.build()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("gloo")
        dist.barrier()
    from activesetmethods_b200 import capi, shard
    from activesetmethods_b200.sublp import SubLp, B200RowPartitionedLP, nccl_unique_id
    net = network(a.case)
    mdl, d = linearise(net, [1])
    n, m, nnz = mdl.n, mdl.m, mdl.nnz
    lp = SubLp(n, m, mdl.j_str, d["xL"][0], d["xU"][0], d["gL"][0], d["gU"][0], batch=1, device=local, eps_rel=a.eps,
               engine=a.engine, max_iter=a.max_iter)
    args = (d["x"][0], d["f"][0], d["df"][0], d["E"][0], d["dE"][0], a.delta, False)
    lp.update(*args)
    if world == 1:
        def step():
            t0 = time.perf_counter()
            out = lp.sub_optimize(*args)
            dt = time.perf_counter() - t0
            res = dict(zip(("p", "lambda", "mult_x_U", "mult_x_L", "p_slack", "status"), out))
            return dt, lp.last_info[0], lp.last_solve_timing(), res
    else:
        rp, ci, vals = lp.jacobian_csr()                       # device-assembled CSR of this linearisation
        x = d["x"][0]
        lb = np.maximum(-a.delta, d["xL"][0] - x)              # subproblem.jl:427-434
        ub = np.minimum(a.delta, d["xU"][0] - x)
        gl, gu, E = d["gL"][0], d["gU"][0], d["E"][0]
        eq = gl == gu
        rl = np.where(np.isfinite(gl), gl - E, -np.inf)        # subproblem.jl:461-484
        ru = np.where(eq, gl - E, np.where(np.isfinite(gu), gu - E, np.inf))
        ids = [nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        plp = B200RowPartitionedLP(n, m, rp, ci, rank, world, ids[0], device=local, eps_rel=a.eps, max_iter=a.max_iter)

        def step():
            dist.barrier()
            t0 = time.perf_counter()
            plp.set_matrix_values(vals)
            plp.set_objective(d["df"][0], float(d["f"][0]))
            plp.set_col_bounds(lb, ub)
            plp.set_row_bounds(rl, ru)
            info = plp.optimize()[0]
            primal = plp.primal()
            row_dual = plp.row_dual()
            return time.perf_counter() - t0, info, (0.0, info["iterations"]), {"primal": primal, "row_dual": row_dual}
    for _ in range(a.warmup):
        step()
    clocks = ClockSampler(local)
    clocks.start()
    tot, info, timing = 0.0, None, None
    for _ in range(a.steps):
        dt, info, timing, res = step()
        tot += dt
    clk = clocks.stop()
    tot = shard.max_over_ranks(tot)
    if rank == 0:
        loop_ms, its = timing
        b_iter = 24 * lp.nnz_csr + 76 * n + 60 * m + 8           # SURVEY.md 8(d), single LP
        out = {"metric": "sub-LP solves/s, single instance (config 4)", "value": a.steps / tot, "unit": "sub-LP/s",
               "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": {"workload": f"{a.case} single instance, first SLP linearisation, step bound {a.delta:g}",
                          "n": n, "m": m, "nnz_csr": lp.nnz_csr, "eps_rel": a.eps, "status": info["status"],
                          "objective": info["objective"], "pdhg_iterations": info["iterations"],
                          "engine": lp.engine_info() if world == 1 else "row-partitioned, NCCL all-reduce per iteration",
                          "us_per_iteration": 1e6 * tot / a.steps / max(1, info["iterations"]),
                          "algorithmic_GBs": b_iter * info["iterations"] / (tot / a.steps) / 1e9},
               "e2e": {"value": a.steps / tot, "unit": "sub-LP/s", "h2d_bytes_per_step": 8 * (2 * n + m + nnz + 2),
                       "d2h_bytes_per_step": 8 * (3 * n + 3 * m)},
               "clocks": clk}
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {"status": info["status"], "objective": info["objective"], **res})
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "single":
        run_single(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
