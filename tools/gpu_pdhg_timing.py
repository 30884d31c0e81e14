"""Device time of the PDHG hot kernels: one streaming primal / dual half iteration (k_primal2 / k_dual2 at B = 128) and
the per-iteration time of a single-LP group-kernel solve (engine 2), on case1354pegase sub-LPs.  Prints one JSON line.

    python tools/gpu_pdhg_timing.py [--reps N]

Run two builds alternately in one session to compare them: the numbers move with the clocks of a shared card."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import bench
    from activesetmethods_b200.sublp import SubLp
    net = bench.network("case1354pegase")
    S = 128
    mdl, d = bench.linearise(net, list(range(1, S + 1)))
    lp = SubLp(mdl.n, mdl.m, mdl.j_str, d["xL"], d["xU"], d["gL"], d["gU"], batch=S, engine=1, eps_rel=1e-6,
               max_iter=256)
    lp.sub_optimize(d["x"], d["f"], d["df"], d["E"], d["dE"], 1000.0, False)   # data in place, graph warm
    lp.kernel_timing(reps=20)
    primal_ms, dual_ms = lp.kernel_timing(reps=args.reps)
    lp.close()
    one = SubLp(mdl.n, mdl.m, mdl.j_str, d["xL"][0], d["xU"][0], d["gL"][0], d["gU"][0], engine=2, eps_rel=1e-6,
                max_iter=8_000_000)
    for _ in range(2):   # the first solve builds the group plan
        one.sub_optimize(d["x"][0], d["f"][0], d["df"][0], d["E"][0], d["dE"][0], 1000.0, False)
    ms, iters = one.last_solve_timing()
    one.close()
    print(json.dumps({"streaming_b128_primal_ms": primal_ms, "streaming_b128_dual_ms": dual_ms,
                      "group_single_lp_ms": ms, "group_single_lp_iterations": iters,
                      "group_single_lp_us_per_iteration": 1e3 * ms / max(iters, 1)}), flush=True)


if __name__ == "__main__":
    main()
