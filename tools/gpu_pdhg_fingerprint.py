"""Bitwise fingerprint of the PDHG engines (and of the barrier engine's shared preconditioning) on seeded ACOPF
sub-LPs: per scenario the status, iterations, restarts and a SHA-256 of the bytes of x, y, both bound duals and the
objective.  Two builds that compute the same doubles print the same file.

    python tools/gpu_pdhg_fingerprint.py [--out FILE]

Paths covered: engine 1 with B = 1 (the single-LP kernels), B = 32 (the batch kernels) and B = 64 (the two-lane
kernels), each followed by a warm-started second solve; engine 2 on one LP with the cluster exchange through
distributed shared memory, with ASM_NO_PUSH (through L2) and in grid mode (group_size 32); engine 5 on a
64-scenario case1354 batch (streams, compacts, hands over to the group kernel); engine 0 (barrier) at B = 64."""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def fingerprint(lp, out):
    p, lam, mu_u, mu_l = (np.atleast_2d(a) for a in out[:4])
    rows = []
    for s, info in enumerate(lp.last_info):
        h = hashlib.sha256()
        for a in (p[s], lam[s], mu_l[s], mu_u[s], np.float64(info["objective"])):
            h.update(np.ascontiguousarray(a, dtype=np.float64).tobytes())
        rows.append({"status": info["status"], "iterations": info["iterations"], "restarts": info["restarts"],
                     "sha256": h.hexdigest()})
    return rows


def run(name, case, S, solves=1, env=None, **params):
    import bench
    from activesetmethods_b200.sublp import SubLp
    mdl, d = bench.linearise(bench.network(case), list(range(1, S + 1)))
    pick = (lambda k: d[k]) if S > 1 else (lambda k: d[k][0])
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        lp = SubLp(mdl.n, mdl.m, mdl.j_str, pick("xL"), pick("xU"), pick("gL"), pick("gU"), batch=S, **params)
        res = []
        for _ in range(solves):
            out = lp.sub_optimize(pick("x"), pick("f"), pick("df"), pick("E"), pick("dE"), 1000.0, False)
            res.append({"engine_info": lp.engine_info(), "scenarios": fingerprint(lp, out)})
        lp.close()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    print(f"[fingerprint] {name}: " + "; ".join(
        f"engine_info {r['engine_info']}, iterations {[x['iterations'] for x in r['scenarios']][:4]}..." for r in res),
        flush=True)
    return {name: res}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    warm = dict(warm_start=1)
    res = {}
    res.update(run("engine1_b1_warm", "case118", 1, solves=2, engine=1, eps_rel=1e-6, **warm))
    res.update(run("engine1_b32_warm", "case118", 32, solves=2, engine=1, eps_rel=1e-6, **warm))
    res.update(run("engine1_b64_warm", "case118", 64, solves=2, engine=1, eps_rel=1e-6, **warm))
    res.update(run("engine2_cluster_push", "case118", 1, engine=2, eps_rel=1e-6))
    res.update(run("engine2_cluster_l2", "case118", 1, env={"ASM_NO_PUSH": "1"}, engine=2, eps_rel=1e-6))
    res.update(run("engine2_grid", "case118", 1, engine=2, group_size=32, eps_rel=1e-6))
    res.update(run("engine5_case1354_b64", "case1354pegase", 64, engine=5, eps_rel=5e-7, max_iter=8_000_000))
    res.update(run("engine0_case1354_b64", "case1354pegase", 64, engine=0))
    text = json.dumps(res, indent=1, sort_keys=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
