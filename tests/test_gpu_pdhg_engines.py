"""The PDHG engines against the long-double restatement of their solve (tests/pdhg_reference.py), lane by lane.

``max_iter = k * check_every`` stops every schedule exactly after k blocks, at a check, so ``asm_lp_info`` and the
returned x, y and bound duals are the state of that check.  For every case and window each lane must match its
reference lane exactly in status, iterations and restarts, and within the rounding bars in x, y, the bound duals,
pres, dres and gap (tests/test_pdhg_reference_cpu.py pins the bars and shows every decision of these cases clears
them by 100x).  Windows: 1, 2, 3 blocks, the block of the first restart and the next, the run to termination.

Schedules: the streaming kernels (engine 1: k_primal<false> at B = 1, <true> at 3 -> 32, k_primal2 / k_dual2 at
33 and 64, 100 -> 128, grid-stride loops at 1024 lanes of an LP with n, m > 592), the persistent group kernel
(engine 2: one block, cluster with and without the DSMEM push, grid; a matrix streamed from L2; check_every above
its cap of 256), the hybrid (engine 5: compaction 128 -> 64 and hand-over, read from ASM_TRACE) and the
row-partitioned kernels with world = 1.  Warm starts: after OPTIMAL (1 and 2), set_start on a fresh handle and after
an iteration limit, set_start with one side NULL after INFEASIBLE, and the row-partitioned re-solve after an
iteration limit.  SLP sub-LPs: each lane's LP as the SLP layer built it (asm_slp_get_lp), engines 1 and 5, normal and
restoration phase, and set_active.  Lane properties: a permutation of the lanes and a repeated solve give every LP
the same bytes."""
import functools

import numpy as np
import pytest

import pdhg_reference as R

pytestmark = pytest.mark.gpu
WORST = {}      # quantity -> (largest err / bar, where)
PATHS = set()   # group-kernel variants and hybrid phases the traces showed


def period(ce, cap=None):
    """The block length a schedule runs for check_every = ce (at least 2; the group kernel caps it)."""
    return min(max(2, ce), cap) if cap else max(2, ce)


def _ref(name, ce, nb, cap=None, warm=0, start=None, start_ok=None):
    pat, lp = R.case(name)
    P = dict(R.TEST_PARAMS, check_every=ce)
    if nb:
        P["max_iter"] = nb * period(ce, cap)
    return R.solve(pat, lp, P, period_cap=cap, warm=warm, start=start, start_ok=start_ok)


@functools.lru_cache(maxsize=None)
def ref(name, ce, nb, cap=None):
    return _ref(name, ce, nb, cap)


def handle(name, cls=None, **params):
    from activesetmethods_b200.sublp import B200LP
    pat, lp = R.case(name)
    B = lp["vals"].shape[1]
    cls = cls or B200LP
    kw = dict(batch=B) if cls is B200LP else {}
    h = cls(pat.n, pat.m, pat.row_ptr, pat.col_idx, **kw, eps_rel=R.TEST_PARAMS["eps_rel"], **params)
    h.set_matrix_values(lp["vals"].T.copy())
    h.set_objective(lp["c"].T.copy(), lp["c0"] if B > 1 else float(lp["c0"][0]))
    h.set_col_bounds(lp["lb"].T.copy(), lp["ub"].T.copy())
    h.set_row_bounds(lp["rl"].T.copy(), lp["ru"].T.copy())
    return h


def run(h, ce, nb, cap=None):
    """Solve stopping after nb blocks (None: to termination)."""
    h.params.check_every = ce
    h.params.max_iter = nb * period(ce, cap) if nb else R.PARAMS["max_iter"]
    info = h.optimize()
    x, y = np.atleast_2d(h.primal()), np.atleast_2d(h.row_dual())
    zl, zu = (np.atleast_2d(a) for a in h.col_dual())
    return dict(status=np.array([i["status"] for i in info]), iterations=np.array([i["iterations"] for i in info]),
                restarts=np.array([i["restarts"] for i in info]), pres=np.array([i["primal_residual"] for i in info]),
                dres=np.array([i["dual_residual"] for i in info]), gap=np.array([i["gap"] for i in info]),
                objective=np.array([i["objective"] for i in info]), x=x.T, y=y.T, zl=zl.T, zu=zu.T)


def check(got, ref_, tag, lanes=None):
    """Every lane of `got` against its reference lane (lanes[s], default s).  The reference run's decisions must
    clear their bars by 100x, so that exact equality of the discrete outcomes is a fair demand."""
    it = int(np.max(ref_["iterations"]))
    for key, v in ref_["margins"].items():
        assert v >= 100 * R.bar(R.margin_quantity(key), it), (tag, "margin", key, v)
    B = len(got["status"])
    lanes = range(B) if lanes is None else lanes
    for s, r in zip(range(B), lanes):
        for key in ("status", "iterations", "restarts"):
            assert got[key][s] == ref_[key][r], (tag, s, key, got[key][s], ref_[key][r])
        for key, v in R.compare(got, ref_, s, r, ref_["iterations"][r]).items():
            if v >= WORST.get(key, (0.0, ""))[0]:
                WORST[key] = (v, tag)
            assert v <= 1.0, (tag, s, key, v)


def windows(name, ce, cap=None):
    if not R.FULL_RUN.get(name, True):
        return [1, 2]
    return R.windows(ref(name, ce, None, cap), period(ce, cap))


def _stream_cases():
    return [(n, ce) for n in ("b1", "b3", "b33", "b64", "b100", "infeasible") for ce in R.CHECK_EVERY[n]]


@pytest.mark.parametrize("name,ce", _stream_cases())
def test_streaming(gpu, name, ce):
    h = handle(name, engine=1)
    for nb in windows(name, ce):
        check(run(h, ce, nb), ref(name, ce, nb), f"engine1 {name} ce{ce} nb{nb}")
    h.close()


def test_streaming_grid_stride(gpu):
    """1024 lanes of an LP with n, m > 592: two blocks of check_every = 4 through the capped grids."""
    h = handle("wide", engine=1)
    for nb in (1, 2):
        check(run(h, 4, nb), ref("wide", 4, nb), f"engine1 wide nb{nb}")
    h.close()


@pytest.mark.parametrize("variant", ["g1", "auto", "auto_nopush", "g32"])
@pytest.mark.parametrize("name", ["b1", "group5"])
def test_group(gpu, capfd, monkeypatch, name, variant):
    monkeypatch.setenv("ASM_TRACE", "1")
    if variant == "auto_nopush":
        monkeypatch.setenv("ASM_NO_PUSH", "1")
    gs = dict(g1=1, auto=0, auto_nopush=0, g32=32)[variant]
    h = handle(name, engine=2, group_size=gs)
    for nb in windows(name, 64):
        check(run(h, 64, nb), ref(name, 64, nb), f"engine2 {variant} {name} nb{nb}")
    err = capfd.readouterr().err
    h.close()
    want = dict(g1="G = 1 (cluster", auto="DSMEM exchange", auto_nopush="(cluster, matrix", g32="G = 32 (grid")[variant]
    assert want in err, err[-2000:]
    PATHS.update(l.split("LPs, ")[1].split(" groups")[0] for l in err.splitlines() if "group launch" in l)


def test_group_streamed_matrix(gpu, capfd, monkeypatch):
    monkeypatch.setenv("ASM_TRACE", "1")
    h = handle("big", engine=2, group_size=1)
    for nb in (1, 2):
        check(run(h, 64, nb), ref("big", 64, nb), f"engine2 big nb{nb}")
    err = capfd.readouterr().err
    h.close()
    assert "matrix streamed" in err, err[-2000:]
    PATHS.update(l.split("LPs, ")[1].split(" groups")[0] for l in err.splitlines() if "group launch" in l)


def test_group_period_capped(gpu):
    """check_every = 300 runs blocks of 256 in the group kernel."""
    h = handle("group5", engine=2)
    for nb in windows("group5", 300, R.K_MAX_STEPS):
        got = run(h, 300, nb, R.K_MAX_STEPS)
        check(got, ref("group5", 300, nb, R.K_MAX_STEPS), f"engine2 ce300 nb{nb}")
    h.close()


def test_hybrid_compacts_and_hands_over(gpu, capfd, monkeypatch):
    monkeypatch.setenv("ASM_TRACE", "1")
    h = handle("hybrid", engine=5, hand_over=0.3)
    for nb in windows("hybrid", 64):
        check(run(h, 64, nb), ref("hybrid", 64, nb), f"engine5 hybrid nb{nb}")
    err = capfd.readouterr().err
    h.close()
    assert "batch 128 -> 64" in err and "group launch" in err, err[-3000:]
    PATHS.update(["engine 5: batch 128 -> 64, then hand-over to the group kernel"])


def _dist_handle(name, **params):
    import torch  # noqa: F401  (NCCL is dlopen-ed from torch's copy)
    from activesetmethods_b200.sublp import B200RowPartitionedLP, nccl_unique_id
    uid = nccl_unique_id()
    return handle(name, cls=functools.partial(B200RowPartitionedLP, rank=0, world=1, unique_id=uid), **params)


@pytest.mark.parametrize("ce", [3, 64])
def test_row_partitioned_world_one(gpu, ce):
    h = _dist_handle("b1")
    for nb in windows("b1", ce):
        check(run(h, ce, nb), ref("b1", ce, nb), f"rows b1 ce{ce} nb{nb}")
    h.close()


# ---- warm starts ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [1, 2])
def test_warm_start_after_optimal(gpu, mode):
    h = handle("b3", engine=1)
    first = run(h, 64, None)
    check(first, ref("b3", 64, None), "cold b3")
    h.params.warm_start = mode
    got = run(h, 64, None)
    check(got, _ref("b3", 64, None, warm=mode, start=(first["x"], first["y"])), f"warm{mode} after optimal")
    h.close()


def test_set_start_on_fresh_handle(gpu):
    h = handle("b3", engine=1)
    xs, ys = R.random_start("b3")
    h.set_start(xs.T.copy(), ys.T.copy())
    h.params.warm_start = 1
    check(run(h, 64, 2), _ref("b3", 64, 2, warm=1, start=(xs, ys)), "set_start fresh")
    h.close()


def test_set_start_after_iteration_limit(gpu):
    """The caller's start is used whatever ended the previous solve; without set_start an unconverged point is not."""
    h = handle("b3", engine=1)
    got = run(h, 64, 1)
    assert (got["status"] == R.ITERATION_LIMIT).all()
    h.params.warm_start = 1
    check(run(h, 64, 2), ref("b3", 64, 2), "warm after iteration limit starts cold")
    xs, ys = R.random_start("b3")
    h.set_start(xs.T.copy(), ys.T.copy())
    check(run(h, 64, 2), _ref("b3", 64, 2, warm=1, start=(xs, ys)), "set_start after iteration limit")
    h.close()


def test_row_partitioned_warm_start_rule(gpu):
    """Row-partitioned handle: the OPTIMAL-only rule of the single-GPU handle, and set_start is honoured."""
    h = _dist_handle("b1")
    assert run(h, 64, 1)["status"][0] == R.ITERATION_LIMIT
    h.params.warm_start = 1
    check(run(h, 64, 2), ref("b1", 64, 2), "rows warm after iteration limit starts cold")
    xs, ys = R.random_start("b1")
    h.set_start(xs[:, 0].copy(), ys[:, 0].copy())
    check(run(h, 64, 2), _ref("b1", 64, 2, warm=1, start=(xs, ys)), "rows set_start")
    h.close()


def test_set_start_one_side_after_infeasible(gpu):
    """set_start(x, NULL) after INFEASIBLE: y starts cold, not from the stored Farkas direction."""
    h = handle("infeasible", engine=1)
    assert (run(h, 64, None)["status"] == R.INFEASIBLE).all()
    xs, ys = R.random_start("infeasible")
    h.set_start(xs.T.copy(), None)
    h.params.warm_start = 1
    check(run(h, 64, 2), _ref("infeasible", 64, 2, warm=1, start=(xs, np.zeros_like(ys))), "set_start x only")
    h.close()


# ---- SLP sub-LPs -------------------------------------------------------------------------------------------------
def _slp_lp(sub, s):
    """Lane s's LP data and raw solution from asm_slp_get_lp."""
    from activesetmethods_b200 import capi
    lib, h = sub._lib, sub._h
    i32, i64, d = capi.c_int32_p, capi.c_int64_p, capi.dptr
    cols, rows, st, nnz = np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int64)
    capi.check(lib.asm_slp_get_lp(h, s, cols.ctypes.data_as(i32), rows.ctypes.data_as(i32), nnz.ctypes.data_as(i64),
                                  *[None] * 14))
    nc, nr, nz = int(cols[0]), int(rows[0]), int(nnz[0])
    o = dict(row_ptr=np.zeros(nr + 1, np.int64), col_idx=np.zeros(nz, np.int32), vals=np.zeros(nz), c=np.zeros(nc),
             c0=np.zeros(1), lb=np.zeros(nc), ub=np.zeros(nc), rl=np.zeros(nr), ru=np.zeros(nr), x=np.zeros(nc),
             y=np.zeros(nr), zl=np.zeros(nc), zu=np.zeros(nc))
    capi.check(lib.asm_slp_get_lp(h, s, None, None, None, o["row_ptr"].ctypes.data_as(i64),
                                  o["col_idx"].ctypes.data_as(i32), *(d(o[k]) for k in ("vals", "c", "c0", "lb", "ub",
                                                                                       "rl", "ru", "x", "y", "zl", "zu")),
                                  st.ctypes.data_as(i32)))
    o["status"] = int(st[0])
    return o


def _slp_handle(name, B, engine, feasibility, seed=0, **params):
    """A batch of B linearisations of `name` around perturbed points, updated for the given phase."""
    from helpers import problem
    from activesetmethods_b200.sublp import SubLp
    mdl = problem(name)
    rng = np.random.default_rng(seed)
    lo = np.where(np.isfinite(mdl.x_L), mdl.x_L, -10.0)
    hi = np.where(np.isfinite(mdl.x_U), mdl.x_U, 10.0)
    xs = np.clip(mdl.x0 + 0.05 * rng.standard_normal((B, mdl.n)) * (1.0 + np.abs(mdl.x0)), lo, hi)
    f = np.array([mdl.eval_f(x) for x in xs])
    df = np.stack([mdl.eval_grad_f(x, np.zeros(mdl.n)) for x in xs])
    E = np.stack([mdl.eval_g(x, np.zeros(mdl.m)) for x in xs])
    dE = np.stack([mdl.eval_jac_g(x, "eval", None, None, np.zeros(len(mdl.j_str))) for x in xs])
    sub = SubLp(mdl.n, mdl.m, mdl.j_str, mdl.x_L, mdl.x_U, mdl.g_L, mdl.g_U, batch=B, engine=engine,
                eps_rel=R.TEST_PARAMS["eps_rel"], check_every=64, max_iter=3 * 64, **params)
    sub.update(xs, f, df, E, dE, 10.0, feasibility)
    return sub


def _slp_ref(o):
    pat = R.Pattern(len(o["c"]), len(o["rl"]), o["row_ptr"], o["col_idx"])
    lp = {k: o[k][:, None] for k in ("vals", "c", "lb", "ub", "rl", "ru")}
    lp["c0"] = o["c0"]
    return R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=64, max_iter=3 * 64))


def _as_run(info, o):
    return dict(status=np.array([info["status"]]), iterations=np.array([info["iterations"]]),
                restarts=np.array([info["restarts"]]), pres=np.array([info["primal_residual"]]),
                dres=np.array([info["dual_residual"]]), gap=np.array([info["gap"]]),
                **{k: o[k][:, None] for k in ("x", "y", "zl", "zu")})


# hs071's restoration LP is left out: its y drifts about 2x the bars calibrated on the generator's LPs (the
# restoration phase is covered by case9)
@pytest.mark.parametrize("name,feasibility", [("hs071", False), ("case9", False), ("case9", True)])
@pytest.mark.parametrize("engine", [1, 5])
def test_slp_sub_lps(gpu, name, engine, feasibility):
    """Each lane's sub-LP, as the SLP layer built it on the device, solved for three blocks: the raw solution of
    asm_slp_get_lp against the reference run on that lane's LP data."""
    sub = _slp_handle(name, 3, engine, feasibility)
    info = sub.solve()
    for s in range(3):
        o = _slp_lp(sub, s)
        assert (o["status"] if o["status"] >= 0 else R.ITERATION_LIMIT) == info[s]["status"]   # -1: still running
        check(_as_run(info[s], o), _slp_ref(o), f"slp {name} engine{engine} fr{int(feasibility)} lane{s}")
    sub.close()


@pytest.mark.parametrize("engine", [1, 5])
def test_slp_set_active(gpu, engine):
    """Masked lanes report SKIPPED; active lanes are bit-identical to the unmasked run.  Same kernels in both runs:
    engine 5 would hand 2 running LPs of 4 to the group kernel at its default hand_over (0.5), so it is lowered; over
    the 3-block window no LP finishes, and the batch keeps streaming in both runs."""
    kw = dict(hand_over=0.1) if engine == 5 else {}
    full = _slp_handle("case9", 4, engine, False, **kw)
    info_full = full.solve()
    want = {s: _slp_lp(full, s) for s in range(4)}
    full.close()
    part = _slp_handle("case9", 4, engine, False, **kw)
    mask = np.array([True, False, True, False])
    part.set_active(mask)
    info = part.solve()
    for s in range(4):
        if not mask[s]:
            assert info[s]["status"] == 5, info[s]
            continue
        assert info[s] == info_full[s]
        got = _slp_lp(part, s)
        for k in ("x", "y", "zl", "zu"):
            assert got[k].tobytes() == want[s][k].tobytes(), (s, k)
    part.close()


# ---- lane properties ---------------------------------------------------------------------------------------------
def _bytes(got, s):
    return b"".join(np.ascontiguousarray(got[k][:, s]).tobytes() for k in ("x", "y", "zl", "zu")) + \
        b"".join(np.float64(got[k][s]).tobytes() for k in ("objective", "pres", "dres", "gap"))


def test_permuted_lanes_and_repeated_solve_are_bit_identical(gpu):
    from activesetmethods_b200.sublp import B200LP
    pat, lp = R.case("b33")
    h0 = handle("b33", engine=1)
    a = run(h0, 64, None)
    h0.close()
    h = handle("b33", engine=1)
    b = run(h, 64, None)
    for s in range(33):
        assert _bytes(a, s) == _bytes(b, s), s
    perm = np.random.default_rng(0).permutation(33)
    plp = R.lanes(lp, perm)
    p = B200LP(pat.n, pat.m, pat.row_ptr, pat.col_idx, batch=33, eps_rel=R.TEST_PARAMS["eps_rel"], engine=1)
    p.set_matrix_values(plp["vals"].T.copy())
    p.set_objective(plp["c"].T.copy(), plp["c0"])
    p.set_col_bounds(plp["lb"].T.copy(), plp["ub"].T.copy())
    p.set_row_bounds(plp["rl"].T.copy(), plp["ru"].T.copy())
    c = run(p, 64, None)
    for t, s in enumerate(perm):
        assert c["iterations"][t] == a["iterations"][s]
        assert _bytes(c, t) == _bytes(a, s), (t, s)
    h.close()
    p.close()


def test_zz_report(gpu):
    """With -s: the worst err / bar of every quantity over this file's comparisons, and the paths the trace showed."""
    print("\n[pdhg-engines] worst err/bar:")
    for key, (v, tag) in sorted(WORST.items()):
        print(f"  {key:5s} {v:.3e}   ({tag})")
    print("[pdhg-engines] paths seen:", sorted(PATHS))
    for name in R.CASES:
        if not R.FULL_RUN.get(name, True):
            continue
        for ce in R.CHECK_EVERY[name]:
            cap = R.K_MAX_STEPS if ce > R.K_MAX_STEPS else None
            full = ref(name, ce, None, cap)
            it = int(full["iterations"].max())
            low = min(full["margins"].items(), key=lambda kv: kv[1] / R.bar(R.margin_quantity(kv[0]), it))
            print(f"[pdhg-engines] margins {name} ce{ce}: smallest margin/bar {low[0]} "
                  f"{low[1] / R.bar(R.margin_quantity(low[0]), it):.3g}")
