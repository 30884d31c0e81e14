"""Continuous batching on the B200: ``asm_slp_load_lanes`` / ``asm_slp_acopf_branch_coef_lanes`` replace the scenarios
of some lanes of a handle, and the lock-step drivers refill finished lanes from a queue (``lanes``).  A handle after a
load must hold exactly what a fresh handle created with the final assignment holds: the sub-LP data of both phases,
the device evaluator's results, and a cold PDHG start for the loaded lanes.  Whole queued runs must give every problem
the status and iteration count of the one-batch run."""
import numpy as np
import pytest

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf
from test_gpu_acopf_contingency import _check_models, _handle
from test_gpu_slp_kernels import get_lp

pytestmark = pytest.mark.gpu

LP = dict(eps_rel=1e-7, max_iter=3_000_000)
LANES = [0, 7, 31, 39]


def _net118():
    return acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])


def _assignments():
    """40 case118 load scenarios, and the final assignment with lanes LANES replaced by two branch outages, a load
    scenario and a generator outage (new lanes in the order of LANES)."""
    net = _net118()
    first = [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(40)]
    out = acopf.branch_contingencies(net, 12)
    new = [acopf.AcopfModel(out[5]), acopf.AcopfModel(out[11]), acopf.AcopfModel(acopf.perturb_loads(net, 101)),
           acopf.AcopfModel(acopf.generator_contingencies(net)[2])]
    final = list(first)
    for s, md in zip(LANES, new):
        final[s] = md
    return first, new, final


def _bounds(models):
    return [np.array([getattr(m, k) for m in models]) for k in ("x_L", "x_U", "g_L", "g_U")]


def _inputs(models, seed):
    """x, f, df, E, dE of each model at a random point inside its bounds: the same host inputs for every handle."""
    rng = np.random.default_rng(seed)
    n, m = models[0].n, models[0].m
    x = np.array([rng.uniform(np.where(np.isfinite(md.x_L), md.x_L, -0.5), np.where(np.isfinite(md.x_U), md.x_U, 0.5))
                  for md in models])
    f = np.array([md.eval_f(x[s]) for s, md in enumerate(models)])
    df = np.array([md.eval_grad_f(x[s], np.zeros(n)) for s, md in enumerate(models)])
    E = np.array([md.eval_g(x[s], np.zeros(m)) for s, md in enumerate(models)])
    dE = np.array([md.eval_jac_g(x[s], "eval", None, None, np.zeros(md.nnz)) for s, md in enumerate(models)])
    delta = rng.uniform(0.1, 2.0, len(models))
    return x, f, df, E, dE, delta


def _same_lps(a, b, B):
    for s in range(B):
        la, lb = get_lp(a, s, False), get_lp(b, s, False)
        for k in la:
            assert np.array_equal(la[k], lb[k]), (s, k)


@pytest.mark.parametrize("fr_first", [False, True], ids=["restoration_after", "restoration_before"])
def test_lp_data_bit_for_bit(gpu, fr_first):
    """B = 40 (64 lanes): after loading LANES and an update with the same inputs, asm_slp_get_lp of every lane equals a
    fresh handle's in both phases; ``restoration_before`` builds the restoration solver before the load."""
    first, new, final = _assignments()
    inp = _inputs(final, 11)
    lp = _handle(first, **LP)
    if fr_first:
        lp.update(*_inputs(first, 3), True)
        lp.solve()
    lp.load_lanes(LANES, *_bounds(new))
    ref = _handle(final, **LP)
    for fr in (False, True):
        lp.update(*inp, fr)
        ref.update(*inp, fr)
        _same_lps(lp, ref, 40)
    lp.close()
    ref.close()


def test_error_codes(gpu):
    first, new, final = _assignments()
    lp = _handle(first, **LP)
    lib, h = lp._lib, lp._h
    xL, xU, gL, gU = (np.ascontiguousarray(a) for a in _bounds(new))
    d = capi.dptr
    i32 = capi.c_int32_p

    def load(lanes, gL=gL, gU=gU, xL=xL, handle=h):
        ln = np.ascontiguousarray(lanes, dtype=np.int32)
        return lib.asm_slp_load_lanes(handle, len(ln), ln.ctypes.data_as(i32), d(xL[:len(ln)]), d(xU[:len(ln)]),
                                      d(gL[:len(ln)]), d(gU[:len(ln)]))

    assert load([0, 40]) == capi.E_INVALID                      # out of range (batch 40, padded to 64)
    assert load([-1]) == capi.E_INVALID
    assert load([3, 5, 3]) == capi.E_INVALID                    # repeated
    assert load([0, 1], handle=None) == capi.E_INVALID
    ln = np.array([0], dtype=np.int32)
    assert lib.asm_slp_load_lanes(h, 1, ln.ctypes.data_as(i32), None, d(xU), d(gL), d(gU)) == capi.E_INVALID
    assert lib.asm_slp_load_lanes(h, 1, None, d(xL), d(xU), d(gL), d(gU)) == capi.E_INVALID
    assert lib.asm_slp_load_lanes(h, 0, None, None, None, None, None) == capi.OK
    eq = int(np.nonzero(first[0].g_L == first[0].g_U)[0][0])
    cls = gU.copy()
    cls[1, eq] += 1.0                                            # an equality row becomes a range row
    assert load([0, 1], gU=cls) == capi.E_INVALID
    free_L, free_U = gL.copy(), gU.copy()
    free_L[0, eq], free_U[0, eq] = -np.inf, np.inf
    assert load([2], gL=free_L, gU=free_U) == capi.E_FREE_ROW
    # a rejected load changes nothing; the handle still answers
    lp.update(*_inputs(first, 4), False)
    lp.solve()
    assert load(LANES) == capi.OK
    # back in the state before an update: solve, extract, reductions and get_lp refuse until the next update
    info = (capi.LpInfo * 40)()
    assert lib.asm_slp_solve(h, None, info) == capi.E_STATE
    assert lib.asm_slp_extract(h, None, None, None, None, None, None) == capi.E_STATE
    out = np.zeros(40)
    assert lib.asm_slp_norm_violations(h, None, None, 0, d(out)) == capi.E_STATE
    assert lib.asm_slp_row_norms(h, d(np.zeros((40, first[0].m)))) == capi.E_STATE
    lam = np.zeros((40, first[0].m))
    assert lib.asm_slp_norm_complementarity(h, None, d(lam), d(out)) == capi.E_STATE
    assert lib.asm_slp_merit_derivative(h, d(lam), 0, d(out)) == capi.E_STATE
    rows = np.zeros(1, np.int32)
    assert lib.asm_slp_get_lp(h, 0, None, rows.ctypes.data_as(i32), *[None] * 15) == capi.E_STATE
    lp.update(*_inputs(final, 5), False)
    lp.solve()
    # branch coefficients per lane: before an attach, non-finite, null
    coef = np.ascontiguousarray(np.stack([lp._acopf_arrays(m)["coef"] for m in new]))
    lnl = np.ascontiguousarray(LANES, dtype=np.int32)
    assert lib.asm_slp_acopf_branch_coef_lanes(h, 4, lnl.ctypes.data_as(i32), d(coef)) == capi.E_STATE
    lp.attach_acopf(final[0])
    bad = coef.copy()
    bad[2, 7, 3] = np.inf
    assert lib.asm_slp_acopf_branch_coef_lanes(h, 4, lnl.ctypes.data_as(i32), d(bad)) == capi.E_INVALID
    assert lib.asm_slp_acopf_branch_coef_lanes(h, 4, lnl.ctypes.data_as(i32), None) == capi.E_INVALID
    assert lib.asm_slp_acopf_branch_coef_lanes(None, 4, lnl.ctypes.data_as(i32), d(coef)) == capi.E_INVALID
    rep = np.ascontiguousarray([1, 1], dtype=np.int32)
    assert lib.asm_slp_acopf_branch_coef_lanes(h, 2, rep.ctypes.data_as(i32), d(coef)) == capi.E_INVALID
    assert lib.asm_slp_acopf_branch_coef_lanes(h, 4, lnl.ctypes.data_as(i32), d(coef)) == capi.OK
    lp.close()
    # a handle whose batch shares one set of bounds cannot take per-lane bounds
    m0 = first[0]
    from activesetmethods_b200.sublp import SubLp
    shared = SubLp(m0.n, m0.m, m0.j_str, m0.x_L, m0.x_U, m0.g_L, m0.g_U, batch=4)
    assert lib.asm_slp_load_lanes(shared._h, 1, ln.ctypes.data_as(i32), d(xL), d(xU), d(gL), d(gU)) == capi.E_STATE
    shared.close()
    # Python: a model that differs from the attached network in more than its branch coefficients
    lp = _handle(first, **LP)
    lp.attach_acopf(first[0])
    other = _net118()
    other.bs = other.bs + 0.01
    with pytest.raises(ValueError, match="differs from scenario 0"):
        lp.load_lanes([3], *_bounds([new[0]]), acopf=[acopf.AcopfModel(other)])
    lp.close()


def test_evaluator_per_lane(gpu):
    """A handle on shared coefficients gets outages in some lanes and load scenarios in others: at random points its
    evaluations are bit-identical to a fresh handle's, and every lane agrees with its host model (f, df, E, dE to 1e-12,
    the merit at a trial point to 1e-10)."""
    first, new, final = _assignments()
    lp = _handle(first, **LP)
    lp.attach_acopf(first[0])
    lp.load_lanes(LANES, *_bounds(new), acopf=new)
    ref = _handle(final, **LP)
    ref.attach_acopf(final)
    rng = np.random.default_rng(21)
    for _ in range(3):
        x = _inputs(final, int(rng.integers(1 << 30)))[0]
        lp.eval_acopf(x, 1000.0, False)
        ref.eval_acopf(x, 1000.0, False)
        for a, b in zip(lp.get_eval(), ref.get_eval()):
            assert np.array_equal(a, b)
    st = _check_models(lp, final, np.random.default_rng(22))
    print(f"case118 x 40 after the load: sub-LP statuses {np.unique(st, return_counts=True)}")
    lp.close()
    ref.close()


def _start_inputs(models):
    """The host inputs at each model's clipped start point with the line search's step bound: linearisations whose
    sub-LPs are optimal (all 40 of ``_assignments`` on a B200), so that a PDHG warm start applies to every lane."""
    n, m = models[0].n, models[0].m
    x = np.array([np.clip(md.x0, md.x_L, md.x_U) for md in models])
    f = np.array([md.eval_f(x[s]) for s, md in enumerate(models)])
    df = np.array([md.eval_grad_f(x[s], np.zeros(n)) for s, md in enumerate(models)])
    E = np.array([md.eval_g(x[s], np.zeros(m)) for s, md in enumerate(models)])
    dE = np.array([md.eval_jac_g(x[s], "eval", None, None, np.zeros(md.nnz)) for s, md in enumerate(models)])
    return x, f, df, E, dE, np.full(len(models), 1000.0)


def test_warm_start_forgotten(gpu):
    """Streaming PDHG (engine 1: no compaction, no group hand-over) with warm starts: solve, reload lane 7, update with
    the same linearisations and solve again.  The other lanes restart from their optimum (fewer iterations than cold);
    lane 7 solves its new scenario exactly like a cold solve on a fresh handle -- same status, iterations, objective."""
    first, new, final = _assignments()
    opts = dict(eps_rel=1e-6, max_iter=2_000_000, engine=1, warm_start=1)
    lp = _handle(first, **opts)
    lp.update(*_start_inputs(first), False)
    before = lp.solve()
    assert before[7]["status"] == before[8]["status"] == 0          # so both lanes would warm-start
    lp.load_lanes([7], *_bounds([new[1]]))
    mixed = list(first)
    mixed[7] = new[1]
    inp = _start_inputs(mixed)
    lp.update(*inp, False)
    warm = lp.solve()
    ref = _handle(mixed, **opts)
    ref.update(*inp, False)
    cold = ref.solve()
    print(f"lane 7: reloaded {warm[7]}, fresh {cold[7]}; lane 8: {before[8]['iterations']} iterations cold, "
          f"{warm[8]['iterations']} warm")
    assert warm[8]["iterations"] < before[8]["iterations"]          # the warm start is on for the other lanes
    assert warm[7]["status"] == cold[7]["status"] == 0
    assert warm[7]["iterations"] == cold[7]["iterations"]
    assert warm[7]["objective"] == cold[7]["objective"]
    lp.close()
    ref.close()


def _problems24():
    net = _net118()
    nets = [net] + acopf.branch_contingencies(net, 16) + [acopf.perturb_loads(net, s) for s in range(1, 7)] + \
        [acopf.generator_contingencies(net)[1]]
    assert len(nets) == 24
    return [acopf.AcopfModel(n) for n in nets]


def _traced(cls):
    """``cls`` recording, for every problem and every sub-LP solved for it, the solution it got (step and
    multipliers) and whether the barrier engine escalated its refinement passes in that batch solve (more than one
    substitution pair per factorisation: ``need_refine`` in lp_solver.cuh, raised when any lane of the batch sits at the
    acceptable level)."""
    class Traced(cls):
        def _solve_phase(self, fr, sel, delta):
            out = super()._solve_phase(fr, sel, delta)
            info = self.optimizer.ipm_info()
            escalated = info["substitution_pairs"] > 2 * info["factorisations"]
            for s in np.nonzero(sel)[0]:
                q = s if self._queue is None else self._slot[s]
                self.trace.setdefault(q, []).append((b"".join(a[s].tobytes() for a in out[:4]), escalated))
            return out
    return Traced


@pytest.mark.parametrize("algorithm", ["Line Search", "Trust Region"])
def test_whole_runs(gpu, algorithm):
    """24 case118 problems through 8 lanes with the device evaluator: every problem gets the status of the one-batch
    run of all 24, and its SLP iteration count and objective (1e-6 relative) too unless its trajectory leaves the
    one-batch run's.

    The lanes of a batch are independent but for one coupling in the barrier engine: when any lane sits at the
    acceptable level without reaching the target, the whole batch's later linear solves get more refinement passes
    (``need_refine``), which moves every lane's iterate in the last bits.  A problem shares its batch with other
    problems in the two runs, so it may see escalated refinement in one run and not in the other.  The line search
    absorbs that; a trust-region ratio of two tiny merit differences may not (on a B200 a few of the 24 problems end one
    iteration apart).  So each problem's sub-LP solutions are compared bit for bit, and the first one that differs must
    come from a batch solve with escalated refinement in at least one of the two runs; any other difference would be a
    lane coupling that continuous batching must not have."""
    from activesetmethods_b200.slp import Parameters, SlpLSBatch, SlpTRBatch
    cls = _traced(SlpLSBatch if algorithm == "Line Search" else SlpTRBatch)
    prm = lambda: Parameters(algorithm=algorithm, max_iter=25, lp_options=LP)  # noqa: E731
    one = cls(_problems24(), prm(), device_evaluator=True)
    one.trace = {}
    one.run()
    q = cls(_problems24(), prm(), device_evaluator=True, lanes=8)
    q.trace = {}
    q.run()
    print(f"{algorithm}: one batch ret {one.ret} iter {one.iter} ({one.rounds} rounds)\n"
          f"{algorithm}: 8 lanes   ret {q.ret} iter {q.iter} ({q.rounds} rounds, {len(q.loads)} loads)")
    assert q.B == 8 and len(q.loads) >= 2 and sum(len(l) for _, l in q.loads) == 16
    assert np.array_equal(q.ret, one.ret)
    for k in range(24):
        a, b = one.trace[k], q.trace[k]
        first = next((j for j in range(min(len(a), len(b))) if a[j][0] != b[j][0]), None)
        if first is None and len(a) == len(b):
            assert q.iter[k] == one.iter[k], k
            assert abs(q.obj_val[k] - one.obj_val[k]) <= 1e-6 * abs(one.obj_val[k]), k
            continue
        assert first is not None, (k, len(a), len(b))
        print(f"problem {k}: steps differ from sub-LP {first} on (escalated refinement: one batch {a[first][1]}, "
              f"8 lanes {b[first][1]}); iterations {one.iter[k]} / {q.iter[k]}, objectives {one.obj_val[k]:.10g} / "
              f"{q.obj_val[k]:.10g}")
        assert a[first][1] or b[first][1], k
