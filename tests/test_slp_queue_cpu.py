"""Continuous batching in the lock-step SLP drivers (``lanes`` of ``SlpLSBatch`` / ``SlpTRBatch``,
activesetmethods_b200/slp.py) on the CPU.  A list of problems longer than the batch runs through a few lanes that
are refilled from the queue as runs end.  With the oracle's LP solver behind a batch engine that can replace the
scenario of a lane, every problem must walk exactly the trajectory of its own one-scenario run: this is the check of
the lane reset."""
import ctypes as C

import numpy as np
import pytest

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf
from activesetmethods_b200.slp import Model, Parameters, SlpLS, SlpLSBatch, SlpTR, SlpTRBatch
from cpu_engine import OracleBatchEngine, OracleEngine

LP_SKIPPED = 5      # include/asm_b200.h: status of a scenario masked out of a solve


class OracleQueueEngine(OracleBatchEngine):
    """``OracleBatchEngine`` with what a queued trust-region run needs besides: ``load_lanes`` (a fresh
    ``OracleEngine`` per loaded lane), a radius per scenario in ``update``, ``row_norms``, and ``set_active`` (masked
    scenarios are not solved and come back as ``LP_SKIPPED``, as on the device: a solve of a scenario in the other
    phase would replace the step and slacks its merit calls read).  ``loads`` lists the lanes of every ``load_lanes``
    call."""

    def __init__(self, n, m, j_str, x_L, x_U, g_L, g_U, batch=1, **kw):
        super().__init__(n, m, j_str, x_L, x_U, g_L, g_U, batch=batch, **kw)
        self.n, self.m, self.j_str = n, m, j_str
        self.active = np.ones(batch, dtype=bool)
        self.loads = []

    def set_active(self, mask=None):
        self.active = np.ones(self.B, dtype=bool) if mask is None else np.array(mask, dtype=bool)

    def solve_extract(self):
        B, n, m = self.B, self.n, self.m
        p, lam, mu_u, mu_l = np.zeros((B, n)), np.zeros((B, m)), np.zeros((B, n)), np.zeros((B, n))
        slack, status = np.zeros((B, m, 2)), np.full(B, LP_SKIPPED)
        self.last_info = []
        for s, e in enumerate(self.eng):
            if not self.active[s]:
                self.last_info.append(dict(status=LP_SKIPPED, objective=0.0, iterations=0))
                continue
            p[s], lam[s], mu_u[s], mu_l[s], slack[s], status[s] = e.solve_extract()
            self.last_info.append(e.last_info[0])
        return p, lam, mu_u, mu_l, slack, status

    def load_lanes(self, lanes, x_L, x_U, g_L, g_U):
        self.loads.append([int(s) for s in lanes])
        for j, s in enumerate(lanes):
            self.eng[s] = OracleEngine(self.n, self.m, self.j_str, x_L[j], x_U[j], g_L[j], g_U[j])

    def update(self, x_k, f, df, E, dE, delta, feasibility=False):
        delta = np.broadcast_to(np.asarray(delta, dtype=float), (self.B,))
        for s, e in enumerate(self.eng):
            e.update(x_k[s], f[s], df[s], E[s], dE[s], delta[s], feasibility)

    def row_norms(self):
        return np.array([e.row_norms() for e in self.eng])


def _case9_problems():
    """11 case9 problems: the base case, its 6 non-islanding branch outages, 3 load scenarios, generator outage 1."""
    net = acopf.case9()
    nets = [net] + acopf.branch_contingencies(net) + [acopf.perturb_loads(net, s) for s in (1, 2, 3)] + \
        [acopf.generator_contingencies(net)[1]]
    assert len(nets) == 11
    return [acopf.AcopfModel(n) for n in nets]


ALGOS = {
    "line_search": (SlpLSBatch, SlpLS, "Line Search"),
    "trust_region": (SlpTRBatch, SlpTR, "Trust Region"),
}
MAX_ITER = 60


def _params(algorithm, engine):
    return Parameters(algorithm=algorithm, max_iter=MAX_ITER, external_optimizer=engine)


@pytest.fixture(scope="module")
def problems():
    return _case9_problems()


@pytest.fixture(scope="module")
def singles(problems):
    out = {}
    for key, (_, single, algorithm) in ALGOS.items():
        out[key] = [single(Model.from_problem(pr, _params(algorithm, OracleEngine))).run() for pr in problems]
    return out


@pytest.mark.parametrize("key", list(ALGOS))
def test_queue_equals_single_runs(key, problems, singles):
    """11 problems through 3 lanes: every problem ends exactly where its own one-scenario run ends (status, iteration
    count, sub-LP statuses and phases, iterate to 1e-9, objective to 1e-9 relative), each problem is loaded once, and
    there is at most one load per round."""
    batch_cls, _, algorithm = ALGOS[key]
    b = batch_cls(problems, _params(algorithm, OracleQueueEngine), lanes=3)
    b.run()
    N = len(problems)
    assert b.B == 3 and len(b.ret) == N and len(b.lp_log) == N and b.x.shape == (N, problems[0].n)
    for q, ref in enumerate(singles[key]):
        assert b.ret[q] == ref.ret, q
        assert b.iter[q] == ref.iter, q
        assert [(st, fr) for st, _, fr, _ in b.lp_log[q]] == [(st, fr) for st, _, fr, _ in ref.lp_log], q
        assert b.lp_solves[q] == len(ref.lp_log), q
        np.testing.assert_allclose(b.x[q], ref.x, rtol=0, atol=1e-9)
        assert b.obj_val[q] == pytest.approx(ref.obj_val, rel=1e-9, abs=0)
        if key == "trust_region":
            assert b.delta[q] == pytest.approx(ref.delta, rel=1e-12, abs=0)
    # the queue was exercised: lanes freed at many different rounds, and restoration ran
    rounds = [r for r, _ in b.loads]
    assert len(rounds) == len(set(rounds)), "more than one load in a round"
    loaded = sorted(s for _, lanes in b.loads for s in lanes)
    assert sum(len(lanes) for lanes in b.optimizer.loads) == N - 3
    assert [list(lanes) for _, lanes in b.loads] == b.optimizer.loads
    assert len(loaded) == N - 3 and len(set(rounds)) >= 4
    if key == "trust_region":   # restoration LPs in lanes that were loaded from the queue
        assert b.two_phase_rounds > 0
        assert any(fr for q in range(3, N) for _, _, fr, _ in b.lp_log[q])
    assert len(set(b.iter.tolist())) > 3


def test_queue_statuses_cover_restoration(problems, singles):
    """The measured spread of the problem set, which makes the queue test above meaningful: line search ends in
    {0, -1} after 23 to 60 iterations; trust region ends in {0, 6, -1} with two-phase rounds."""
    ls = singles["line_search"]
    assert {r.ret for r in ls} == {0, -1}
    assert min(r.iter for r in ls) >= 20 and max(r.iter for r in ls) == MAX_ITER
    assert {r.ret for r in singles["trust_region"]} == {0, 6, -1}


@pytest.mark.parametrize("key", list(ALGOS))
@pytest.mark.parametrize("lanes", [None, 11, 40])
def test_default_path_unchanged(key, lanes, problems):
    """``lanes=None`` and ``lanes >= N`` run the one-batch path: results bit-identical to the driver without it."""
    batch_cls, _, algorithm = ALGOS[key]
    probs = problems[:5]
    ref = batch_cls(probs, _params(algorithm, OracleQueueEngine)).run()
    b = batch_cls(probs, _params(algorithm, OracleQueueEngine), lanes=lanes).run()
    assert b.B == len(probs) and b.optimizer.loads == []
    assert b.rounds == ref.rounds and b.two_phase_rounds == ref.two_phase_rounds
    for name in ("ret", "iter", "x", "obj_val", "prim_infeas", "dual_infeas", "compl", "lp_solves", "p", "lam", "nu"):
        np.testing.assert_array_equal(getattr(b, name), getattr(ref, name), err_msg=name)
    assert b.lp_log == ref.lp_log


def test_lanes_argument_errors(problems):
    for batch_cls in (SlpLSBatch, SlpTRBatch):
        with pytest.raises(ValueError):
            batch_cls(problems, _params("Line Search", OracleQueueEngine), lanes=0)
        with pytest.raises(ValueError):       # an optimizer that cannot replace a lane's scenario
            batch_cls(problems, _params("Line Search", OracleBatchEngine), lanes=3)
        batch_cls(problems, _params("Line Search", OracleBatchEngine), lanes=len(problems))   # no queue: accepted


def test_load_lanes_null_handle():
    """Both entry points reject a null handle with ASM_E_INVALID (no device needed)."""
    lib = capi.load()
    lanes = (C.c_int32 * 1)(0)
    d = (C.c_double * 4)()
    assert lib.asm_slp_load_lanes(None, 1, lanes, d, d, d, d) == capi.E_INVALID
    assert lib.asm_slp_acopf_branch_coef_lanes(None, 1, lanes, d) == capi.E_INVALID
