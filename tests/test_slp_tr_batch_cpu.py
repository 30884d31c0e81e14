"""SlpTRBatch (lock-step trust-region SLP over scenarios, activesetmethods_b200/slp.py) on the CPU: with the oracle's
LP solver behind a batch engine that has the ``SubLp(batch=B)`` interface, every scenario must walk exactly the
trajectory of its own ``SlpTR`` run — same sub-LPs in the same phases, status, iteration count, trust-region radius
and iterate — and must be solved only while it runs, and only in its own phase."""
import numpy as np
import pytest

from activesetmethods_b200.examples import acopf, small_nlps
from activesetmethods_b200.slp import Model, Parameters, SlpTR, SlpTRBatch
from cpu_engine import OracleBatchEngine, OracleEngine

LP_SKIPPED = 5      # include/asm_b200.h: status of a scenario masked out of a solve


class OracleMaskedBatchEngine(OracleBatchEngine):
    """``OracleBatchEngine`` with the rest of the ``SubLp(batch=B)`` interface a trust-region round uses: a radius
    per scenario, ``row_norms`` and ``set_active`` (masked scenarios are not solved and come back as
    ``LP_SKIPPED`` with zeroed outputs).  ``solves[s]`` lists (status, restoration flag) of every sub-LP solved
    for scenario ``s``."""

    def __init__(self, n, m, j_str, x_L, x_U, g_L, g_U, batch=1, **kw):
        super().__init__(n, m, j_str, x_L, x_U, g_L, g_U, batch=batch, **kw)
        self.n, self.m = n, m
        self.active = np.ones(batch, dtype=bool)
        self.solves = [[] for _ in range(batch)]

    def update(self, x_k, f, df, E, dE, delta, feasibility=False):
        delta = np.broadcast_to(np.asarray(delta, dtype=float), (self.B,))
        for s, e in enumerate(self.eng):
            e.update(x_k[s], f[s], df[s], E[s], dE[s], delta[s], feasibility)

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
            self.solves[s].append((int(status[s]), e._d["fr"]))
        return p, lam, mu_u, mu_l, slack, status

    def row_norms(self):
        return np.array([e.row_norms() for e in self.eng])


def _case9_scenarios():
    net = acopf.case9()
    return [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(4)], 100


def _toy_starts():
    toys = [small_nlps.ToyNlp() for _ in range(3)]
    toys[1].x0 = np.array([0.5, -0.5])
    toys[2].x0 = np.array([-2.0, -0.4])
    return toys, 60


def _single(problem, max_iter):
    mdl = Model.from_problem(problem, Parameters(algorithm="Trust Region", max_iter=max_iter,
                                                 external_optimizer=OracleEngine))
    return SlpTR(mdl).run()


@pytest.mark.parametrize("make", [_case9_scenarios, _toy_starts], ids=["case9_loads", "toy_starts"])
def test_batched_trust_region_equals_single_runs(make):
    """Every scenario ends exactly where its own SlpTR run ends: status, iteration count, final radius, iterate
    (1e-9) and objective (1e-9 relative), and the batch solved the same sub-LPs for it, in the same phases."""
    probs, max_iter = make()
    batch = SlpTRBatch(probs, Parameters(algorithm="Trust Region", max_iter=max_iter,
                                         external_optimizer=OracleMaskedBatchEngine)).run()
    eng = batch.optimizer
    restored = 0
    for s in range(batch.B):
        again, _ = make()
        one = _single(again[s], max_iter)
        assert batch.ret[s] == one.ret and batch.iter[s] == one.iter, (s, batch.ret[s], one.ret, batch.iter[s], one.iter)
        assert batch.delta[s] == one.delta, (s, batch.delta[s], one.delta)
        assert np.allclose(batch.x[s], one.x, rtol=0, atol=1e-9)
        assert abs(batch.obj_val[s] - one.obj_val) <= 1e-9 * max(1.0, abs(one.obj_val))
        # masking: one solve per entry of the single run's LP log, each in the phase the single run was in
        assert eng.solves[s] == [(int(e[0]), bool(e[2])) for e in one.lp_log], s
        assert batch.lp_solves[s] == len(one.lp_log)
        restored += any(e[2] for e in one.lp_log)
    assert restored >= 1
    # a running scenario is solved once per round, in one phase
    assert not batch.running.any() and batch.rounds == int(np.max(batch.lp_solves))


def test_device_evaluator_needs_b200_engine():
    probs, _ = _case9_scenarios()
    batch = SlpTRBatch(probs, Parameters(algorithm="Trust Region", external_optimizer=OracleMaskedBatchEngine),
                       device_evaluator=True)
    with pytest.raises(ValueError):
        batch.run()


def test_scenarios_must_share_the_jacobian_pattern():
    probs, _ = _case9_scenarios()
    other = acopf.AcopfModel(acopf.case9())
    other.j_str = np.array(other.j_str)[::-1].copy()
    with pytest.raises(ValueError):
        SlpTRBatch(probs[:2] + [other], Parameters(algorithm="Trust Region", external_optimizer=OracleMaskedBatchEngine))
