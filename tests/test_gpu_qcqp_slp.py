"""Whole SLP runs of the rectangular-voltage OPF (acopf.AcrModel) on the device-side QCQP evaluator: against the CPU
oracle's ACR runs (the tolerances of test_gpu_slp_parity.py), and a case118 load / generator-outage queue through fewer
lanes against the one-batch run (the check test_gpu_slp_queue.py makes for ACOPF)."""
import numpy as np
import pytest

from activesetmethods_b200.examples import acopf
from helpers import problem
from oracle import slp_oracle as so
from test_gpu_slp_queue import LP, _traced

pytestmark = pytest.mark.gpu

TIGHT = dict(tol_residual=1e-7, tol_infeas=1e-7)


def _viol(pr, x):
    return so.norm_violations(pr.eval_g(x, np.zeros(pr.m)), pr.g_L, pr.g_U, x, pr.x_L, pr.x_U, np.inf)


def test_case9_trust_region_tight(gpu):
    """200 SLP iterations, as test_gpu_slp_parity.py gives the tight trust region: at 1e-7 the barrier engine's
    interior sub-LP solutions need more trust-region iterations than the oracle's vertex solutions."""
    from activesetmethods_b200.slp import Model, Parameters, SlpTR
    pr = acopf.AcrModel(acopf.case9())
    slp = SlpTR(Model.from_problem(pr, Parameters(algorithm="Trust Region", max_iter=200, device_evaluator=True,
                                                  **TIGHT))).run()
    ref = so.SlpTR(acopf.AcrModel(acopf.case9()), so.Parameters(algorithm="Trust Region", max_iter=200, **TIGHT)).run()
    rel = abs(slp.obj_val - ref.obj_val) / abs(ref.obj_val)
    print(f"ACR case9 TR: gpu ret {slp.ret} {slp.iter} it obj {slp.obj_val:.10f} | oracle ret {ref.ret} {ref.iter} it "
          f"obj {ref.obj_val:.10f} | rel {rel:.2e}")
    assert slp.ret in (0, 6)
    assert rel <= 1e-6


def test_case118_line_search_reference_tolerances(gpu):
    from activesetmethods_b200.slp import Model, Parameters, SlpLS
    pr = acopf.AcrModel(problem("case118").net)
    slp = SlpLS(Model.from_problem(pr, Parameters(max_iter=200, device_evaluator=True))).run()
    ref = so.SlpLS(acopf.AcrModel(problem("case118").net), so.Parameters(max_iter=200)).run()
    rel = abs(slp.obj_val - ref.obj_val) / abs(ref.obj_val)
    print(f"ACR case118 LS: gpu ret {slp.ret} {slp.iter} it obj {slp.obj_val:.6f} | oracle ret {ref.ret} {ref.iter} it "
          f"obj {ref.obj_val:.6f} | rel {rel:.2e}")
    assert slp.ret == ref.ret == 0
    assert _viol(pr, slp.x) <= 1e-2
    assert rel <= 1e-3


def test_device_and_host_callbacks_agree_case9(gpu):
    """The device evaluator replaces the host callbacks without changing the outcome: the same statuses and objectives
    to 1e-6 for a small load batch."""
    from activesetmethods_b200.slp import Parameters, SlpLSBatch
    net = acopf.case9()
    probs = lambda: [acopf.AcrModel(acopf.perturb_loads(net, s)) for s in range(4)]  # noqa: E731
    host = SlpLSBatch(probs(), Parameters(max_iter=100, lp_options=LP)).run()
    dev = SlpLSBatch(probs(), Parameters(max_iter=100, lp_options=LP), device_evaluator=True).run()
    print(f"ACR case9 x4 LS: host ret {host.ret} iter {host.iter} | device ret {dev.ret} iter {dev.iter}")
    assert np.array_equal(host.ret, dev.ret)
    assert np.all(np.abs(host.obj_val - dev.obj_val) <= 1e-6 * np.abs(host.obj_val))


def _problems12():
    net = problem("case118").net
    nets = [net] + [acopf.perturb_loads(net, s) for s in range(1, 9)] + acopf.generator_contingencies(net)[:3]
    return [acopf.AcrModel(n) for n in nets]


@pytest.mark.parametrize("algorithm", ["Line Search", "Trust Region"])
def test_queue_matches_one_batch(gpu, algorithm):
    """12 ACR case118 problems through 4 lanes with the QCQP evaluator give each problem the status of the one-batch run,
    and its iteration count and objective (1e-6) unless its trajectory leaves the one-batch run's through the barrier
    engine's batch-wide refinement escalation (see test_gpu_slp_queue.test_whole_runs for why that is the only
    coupling)."""
    from activesetmethods_b200.slp import Parameters, SlpLSBatch, SlpTRBatch
    cls = _traced(SlpLSBatch if algorithm == "Line Search" else SlpTRBatch)
    prm = lambda: Parameters(algorithm=algorithm, max_iter=25, lp_options=LP)  # noqa: E731
    one = cls(_problems12(), prm(), device_evaluator=True)
    one.trace = {}
    one.run()
    q = cls(_problems12(), prm(), device_evaluator=True, lanes=4)
    q.trace = {}
    q.run()
    print(f"ACR {algorithm}: one batch ret {one.ret} iter {one.iter} ({one.rounds} rounds)\n"
          f"ACR {algorithm}: 4 lanes   ret {q.ret} iter {q.iter} ({q.rounds} rounds, {len(q.loads)} loads)")
    assert q._dev == one._dev == "qcqp"
    assert q.B == 4 and len(q.loads) >= 2 and sum(len(l) for _, l in q.loads) == 8
    assert np.array_equal(q.ret, one.ret)
    for k in range(12):
        a, b = one.trace[k], q.trace[k]
        first = next((j for j in range(min(len(a), len(b))) if a[j][0] != b[j][0]), None)
        if first is None and len(a) == len(b):
            assert q.iter[k] == one.iter[k], k
            assert abs(q.obj_val[k] - one.obj_val[k]) <= 1e-6 * abs(one.obj_val[k]), k
            continue
        assert first is not None, (k, len(a), len(b))
        print(f"problem {k}: steps differ from sub-LP {first} on (escalated refinement: one batch {a[first][1]}, "
              f"4 lanes {b[first][1]})")
        assert a[first][1] or b[first][1], k
