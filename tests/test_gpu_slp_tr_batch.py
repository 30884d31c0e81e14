"""Trust-region SLP on the device: the lock-step batch ``SlpTRBatch`` against single ``SlpTR`` runs on the same
engine, against the oracle's tight-tolerance optimum, and the device-side ACOPF evaluator against the host callbacks,
for the batch and for ``SlpTR``."""
import numpy as np
import pytest

from activesetmethods_b200.examples import acopf
from oracle import slp_oracle as so

pytestmark = pytest.mark.gpu

LP = dict(eps_rel=1e-7, max_iter=3_000_000)
IDS = [1, 2, 3, 4, 5, 6]


def _params(**kw):
    from activesetmethods_b200.slp import Parameters
    return Parameters(algorithm="Trust Region", max_iter=100, lp_options=LP, **kw)


def _scenarios():
    net = acopf.case9()
    return [acopf.AcopfModel(acopf.perturb_loads(net, s)) for s in IDS]


def _violation(pr, x):
    return so.norm_violations(pr.eval_g(x, np.zeros(pr.m)), pr.g_L, pr.g_U, x, pr.x_L, pr.x_U, np.inf)


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(1.0, np.abs(np.asarray(b)))


def test_batch_of_one_equals_single_run(gpu):
    """B = 1: the same engine and the same arithmetic as SlpTR, so the same status, iteration count and radius, and
    the iterate and objective to 1e-12."""
    from activesetmethods_b200.slp import Model, SlpTR, SlpTRBatch
    one = SlpTR(Model.from_problem(acopf.AcopfModel(acopf.case9()), _params())).run()
    batch = SlpTRBatch([acopf.AcopfModel(acopf.case9())], _params()).run()
    print(f"case9 TR: single ret {one.ret} iter {one.iter} delta {one.delta:.3e} obj {one.obj_val:.10f}; "
          f"batch ret {batch.ret[0]} iter {batch.iter[0]} delta {batch.delta[0]:.3e} obj {batch.obj_val[0]:.10f}")
    assert batch.ret[0] == one.ret and batch.iter[0] == one.iter and batch.delta[0] == one.delta
    assert batch.lp_solves[0] == len(one.lp_log)
    assert np.all(_rel(batch.x[0], one.x) <= 1e-12)
    assert _rel(batch.obj_val[0], one.obj_val) <= 1e-12


def test_batched_scenarios_trust_region(gpu):
    """Six load scenarios of case9: every scenario ends with a regular status, feasible, and within the reference's
    suite tolerance of the optimum the oracle's tight-tolerance trust-region run finds for that scenario."""
    from activesetmethods_b200.slp import SlpTRBatch
    net = acopf.case9()
    probs = _scenarios()
    batch = SlpTRBatch(probs, _params()).run()
    print(f"case9 x 6 TR: ret {batch.ret} iter {batch.iter} delta {batch.delta} rounds {batch.rounds} "
          f"(two-phase {batch.two_phase_rounds}) objectives {batch.obj_val}")
    assert batch.lp_iterations > 0
    for k, s in enumerate(IDS):
        ref = so.optimize(acopf.AcopfModel(acopf.perturb_loads(net, s)),
                          so.Parameters(algorithm="Trust Region", max_iter=200, tol_residual=1e-4, tol_infeas=1e-4))
        assert batch.ret[k] in (0, 6), (s, batch.ret[k])
        assert _violation(probs[k], batch.x[k]) <= 1e-2
        assert ref.ret in (0, 6)
        assert abs(batch.obj_val[k] - ref.obj_val) <= 1e-2 * abs(ref.obj_val), (s, batch.obj_val[k], ref.obj_val)


def _check_trial(checked, opt, problems, x, p, nu, prim_infeas, fr, idx):
    """ϕ(x + p) of the device evaluator (``acopf_trial``) against the host callbacks + ``merit_phi`` at the same point
    and with the same device state (step, slacks, g(x)).  The evaluators agree to 1e-12 per term
    (test_gpu_acopf_device.py), so the bound is 1e-11 of the sum of the terms' magnitudes."""
    B = len(x)
    dev = np.atleast_1d(opt.acopf_trial(np.ones(B), nu, prim_infeas if fr else None, fr))
    base = np.array(prim_infeas, dtype=float) if fr else np.zeros(B)
    Et = np.zeros((B, problems[0].m))
    for s in idx:
        xt = x[s] + p[s]
        problems[s].eval_g(xt, Et[s])
        if not fr:
            base[s] = problems[s].eval_f(xt)
    host = np.atleast_1d(opt.merit_phi(base, Et, nu, np.ones(B), fr))
    for s in idx:
        scale = 1.0 + abs(base[s]) + float(np.sum(nu[s] * (1.0 + np.abs(Et[s]))))
        checked.append((bool(fr), float(dev[s]), float(host[s]), scale))


def _assert_trials(checked):
    assert any(c[0] for c in checked) and any(not c[0] for c in checked), "both phases must be checked"
    worst = max(abs(d - h) / sc for _, d, h, sc in checked)
    print(f"{len(checked)} trial merits checked, worst error / scale {worst:.2e}")
    assert worst <= 1e-11


def test_batched_scenarios_trust_region_device_evaluator(gpu):
    """The six-scenario batch with f, g, the Jacobian and ϕ(x + p) evaluated on the device.

    Every step-quality evaluation of the device run is checked against the host callbacks at the same point and
    device state, in both phases.  The runs end with the same statuses and iteration counts as the host-evaluator
    run (all scenarios stop at max_iter).  The objectives agree to the reference's suite tolerance (1e-2), not to
    the 1e-6 the line-search pair meets.  On case9 the trajectories part at the third sub-LP, a restoration LP with a
    face of minimisers: same iterate, the two evaluators' inputs differ by round-off, the LP objectives agree to 1e-13
    and the steps differ by 7e-4 (still 7e-5 at an LP tolerance of 1e-9).  In restoration ϕ is O(1e-6), so ρ then
    differs too (iteration 12: ρ = -0.043 with host callbacks, +0.652 on the device; the host run cuts Δ from 2 to 0.2)."""
    from activesetmethods_b200.slp import SlpTRBatch

    class Checked(SlpTRBatch):
        def _step_quality(self, fr, idx):
            _check_trial(self.checked, self.optimizer, self.problems, self.x, self.p, self.nu, self.prim_infeas, fr,
                         idx)
            super()._step_quality(fr, idx)

    host = SlpTRBatch(_scenarios(), _params()).run()
    dev = Checked(_scenarios(), _params(), device_evaluator=True)
    dev.checked = []
    dev.run()
    print(f"host ret {host.ret} iter {host.iter} delta {host.delta} obj {host.obj_val}\n"
          f"dev  ret {dev.ret} iter {dev.iter} delta {dev.delta} obj {dev.obj_val}")
    _assert_trials(dev.checked)
    assert np.array_equal(dev.ret, host.ret)
    assert np.array_equal(dev.iter, host.iter)
    assert np.all(np.abs(dev.obj_val - host.obj_val) <= 1e-2 * np.abs(host.obj_val))


def test_trust_region_on_device_evaluator(gpu):
    """SlpTR on case9 with the device-side evaluator: every ϕ(x + p) checked against the host callbacks as above; the
    same status and iteration count as the host-callback run, and the objective within the reference's suite
    tolerance of it and of the public optimum 5296.69 (the trajectories part as described for the batch)."""
    from activesetmethods_b200.slp import Model, SlpTR, SlpTRBatch
    checked = []

    class CheckedBatch(SlpTRBatch):
        def _step_quality(self, fr, idx):
            _check_trial(checked, self.optimizer, self.problems, self.x, self.p, self.nu, self.prim_infeas, fr, idx)
            super()._step_quality(fr, idx)

    class Checked(SlpTR):
        _batch = CheckedBatch

    host = SlpTR(Model.from_problem(acopf.AcopfModel(acopf.case9()), _params())).run()
    dev = Checked(Model.from_problem(acopf.AcopfModel(acopf.case9()), _params(device_evaluator=True)))
    dev.run()
    print(f"case9 TR: host ret {host.ret} iter {host.iter} obj {host.obj_val:.10f}; "
          f"device ret {dev.ret} iter {dev.iter} obj {dev.obj_val:.10f}")
    _assert_trials(checked)
    assert dev.ret == host.ret and dev.iter == host.iter
    assert abs(dev.obj_val - host.obj_val) <= 1e-2 * abs(host.obj_val)
    assert abs(dev.obj_val - 5296.69) <= 1e-2 * 5296.69
