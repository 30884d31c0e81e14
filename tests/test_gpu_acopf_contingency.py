"""Contingency batches on the device-side ACOPF evaluator: per-scenario branch coefficients
(``asm_slp_acopf_branch_coef``) against each scenario's host model, the shared path unchanged bit for bit, the error
codes of the new call, and whole line-search and trust-region batches of case9 outages against the host callbacks."""
import copy

import numpy as np
import pytest

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf
from test_gpu_slp_tr_batch import _check_trial

pytestmark = pytest.mark.gpu

LP = dict(eps_rel=1e-7, max_iter=3_000_000)


def _close(a, b, name, tol=1e-12):
    a, b = np.asarray(a), np.asarray(b)
    err = np.max(np.abs(a - b) / (1.0 + np.abs(b)), initial=0.0)
    assert err <= tol, (name, err)


def _mixed(net, count):
    """Base case, ``count`` branch outages, a tap change, an impedance change, a load scenario and a generator outage."""
    tap = copy.copy(net)
    tap.tap = net.tap.copy()
    tap.tap[3] = 1.05
    imp = copy.copy(net)
    imp.br_x = net.br_x.copy()
    imp.br_x[5] *= 1.3
    return [net] + acopf.branch_contingencies(net, count) + [tap, imp, acopf.perturb_loads(net, 1),
                                                             acopf.generator_contingencies(net)[1]]


def _handle(models, **kw):
    from activesetmethods_b200.sublp import SubLp
    m0 = models[0]
    arr = lambda k: np.array([getattr(m, k) for m in models])  # noqa: E731
    lp = SubLp(m0.n, m0.m, m0.j_str, arr("x_L"), arr("x_U"), arr("g_L"), arr("g_U"), batch=len(models), **kw)
    lp._squeeze = False
    return lp


def _check_models(lp, models, rng):
    """f, grad f, g and the Jacobian values at random points (1e-12), then phi(x + alpha p) after one sub-LP (1e-10)."""
    B, n, m = len(models), models[0].n, models[0].m
    lo = np.array([np.where(np.isfinite(md.x_L), md.x_L, -0.5) for md in models])
    hi = np.array([np.where(np.isfinite(md.x_U), md.x_U, 0.5) for md in models])
    x = rng.uniform(lo, hi)
    lp.eval_acopf(x, 1000.0, False)
    f, df, E, dE = lp.get_eval()
    for s, md in enumerate(models):
        _close(f[s], md.eval_f(x[s]), ("f", s))
        _close(df[s], md.eval_grad_f(x[s], np.zeros(n)), ("df", s))
        _close(E[s], md.eval_g(x[s], np.zeros(m)), ("E", s))
        _close(dE[s], md.eval_jac_g(x[s], "eval", None, None, np.zeros(md.nnz)), ("dE", s))
    x0 = np.array([np.clip(md.x0, md.x_L, md.x_U) for md in models])
    lp.eval_acopf(x0, 1000.0, False)
    p, lam, _, _, _, st = lp.solve_extract()
    p, nu = np.atleast_2d(p), np.abs(np.atleast_2d(lam))
    alpha = rng.uniform(0.05, 1.0, B)
    phi = np.atleast_1d(lp.acopf_trial(alpha, nu))
    for s, md in enumerate(models):
        xt = x0[s] + alpha[s] * p[s]
        Et = md.eval_g(xt, np.zeros(m))
        ref = md.eval_f(xt) + float(np.sum(nu[s] * np.maximum(0.0, np.maximum(Et - md.g_U, md.g_L - Et))))
        assert abs(phi[s] - ref) <= 1e-10 * max(1.0, abs(ref)), (s, phi[s], ref)
    return st


def test_per_scenario_coefficients_case118(gpu):
    """A mixed case118 batch of B = 33 (padded to 64 lanes)."""
    net = acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])
    models = [acopf.AcopfModel(n) for n in _mixed(net, 28)]
    assert len(models) == 33
    lp = _handle(models, eps_rel=1e-7)
    lp.attach_acopf(models)
    st = _check_models(lp, models, np.random.default_rng(5))
    print(f"case118 x 33 mixed: sub-LP statuses {np.unique(st, return_counts=True)}")
    lp.close()


def test_per_scenario_coefficients_single(gpu):
    """B = 1: the handle attached with the base network, then the coefficients of a branch outage through the new call
    (the one-lane layout); the evaluator must follow the outage model."""
    net = acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])
    base = acopf.AcopfModel(net)
    out = acopf.AcopfModel(acopf.branch_contingencies(net, 4)[3])
    lp = _handle([out])
    lp.attach_acopf(base)
    coef = lp._acopf_arrays(out)["coef"]
    assert not np.array_equal(coef, lp._acopf_arrays(base)["coef"])
    capi.check(lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(np.ascontiguousarray(coef))))
    _check_models(lp, [out], np.random.default_rng(6))
    lp.close()


def test_per_scenario_coefficients_case1354_capped_grid(gpu):
    """case1354 with 320 scenarios: the evaluator's grid is capped (236 blocks for 1991 branches and 2708 balance rows
    at 10 lane groups), so every thread walks several branches with its own scenario's coefficients."""
    net = acopf.synthetic_network(*acopf.PEGASE_SHAPES["case1354pegase"])
    models = [acopf.AcopfModel(n) for n in _mixed(net, 315)]
    assert len(models) == 320
    lp = _handle(models, eps_rel=1e-6)
    lp.attach_acopf(models)
    st = _check_models(lp, models, np.random.default_rng(8))
    print(f"case1354 x 320 mixed: sub-LP statuses {np.unique(st, return_counts=True)}")
    lp.close()


def test_shared_path_unchanged(gpu):
    """Per-scenario coefficients that all equal the shared ones give bit-identical evaluations and trial merits."""
    net = acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])
    models = [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(40)]
    lp = _handle(models, eps_rel=1e-7)
    lp.attach_acopf(models[0])
    rng = np.random.default_rng(7)
    x = np.array([rng.uniform(np.where(np.isfinite(md.x_L), md.x_L, -0.5), np.where(np.isfinite(md.x_U), md.x_U, 0.5))
                  for md in models])
    x0 = np.array([np.clip(md.x0, md.x_L, md.x_U) for md in models])
    lp.eval_acopf(x, 1000.0, False)
    shared = lp.get_eval()
    lp.eval_acopf(x0, 1000.0, False)
    lp.solve_extract()
    alpha = rng.uniform(0.05, 1.0, len(models))
    nu = rng.uniform(0.0, 10.0, (len(models), models[0].m))
    phi_shared = lp.acopf_trial(alpha, nu)
    coef = np.ascontiguousarray(np.stack([lp._acopf_arrays(models[0])["coef"]] * len(models)))
    capi.check(lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(coef)))
    phi_scen = lp.acopf_trial(alpha, nu)          # same x_k and step: only the coefficients' layout differs
    assert np.array_equal(phi_scen, phi_shared)
    lp.eval_acopf(x, 1000.0, False)
    for a, b in zip(lp.get_eval(), shared):
        assert np.array_equal(a, b)
    lp.close()


def test_error_codes(gpu):
    net = acopf.case9()
    models = [acopf.AcopfModel(n) for n in acopf.branch_contingencies(net)[:2]]
    lp = _handle(models)
    coef = np.ascontiguousarray(np.stack([lp._acopf_arrays(m)["coef"] for m in models]))
    assert lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(coef)) == capi.E_STATE
    lp.attach_acopf(models[0])
    assert lp._lib.asm_slp_acopf_branch_coef(lp._h, None) == capi.E_INVALID
    assert lp._lib.asm_slp_acopf_branch_coef(None, capi.dptr(coef)) == capi.E_INVALID
    bad = coef.copy()
    bad[1, 4, 2] = np.nan
    assert lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(bad)) == capi.E_INVALID
    assert lp._lib.asm_slp_acopf_branch_coef(lp._h, capi.dptr(coef)) == capi.OK
    # the Python layer: one model or one per scenario, and the shared arrays must agree
    with pytest.raises(ValueError, match="3 models for a batch of 2"):
        lp.attach_acopf(models + models[:1])
    other = copy.copy(net)
    other.bs = net.bs + 0.01
    with pytest.raises(ValueError, match="differs from scenario 0"):
        lp.attach_acopf([models[0], acopf.AcopfModel(other)])
    lp.close()


def _case9_batch():
    net = acopf.case9()
    return [acopf.AcopfModel(n) for n in [net] + acopf.branch_contingencies(net) + acopf.generator_contingencies(net)[:1]]


def test_line_search_contingency_batch(gpu):
    """SlpLSBatch on the base case, the 6 branch outages and a generator outage of case9: the device evaluator gives
    the same statuses and iteration counts as the host callbacks, objectives to 1e-6."""
    from activesetmethods_b200.slp import Parameters, SlpLSBatch
    host = SlpLSBatch(_case9_batch(), Parameters(max_iter=100, lp_options=LP)).run()
    dev = SlpLSBatch(_case9_batch(), Parameters(max_iter=100, lp_options=LP), device_evaluator=True).run()
    print(f"host ret {host.ret} iter {host.iter} obj {host.obj_val}\ndev  ret {dev.ret} iter {dev.iter} obj {dev.obj_val}")
    assert np.array_equal(dev.ret, host.ret) and np.all(np.isin(dev.ret, (0, 6)))
    assert np.array_equal(dev.iter, host.iter)
    assert np.all(np.abs(dev.obj_val - host.obj_val) <= 1e-6 * np.abs(host.obj_val))


def test_trust_region_contingency_batch(gpu):
    """SlpTRBatch with the device evaluator on the same batch: at every step_quality each scenario's device
    phi(x + p) equals the host callbacks' value at the same point and device state (1e-11 of the terms' scale)."""
    from activesetmethods_b200.slp import Parameters, SlpTRBatch

    class Checked(SlpTRBatch):
        def _step_quality(self, fr, idx):
            _check_trial(self.checked, self.optimizer, self.problems, self.x, self.p, self.nu, self.prim_infeas, fr,
                         idx)
            super()._step_quality(fr, idx)

    dev = Checked(_case9_batch(), Parameters(algorithm="Trust Region", max_iter=100, lp_options=LP),
                  device_evaluator=True)
    dev.checked = []
    dev.run()
    worst = max(abs(d - h) / sc for _, d, h, sc in dev.checked)
    print(f"TR ret {dev.ret} iter {dev.iter} obj {dev.obj_val}; {len(dev.checked)} trial merits "
          f"({sum(c[0] for c in dev.checked)} in restoration), worst error / scale {worst:.2e}")
    assert len(dev.checked) >= len(dev.problems)
    assert worst <= 1e-11
