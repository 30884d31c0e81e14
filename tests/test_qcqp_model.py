"""Affine / quadratic models (examples/qcqp.py) and the rectangular-voltage OPF (acopf.AcrModel) on the host: callbacks
against central differences, RandomNlp restated as term lists, the toy problem, and ACR against ACP in the CPU
oracle.  No device: the C ABI is only reached for its argument checks."""
import ctypes as C
import re

import numpy as np
import pytest

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf, small_nlps
from activesetmethods_b200.examples.qcqp import QcqpModel, random_nlp_as_qcqp, toy_qcqp
from helpers import problem
from oracle import slp_oracle as so
from test_abi import header_symbols
from test_oracle_pins import case3_network


def _fd_jacobian_error(M, x, h=1e-6):
    v = M.eval_jac_g(x, "eval", None, None, np.zeros(M.nnz))
    J = np.zeros((M.m, M.n))
    np.add.at(J, (M.j_str[:, 0] - 1, M.j_str[:, 1] - 1), v)
    Jn = np.zeros_like(J)
    for k in range(M.n):
        e = np.zeros(M.n)
        e[k] = h
        Jn[:, k] = (M.eval_g(x + e, np.zeros(M.m)) - M.eval_g(x - e, np.zeros(M.m))) / (2 * h)
    return float(np.max(np.abs(J - Jn)))


def random_qcqp(seed=0, n=9, m=7, n_aff=20, n_quad=25):
    """Random term lists with repeated terms, diagonal terms and a row without terms."""
    rng = np.random.default_rng(seed)
    quad_r = rng.integers(0, m - 1, n_quad)
    qi, qj = rng.integers(0, n, n_quad), rng.integers(0, n, n_quad)
    qj[:4] = qi[:4]
    return QcqpModel(n, np.full(n, -2.0), np.full(n, 2.0), np.full(m, -1.0), np.full(m, 1.0), np.zeros(n),
                     obj_const=0.7, obj_aff=(rng.integers(0, n, 6), rng.standard_normal(6)),
                     obj_quad=(np.r_[0, 1, rng.integers(0, n, 5)], np.r_[0, 2, rng.integers(0, n, 5)],
                               rng.standard_normal(7)),
                     aff=(rng.integers(0, m - 1, n_aff), rng.integers(0, n, n_aff), rng.standard_normal(n_aff)),
                     quad=(quad_r, qi, qj, rng.standard_normal(n_quad)))


def test_qcqp_callbacks_match_central_differences():
    M = random_qcqp()
    x = np.random.default_rng(1).uniform(-1, 1, M.n)
    assert _fd_jacobian_error(M, x) <= 1e-8
    g = M.eval_grad_f(x, np.zeros(M.n))
    gn = np.array([(M.eval_f(x + h) - M.eval_f(x - h)) / 2e-6 for h in 1e-6 * np.eye(M.n)])
    assert np.max(np.abs(g - gn)) <= 1e-8
    # the row without terms has no j_str entries and evaluates to 0
    assert M.m not in set(M.j_str[:, 0]) and M.eval_g(x, np.ones(M.m))[-1] == 0.0


def test_qcqp_pattern_has_reference_layout():
    """One entry per affine term, one per distinct variable of each quadratic term, row by row (duplicates kept)."""
    M = random_qcqp()
    expect = []
    for r in range(M.m):
        for k in np.nonzero(M.a_row == r)[0]:
            expect.append((r + 1, M.a_col[k] + 1))
        for k in np.nonzero(M.q_row == r)[0]:
            expect.append((r + 1, M.q_i[k] + 1))
            if M.q_i[k] != M.q_j[k]:
                expect.append((r + 1, M.q_j[k] + 1))
    assert [tuple(e) for e in M.j_str] == expect
    assert np.all(M.quad_pos[1::2][M.q_i == M.q_j] == -1)


def test_random_nlp_restated_as_qcqp():
    for seed in range(3):
        p = small_nlps.RandomNlp(seed=seed)
        q = random_nlp_as_qcqp(p)
        assert np.array_equal(q.j_str, p.j_str)
        pat = so.JacobianPattern(p.m, p.n, p.j_str)
        for x in np.random.default_rng(seed).uniform(-1.5, 1.5, (4, p.n)):
            rel = lambda a, b: np.max(np.abs(a - b) / (1e-300 + np.maximum(np.abs(a), np.abs(b))), initial=0.0)  # noqa
            assert abs(q.eval_f(x) - p.eval_f(x)) <= 1e-14 * abs(p.eval_f(x))
            assert rel(q.eval_g(x, np.zeros(p.m)), p.eval_g(x, np.zeros(p.m))) <= 1e-14
            assert rel(q.eval_grad_f(x, np.zeros(p.n)), p.eval_grad_f(x, np.zeros(p.n))) <= 1e-14
            Jq = pat.assemble(q.eval_jac_g(x, "eval", None, None, np.zeros(q.nnz)))
            Jp = pat.assemble(p.eval_jac_g(x, "eval", None, None, np.zeros(p.nnz)))
            assert rel(Jq, Jp) <= 1e-14


def test_toy_qcqp_reaches_the_reference_optimum():
    r = so.optimize(toy_qcqp(), so.Parameters(max_iter=100))
    assert r.ret == 0
    assert np.allclose(r.x, [-1.0, -1.0], atol=1e-6)


@pytest.mark.parametrize("name,tol", [("case3", 1e-8), ("case9", 1e-8)])
def test_acr_jacobian_matches_central_differences(name, tol):
    net = case3_network() if name == "case3" else acopf.case9()
    M = acopf.AcrModel(net)
    x = np.random.default_rng(0).uniform(-1, 1, M.n)
    assert _fd_jacobian_error(M, x) <= tol


def test_acr_layout_and_start():
    net = acopf.case9()
    P, A = acopf.AcopfModel(net), acopf.AcrModel(net)
    nb = net.nb
    assert A.n == P.n and A.m == P.m + nb
    assert np.array_equal(A.x_L[2 * nb:], P.x_L[2 * nb:]) and np.array_equal(A.x_U[:nb], net.vmax)
    # the start is ACP's start as a physical point
    v = A.x0[:nb] + 1j * A.x0[nb:2 * nb]
    assert np.allclose(np.abs(v), P.x0[nb:2 * nb]) and np.allclose(np.angle(v), P.x0[:nb])
    # the same point gives the same physical rows
    gA, gP = A.eval_g(A.x0, np.zeros(A.m)), P.eval_g(P.x0, np.zeros(P.m))
    assert np.allclose(gA[A.r_bal:A.r_bal + 2 * nb], gP[P.r_bal:P.r_bal + 2 * nb], atol=1e-12)
    assert np.allclose(gA[A.r_ohm:], gP[P.r_ohm:], atol=1e-12)
    assert A.eval_f(A.x0) == pytest.approx(P.eval_f(P.x0), rel=1e-14)


def test_acr_rejects_branch_outages():
    c = acopf.branch_contingencies(acopf.case9(), count=1)[0]
    with pytest.raises(ValueError):
        acopf.AcrModel(c)
    g = acopf.generator_contingencies(acopf.case9())[0]
    A = acopf.AcrModel(g)          # a generator outage only changes bounds: the terms are the base case's
    assert A.same_terms(acopf.AcrModel(acopf.case9())) is None
    assert A.x_U[A.o_pg] == 0.0


def _pair(net, alg, max_iter):
    P, A = acopf.AcopfModel(net), acopf.AcrModel(net)
    rp = so.optimize(P, so.Parameters(algorithm=alg, max_iter=max_iter))
    ra = so.optimize(A, so.Parameters(algorithm=alg, max_iter=max_iter))
    return rp, ra


def test_acr_and_acp_reach_the_same_optimum_case9_tr():
    net = acopf.case9()
    rp, ra = _pair(net, "Trust Region", 100)
    assert rp.ret == 0 and ra.ret == 0
    assert abs(ra.obj_val - rp.obj_val) <= 1e-9 * abs(rp.obj_val)
    nb = net.nb
    vr, vi = ra.x[:nb], ra.x[nb:2 * nb]
    assert np.max(np.abs(np.hypot(vr, vi) - rp.x[nb:2 * nb])) <= 1e-6
    assert np.max(np.abs(np.arctan2(vi, vr) - rp.x[:nb])) <= 1e-6


def test_acr_and_acp_reach_the_same_optimum_case3_tr():
    rp, ra = _pair(case3_network(), "Trust Region", 100)
    assert rp.ret == 0 and ra.ret == 0
    assert abs(ra.obj_val - rp.obj_val) <= 1e-6 * abs(rp.obj_val)


def test_acr_and_acp_reach_the_same_optimum_case118_ls():
    rp, ra = _pair(problem("case118").net, "Line Search", 200)
    assert rp.ret == 0 and ra.ret == 0
    assert abs(ra.obj_val - rp.obj_val) <= 1e-3 * abs(rp.obj_val)


def test_qcqp_symbols_in_header_and_signatures():
    syms = header_symbols()
    for s in ("asm_slp_attach_qcqp", "asm_slp_eval_qcqp", "asm_slp_qcqp_trial"):
        assert s in syms and s in capi.SIGNATURES
    # the struct binding has the header's fields in the header's order
    hdr = open(capi.os.path.join(capi.os.path.dirname(capi.os.path.dirname(capi.__file__)), "include",
                                 "asm_b200.h")).read()
    body = re.search(r"typedef struct asm_qcqp_desc \{(.*?)\} asm_qcqp_desc;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\*?\s*(\w+)\s*[,;]", body)
    assert names == [f[0] for f in capi.QcqpDesc._fields_]


def test_attach_qcqp_null_handle_is_invalid(built_lib):
    d = capi.QcqpDesc()
    assert built_lib.asm_slp_attach_qcqp(None, C.byref(d)) == capi.E_INVALID
    assert built_lib.asm_slp_eval_qcqp(None, None, None, 0) == capi.E_INVALID
    assert built_lib.asm_slp_qcqp_trial(None, None, None, None, 0, None) == capi.E_INVALID


def test_driver_rejects_batches_with_different_terms():
    """A batch (or queue) whose models differ in anything but bounds and start fails before a handle is made."""
    from activesetmethods_b200.slp import SlpLSBatch, SlpTRBatch
    net = acopf.case9()
    a = acopf.AcrModel(net)
    other = acopf.case9()
    other.gs = other.gs.copy()
    other.gs[4] = 0.05                   # a shunt: an extra term in two balance rows ... and in j_str
    b = acopf.AcrModel(other)
    other2 = acopf.case9()
    other2.cost1 = other2.cost1 * 1.1    # same pattern, other objective coefficients
    c = acopf.AcrModel(other2)
    with pytest.raises(ValueError):
        SlpLSBatch([a, b], device_evaluator=True)
    with pytest.raises(ValueError, match="terms"):
        SlpLSBatch([a, c], device_evaluator=True).run()
    with pytest.raises(ValueError, match="terms"):
        SlpTRBatch([a, a, c], device_evaluator=True, lanes=2).run()
