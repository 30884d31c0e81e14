"""N-1 contingencies of the ACOPF model (activesetmethods_b200/examples/acopf.py): an out-of-service branch or generator
keeps its variables, rows and Jacobian entries and is taken out by values and bounds only.  Checked against the same
network with the element deleted: the shared Jacobian pattern, the callbacks at random points, the implied angle bound,
whole oracle runs, and a mixed batch through the lock-step line-search driver on the CPU engine."""
import copy

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import floyd_warshall

from activesetmethods_b200.examples import acopf
from activesetmethods_b200.slp import Model, Parameters, SlpLS, SlpLSBatch
from cpu_engine import OracleBatchEngine, OracleEngine
from oracle import slp_oracle as so

BRANCH = ("f_bus", "t_bus", "br_r", "br_x", "br_b", "tap", "shift", "rate_a", "angmin", "angmax", "br_status")
GEN = ("gen_bus", "pmin", "pmax", "qmin", "qmax", "cost2", "cost1", "cost0", "gen_status")


def _case118():
    return acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])


def _outage(net, branch=(), gen=()):
    out = copy.copy(net)
    out.br_status = net.br_status.copy()
    out.br_status[list(branch)] = 0
    out.gen_status = net.gen_status.copy()
    out.gen_status[list(gen)] = 0
    return out


def _deleted(net, branch=(), gen=()):
    """The network with the elements removed from its arrays (the formulation the outage must reproduce)."""
    out = copy.copy(net)
    kb = np.ones(net.nl, bool)
    kb[list(branch)] = False
    kg = np.ones(net.ng, bool)
    kg[list(gen)] = False
    for k in BRANCH:
        setattr(out, k, getattr(net, k)[kb])
    for k in GEN:
        setattr(out, k, getattr(net, k)[kg])
    return out, kb, kg


def _maps(full, kb, kg):
    """Indices of the deleted model's variables and rows in the full model."""
    nb, nl, ng, nd = full.nb, full.nl, full.ng, full.nd
    br, gn = np.nonzero(kb)[0], np.nonzero(kg)[0]
    cols = np.concatenate([full.o_va + np.arange(nb), full.o_vm + np.arange(nb), full.o_pg + gn, full.o_qg + gn,
                           full.o_p + br, full.o_p + nl + br, full.o_q + br, full.o_q + nl + br,
                           full.o_pdc + np.arange(2 * nd), full.o_qdc + np.arange(2 * nd)])
    rows = np.concatenate([full.r_angmax + br, full.r_angmin + br, [full.r_ref], full.r_dc + np.arange(nd),
                           (full.r_thermal + 2 * br[:, None] + np.arange(2)).ravel(), full.r_bal + np.arange(2 * nb),
                           (full.r_ohm + 4 * br[:, None] + np.arange(4)).ravel()])
    return cols, rows


def _jac(mdl, x):
    v = mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz))
    return coo_matrix((v, (mdl.j_str[:, 0] - 1, mdl.j_str[:, 1] - 1)), shape=(mdl.m, mdl.n)).toarray()


def _random_point(mdl, rng):
    lo = np.where(np.isfinite(mdl.x_L), mdl.x_L, -0.5)
    hi = np.where(np.isfinite(mdl.x_U), mdl.x_U, 0.5)
    return rng.uniform(lo, hi)


def _arcs(mdl, branch):
    b = np.asarray(branch, dtype=np.int64)
    return np.concatenate([mdl.o_p + b, mdl.o_p + mdl.nl + b, mdl.o_q + b, mdl.o_q + mdl.nl + b])


def _path_bounds(net):
    """All-pairs shortest paths over the in-service branches, weight max(angmax, -angmin), parallel branches by their
    smallest weight: written out independently of the model's own computation."""
    W = np.full((net.nb, net.nb), np.inf)
    for f, t, lo, hi, on in zip(net.f_bus, net.t_bus, net.angmin, net.angmax, net.br_status):
        if on:
            w = max(hi, -lo)
            W[f, t] = W[t, f] = min(W[f, t], w)
    return floyd_warshall(W, directed=False)


# ---- 1. pattern --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["case9", "case118"])
def test_contingencies_share_the_base_pattern(name):
    net = acopf.case9() if name == "case9" else _case118()
    base = acopf.AcopfModel(net)
    branch = acopf.branch_contingencies(net)
    gen = acopf.generator_contingencies(net)
    assert len(branch) == {"case9": 6, "case118": 170}[name]
    assert len(gen) == net.ng
    for c in branch + gen:
        assert int((c.br_status == 0).sum() + (c.gen_status == 0).sum()) == 1
        mdl = acopf.AcopfModel(c)
        assert (mdl.n, mdl.m, mdl.nnz) == (base.n, base.m, base.nnz)
        assert np.array_equal(mdl.j_str, base.j_str)
    # the base network is untouched and the helpers honour count
    assert np.all(net.br_status == 1) and np.all(net.gen_status == 1)
    assert [int(np.argmin(c.br_status)) for c in acopf.branch_contingencies(net, count=3)] == \
        [int(np.argmin(c.br_status)) for c in branch[:3]]


def test_default_status_leaves_the_model_unchanged():
    """A network built without statuses is all in service, and its model's bounds and callbacks are exactly those of
    an explicit all-ones status."""
    net = _case118()
    assert net.br_status.shape == (net.nl,) and net.gen_status.shape == (net.ng,)
    a = acopf.AcopfModel(net)
    b = acopf.AcopfModel(_outage(net))
    x = _random_point(a, np.random.default_rng(0))
    for k in ("x_L", "x_U", "g_L", "g_U", "x0"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert np.array_equal(a.eval_g(x, np.zeros(a.m)), b.eval_g(x, np.zeros(b.m)))


# ---- 2. evaluator equivalence with deletion -----------------------------------------------------------------------
@pytest.mark.parametrize("name,branch,gen", [
    ("case9", (1,), ()), ("case9", (5,), ()), ("case9", (8,), ()), ("case9", (), (0,)), ("case9", (), (2,)),
    ("case118", (0,), ()), ("case118", (150,), ()), ("case118", (130, 170), ()), ("case118", (), (7,)),
    ("case118", (140,), (3,))])
def test_outage_equals_deletion(name, branch, gen):
    net = acopf.case9() if name == "case9" else _case118()
    full = acopf.AcopfModel(_outage(net, branch, gen))
    dnet, kb, kg = _deleted(net, branch, gen)
    dele = acopf.AcopfModel(dnet)
    cols, rows = _maps(full, kb, kg)
    assert (len(cols), len(rows)) == (dele.n, dele.m)
    out_cols = np.setdiff1d(np.arange(full.n), cols)
    gcols = np.concatenate([full.o_pg + np.asarray(gen, dtype=np.int64), full.o_qg + np.asarray(gen, dtype=np.int64)])
    assert np.array_equal(out_cols, np.sort(np.concatenate([_arcs(full, branch), gcols])))
    # bounds: the shared variables and rows keep theirs (the angle rows of the outaged branches are not shared)
    assert np.array_equal(full.x_L[cols], dele.x_L) and np.array_equal(full.x_U[cols], dele.x_U)
    assert np.array_equal(full.g_L[rows], dele.g_L) and np.array_equal(full.g_U[rows], dele.g_U)
    assert np.all(full.x_L[gcols] == 0.0) and np.all(full.x_U[gcols] == 0.0)
    cost0 = float(net.cost0[list(gen)].sum())
    rng = np.random.default_rng(len(branch) * 10 + len(gen))
    for _ in range(3):
        x = _random_point(full, rng)
        x[out_cols] = 0.0            # what the outaged Ohm rows and the generator bounds force
        xd = x[cols]
        assert full.eval_f(x) == pytest.approx(dele.eval_f(xd) + cost0, rel=1e-14, abs=1e-12)
        gf = full.eval_grad_f(x, np.zeros(full.n))
        assert np.array_equal(gf[cols], dele.eval_grad_f(xd, np.zeros(dele.n)))
        g = full.eval_g(x, np.zeros(full.m))
        np.testing.assert_allclose(g[rows], dele.eval_g(xd, np.zeros(dele.m)), rtol=1e-14, atol=1e-14)
        J = _jac(full, x)
        np.testing.assert_allclose(J[np.ix_(rows, cols)], _jac(dele, xd), rtol=1e-14, atol=1e-14)
        # the outaged Ohm rows read p - 0 and q - 0: value and derivative of the arc flow only
        ohm = (full.r_ohm + 4 * np.asarray(branch, dtype=np.int64)[:, None] + np.arange(4)).ravel()
        assert np.all(g[ohm] == 0.0)
        Jo = J[ohm]
        for r, c in zip(ohm, np.stack([full.o_p + np.asarray(branch), full.o_q + np.asarray(branch),
                                       full.o_p + full.nl + np.asarray(branch),
                                       full.o_q + full.nl + np.asarray(branch)], 1).ravel()):
            assert J[r, c] == 1.0
        assert np.count_nonzero(Jo) == len(ohm)
    # at a point with nonzero flows the outaged Ohm rows equal the arc flows
    x = _random_point(full, rng)
    g = full.eval_g(x, np.zeros(full.m))
    for l in branch:
        ro = full.r_ohm + 4 * l
        assert np.array_equal(g[ro:ro + 4], x[[full.o_p + l, full.o_q + l, full.o_p + full.nl + l,
                                               full.o_q + full.nl + l]])


# ---- 3. angle bound and islanding --------------------------------------------------------------------------------
@pytest.mark.parametrize("name,branch", [("case9", (1,)), ("case9", (2,)), ("case9", (8,)), ("case118", (0,)),
                                         ("case118", (20,)), ("case118", (130, 170, 60))])
def test_relaxed_angle_bound_is_the_shortest_path(name, branch):
    net = _outage(acopf.case9() if name == "case9" else _case118(), branch)
    mdl = acopf.AcopfModel(net)
    D = _path_bounds(net)
    for l in range(net.nl):
        if l in branch:
            d = D[net.f_bus[l], net.t_bus[l]]
            assert np.isfinite(d) and d > 0
            assert mdl.g_U[mdl.r_angmax + l] == pytest.approx(d, rel=1e-15)
            assert mdl.g_L[mdl.r_angmin + l] == pytest.approx(-d, rel=1e-15)
        else:
            assert mdl.g_U[mdl.r_angmax + l] == net.angmax[l] and mdl.g_L[mdl.r_angmin + l] == net.angmin[l]


def test_parallel_branches_count_once_in_the_angle_bound():
    """Of two parallel branches the one with the tighter angle limits gives the path length."""
    net = acopf.case9()
    for k in BRANCH:
        a = getattr(net, k)
        setattr(net, k, np.concatenate([a, a[[2]]]))      # a second 5-6 branch ...
    net.angmax[-1], net.angmin[-1] = 0.2, -0.1             # ... with limits of 0.2 rad
    mdl = acopf.AcopfModel(_outage(net, (1,)))             # 4-5 out: 4-9-8-7-6-5, the last hop over the new branch
    assert mdl.g_U[mdl.r_angmax + 1] == pytest.approx(4 * np.pi / 3 + 0.2, rel=1e-15)


def test_islanding_outage_raises():
    net = acopf.case9()
    for l in (0, 3, 6):                                    # the three generator step-up branches are bridges
        with pytest.raises(ValueError, match=f"branch {l} "):
            acopf.AcopfModel(_outage(net, (l,)))
    with pytest.raises(ValueError, match="islands"):
        acopf.AcopfModel(_outage(net, (1, 8)))             # 4-5 and 9-4 together cut bus 4 off the loop
    net = _case118()
    kept = {int(np.argmin(c.br_status)) for c in acopf.branch_contingencies(net)}
    for l in range(net.nl):
        if l in kept:
            continue
        with pytest.raises(ValueError, match="islands"):
            acopf.AcopfModel(_outage(net, (l,)))


# ---- 4. whole runs with the oracle -------------------------------------------------------------------------------
def _oracle(mdl):
    s = so.SlpLS(mdl, so.Parameters())
    s.run()
    return s


@pytest.mark.parametrize("name", ["case9", "case118"])
def test_oracle_runs_match_deletion(name):
    net = acopf.case9() if name == "case9" else _case118()
    for c in acopf.branch_contingencies(net, count=6):
        l = int(np.argmin(c.br_status))
        mdl = acopf.AcopfModel(c)
        a = _oracle(mdl)
        b = _oracle(acopf.AcopfModel(_deleted(net, (l,))[0]))
        assert a.ret == 0 and b.ret == 0, (l, a.ret, b.ret)
        assert abs(a.obj_val - b.obj_val) <= 1e-3 * abs(b.obj_val), (l, a.obj_val, b.obj_val)
        assert np.max(np.abs(a.x[_arcs(mdl, [l])])) <= 1e-9, l


def test_oracle_generator_outage_matches_deletion():
    net = acopf.case9()
    a = _oracle(acopf.AcopfModel(_outage(net, gen=(0,))))
    b = _oracle(acopf.AcopfModel(_deleted(net, gen=(0,))[0]))
    assert a.ret == 0 and b.ret == 0
    assert abs((a.obj_val - net.cost0[0]) - b.obj_val) <= 1e-3 * abs(b.obj_val)


# ---- 5. mixed batch on the CPU engine ----------------------------------------------------------------------------
def _mixed_case9():
    net = acopf.case9()
    nets = [net] + acopf.branch_contingencies(net)[:3]
    tap = copy.copy(net)
    tap.tap = net.tap.copy()
    tap.tap[4] = 1.05
    imp = copy.copy(net)
    imp.br_x = net.br_x.copy()
    imp.br_x[7] *= 1.3
    return nets + [tap, imp, acopf.generator_contingencies(net)[1]]


def test_mixed_batch_equals_single_runs():
    """Base case, branch outages, a tap change, an impedance change and a generator outage in one lock-step batch:
    every scenario gets exactly what its own SlpLS run gets (the bars of test_batched_line_search_equals_single_runs)."""
    nets = _mixed_case9()
    batch = SlpLSBatch([acopf.AcopfModel(n) for n in nets],
                       Parameters(max_iter=100, external_optimizer=OracleBatchEngine)).run()
    for s, n in enumerate(nets):
        one = SlpLS(Model.from_problem(acopf.AcopfModel(n),
                                       Parameters(max_iter=100, external_optimizer=OracleEngine))).run()
        assert batch.ret[s] == one.ret and batch.iter[s] == one.iter, (s, batch.ret[s], one.ret)
        assert np.allclose(batch.x[s], one.x, rtol=0, atol=1e-9)
        assert abs(batch.obj_val[s] - one.obj_val) <= 1e-9 * abs(one.obj_val)
    assert np.all(batch.ret == 0)
