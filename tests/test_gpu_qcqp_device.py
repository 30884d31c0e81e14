"""Device-side QCQP evaluator (asm_slp_attach_qcqp / eval_qcqp / qcqp_trial) lane by lane against a long-double
restatement of the term sums, on ACR case3, case9 and the synthetic case118 at B = 1, 33 and 1024, and on RandomNlp.

Error bars are derived a priori.  The kernels round one operation at a time (no FMA): a term q x_i x_j carries at most
two roundings, and an output that sums K terms in any fixed order is within gamma_{K+2} * sum |term| of the exact sum,
gamma_k = k u / (1 - k u), u = 2^-53 (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., (3.4)-(3.5)).
The restatement computes the exact sum to long-double accuracy, whose own error is two orders below the bar.  Also:
bit-identical repeats and batch permutations, the trial merit against compute_phi on the host in both phases, every
validation failure and call-order error, and the sub-LP an evaluation feeds."""
import numpy as np
import pytest

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf, small_nlps
from activesetmethods_b200.examples.qcqp import QcqpModel, random_nlp_as_qcqp
from helpers import problem
from test_oracle_pins import case3_network

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
LD = np.longdouble


def _model(name):
    if name == "case3":
        return acopf.AcrModel(case3_network())
    if name == "random":
        return random_nlp_as_qcqp(small_nlps.RandomNlp(n=40, m=30, seed=5))
    return acopf.AcrModel(acopf.case9() if name == "case9" else problem(name).net)


def _gamma(k):
    return k * U / (1.0 - k * U)


def _sum_rows(idx, vals, length):
    """[len, B] long-double sums of vals [T, B] into rows idx [T] (and the sums of |vals|, the counts)."""
    B = vals.shape[1]
    out = np.zeros((length, B), dtype=LD)
    mag = np.zeros((length, B), dtype=LD)
    np.add.at(out, idx, vals)
    np.add.at(mag, idx, np.abs(vals))
    return out, mag, np.bincount(idx, minlength=length)


def restate(M, x):
    """Long-double f, df, E, dE at x [B, n] and their bars (same shapes)."""
    X = x.T.astype(LD)                                   # [n, B]
    # objective: c0 + affine + quadratic terms
    to = np.concatenate([M.oa_coef.astype(LD)[:, None] * X[M.oa_col],
                         M.oq_coef.astype(LD)[:, None] * X[M.oq_i] * X[M.oq_j]])
    f = LD(M.c0) + to.sum(axis=0)
    fbar = _gamma(len(to) + 3) * (abs(LD(M.c0)) + np.abs(to).sum(axis=0))
    # rows
    ta = M.a_coef.astype(LD)[:, None] * X[M.a_col]
    tq = M.q_coef.astype(LD)[:, None] * X[M.q_i] * X[M.q_j]
    E, Emag, Ecnt = _sum_rows(np.r_[M.a_row, M.q_row], np.concatenate([ta, tq]), M.m)
    Ebar = _gamma(Ecnt + 2)[:, None] * Emag
    # Jacobian entries and gradient: contributions c * x_v or constants c
    def contrib(coef, var):
        c = coef.astype(LD)[:, None]
        return np.where(var[:, None] >= 0, c * X[np.maximum(var, 0)], c * np.ones_like(X[:1]))
    dE, dmag, dcnt = _sum_rows(M._jac_pos, contrib(M._jac_coef, M._jac_var), M.nnz)
    dEbar = _gamma(dcnt + 1)[:, None] * dmag
    df, gmag, gcnt = _sum_rows(M._grad_col, contrib(M._grad_coef, M._grad_var), M.n)
    dfbar = _gamma(gcnt + 1)[:, None] * gmag
    return (f, df.T, E.T, dE.T), (fbar, dfbar.T, Ebar.T, dEbar.T)


def _points(M, B, seed):
    rng = np.random.default_rng(seed)
    lo = np.where(np.isfinite(M.x_L), M.x_L, -1.5)
    hi = np.where(np.isfinite(M.x_U), M.x_U, 1.5)
    return rng.uniform(lo, hi, (B, M.n))


def _handle(M, B):
    from activesetmethods_b200.sublp import SubLp
    lp = SubLp(M.n, M.m, M.j_str, M.x_L, M.x_U, M.g_L, M.g_U, batch=B, eps_rel=1e-7)
    lp._squeeze = False
    return lp


@pytest.mark.parametrize("name,B", [(n, b) for n in ("case3", "case9", "case118") for b in (1, 33, 1024)] +
                         [("random", 1), ("random", 33)])
def test_eval_against_long_double(gpu, name, B):
    M = _model(name)
    x = _points(M, B, seed=B)
    lp = _handle(M, B)
    lp.attach_qcqp(M)
    lp.eval_qcqp(x, 1000.0, False)
    got = lp.get_eval()
    ref, bar = restate(M, x)
    worst = {}
    for key, g, r, b in zip(("f", "df", "E", "dE"), got, ref, bar):
        err = np.abs(g.astype(LD) - r)
        assert np.all(err <= 1.01 * b + 1e-300), (key, np.argwhere(err > 1.01 * b + 1e-300)[:5])
        worst[key] = float(np.max(err / (b + 1e-300)))
    print(f"{name} B={B}: worst error / bar {worst}")
    # the host callbacks agree with the device to the same bars
    for s in (0, B - 1):
        assert abs(M.eval_f(x[s]) - got[0][s]) <= 2.02 * bar[0][s] + 1e-300
        assert np.all(np.abs(M.eval_jac_g(x[s], "eval", None, None, np.zeros(M.nnz)) - got[3][s]) <= 2.02 * bar[3][s] + 1e-300)
    lp.close()


@pytest.mark.parametrize("name", ["case9", "case118"])
def test_deterministic_and_lane_independent(gpu, name):
    M = _model(name)
    B = 96
    x = _points(M, B, seed=7)
    lp = _handle(M, B)
    lp.attach_qcqp(M)
    lp.eval_qcqp(x, 1000.0, False)
    a = lp.get_eval()
    lp.eval_qcqp(x, 1000.0, False)
    b = lp.get_eval()
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    perm = np.random.default_rng(1).permutation(B)
    lp.eval_qcqp(x[perm], 1000.0, False)
    c = lp.get_eval()
    for u, v in zip(a, c):
        assert np.array_equal(u[perm], v)
    # one scenario alone on a batch-of-one handle: the same bits as its lane of the batch
    one = _handle(M, 1)
    one.attach_qcqp(M)
    one.eval_qcqp(x[5:6], 1000.0, False)
    d = one.get_eval()
    for u, v in zip(a, d):
        assert np.array_equal(u[5:6], v)
    lp.close()
    one.close()


@pytest.mark.parametrize("name,B", [("case9", 1), ("case118", 33)])
def test_trial_merit_both_phases(gpu, name, B):
    """qcqp_trial = compute_phi(x + alpha p) with f, g of the model at the trial point (slp.jl:79-115): normal phase
    against the formula on the host, restoration against merit_phi with g(x + alpha p) from the host callbacks."""
    M = _model(name)
    x0 = np.tile(np.clip(M.x0, M.x_L, M.x_U), (B, 1))
    x0 += 1e-3 * np.random.default_rng(2).standard_normal(x0.shape)
    x0 = np.clip(x0, M.x_L, M.x_U)
    lp = _handle(M, B)
    lp.attach_qcqp(M)
    rng = np.random.default_rng(4)
    for fr in (False, True):
        lp.eval_qcqp(x0, 0.05, fr)
        p, lam = lp.solve_extract()[:2]
        p, lam = np.atleast_2d(p), np.atleast_2d(lam)
        nu = np.abs(lam) + 0.5
        alpha = rng.uniform(0.05, 1.0, B)
        Et = np.array([M.eval_g(x0[s] + alpha[s] * p[s], np.zeros(M.m)) for s in range(B)])
        if fr:
            base = rng.uniform(0.0, 1.0, B)
            phi = lp.qcqp_trial(alpha, nu, base, True)
            ref = lp.merit_phi(base, Et, nu, alpha, True)
        else:
            phi = lp.qcqp_trial(alpha, nu)
            ref = np.array([M.eval_f(x0[s] + alpha[s] * p[s]) + float(np.sum(
                nu[s] * np.maximum(0.0, np.maximum(Et[s] - M.g_U, M.g_L - Et[s])))) for s in range(B)])
        assert np.all(np.abs(phi - ref) <= 1e-10 * np.maximum(1.0, np.abs(ref))), (fr, np.abs(phi - ref).max())
    lp.close()


@pytest.mark.parametrize("name,B", [("case9", 1), ("case118", 33), ("random", 1)])
def test_same_sublp_as_host_handover(gpu, name, B):
    """An evaluation feeds the same sub-LP as a host hand-over (asm_slp_update) of the same numbers."""
    M = _model(name)
    lp = _handle(M, B)
    lp.attach_qcqp(M)
    x0 = np.tile(np.clip(M.x0, M.x_L, M.x_U), (B, 1))
    lp.eval_qcqp(x0, 1000.0, False)
    st = np.atleast_1d(lp.solve_extract()[5])
    obj_dev = np.array([i["objective"] for i in lp.last_info])
    rp, ci, v_dev = lp.jacobian_csr(0)
    f0, df0, E0, dE0 = lp.get_eval()
    out = lp.sub_optimize(x0, f0, df0, E0, dE0, 1000.0, False)
    obj_host = np.array([i["objective"] for i in lp.last_info])
    assert np.array_equal(lp.jacobian_csr(0)[2], v_dev)
    assert np.array_equal(st, np.atleast_1d(out[5]))
    ok = st == 0
    assert np.all(np.abs(obj_dev - obj_host)[ok] <= 1e-6 * np.maximum(1.0, np.abs(obj_host[ok])))
    lp.close()


class _Desc:
    """A QcqpModel's description with some fields replaced."""

    def __init__(self, M, **over):
        self.d = dict(M.qcqp_desc(), **over)

    def qcqp_desc(self):
        return self.d


def _attach_rc(lp, desc):
    try:
        lp.attach_qcqp(desc)
        return capi.OK
    except capi.AsmError as e:
        return e.code


def test_validation_errors(gpu):
    M = _model("case9")
    lp = _handle(M, 1)
    d = M.qcqp_desc()
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)   # noqa: E731
    i64 = lambda a: np.ascontiguousarray(a, dtype=np.int64)   # noqa: E731
    diag = np.nonzero(M.q_i == M.q_j)[0][0]
    off = np.nonzero(M.q_i != M.q_j)[0][0]
    swapped = d["quad_pos"].copy()
    swapped[[2 * off, 2 * off + 1]] = swapped[[2 * off + 1, 2 * off]]
    bad = {
        "n": dict(n=M.n + 1), "m": dict(m=M.m - 1), "nnz": dict(nnz_coo=M.nnz + 1),
        "aff col": dict(aff_col=i32(np.r_[M.n, d["aff_col"][1:]])),
        "aff row": dict(aff_row=i32(np.r_[-1, d["aff_row"][1:]])),
        "quad j": dict(quad_j=i32(np.r_[d["quad_j"][:-1], M.n])),
        "obj col": dict(obj_aff_col=i32(np.r_[d["obj_aff_col"][:-1], -3])),
        "obj quad": dict(obj_quad_i=i32(np.r_[M.n + 5, d["obj_quad_i"][1:]])),
        "nan quad": dict(quad_coef=np.r_[np.nan, d["quad_coef"][1:]]),
        "inf aff": dict(aff_coef=np.r_[d["aff_coef"][:-1], np.inf]),
        "inf obj": dict(obj_quad_coef=np.r_[-np.inf, d["obj_quad_coef"][1:]]),
        "nan c0": dict(c0=np.nan),
        "pos range": dict(aff_pos=i64(np.r_[M.nnz, d["aff_pos"][1:]])),
        "pos negative": dict(aff_pos=i64(np.r_[-1, d["aff_pos"][1:]])),
        # the position of another term: in range, but not at this term's (row, col)
        "aff pos other": dict(aff_pos=i64(np.r_[d["aff_pos"][1], d["aff_pos"][1:]])),
        "quad pos swapped": dict(quad_pos=swapped),
        "diag second pos": dict(quad_pos=i64(np.where(np.arange(2 * len(M.q_i)) == 2 * diag + 1,
                                                      d["quad_pos"][2 * diag], d["quad_pos"]))),
        "off first pos -1": dict(quad_pos=i64(np.where(np.arange(2 * len(M.q_i)) == 2 * off + 1, -1, d["quad_pos"]))),
    }
    for why, over in bad.items():
        assert _attach_rc(lp, _Desc(M, **over)) == capi.E_INVALID, why
        assert lp._lib.asm_last_error().decode(), why
    # a failed attach leaves the handle without an evaluator
    x = np.clip(M.x0, M.x_L, M.x_U)[None]
    with pytest.raises(capi.AsmError) as e:
        lp.eval_qcqp(x)
    assert e.value.code == capi.E_STATE
    assert _attach_rc(lp, M) == capi.OK
    lp.close()


def test_untargeted_entries_are_written_zero(gpu):
    """A j_str entry no term targets (here one appended to a row) reads 0 after every evaluation, whatever the
    handle held there before."""
    M = _model("case3")
    extra = np.array([[M.j_str[0, 0], M.n]])                 # (row of entry 0, last column), 1-based
    j_str = np.vstack([M.j_str, extra])
    from activesetmethods_b200.sublp import SubLp
    lp = SubLp(M.n, M.m, j_str, M.x_L, M.x_U, M.g_L, M.g_U, batch=33)
    lp._squeeze = False
    x = _points(M, 33, 3)
    lp.update(x, np.zeros(33), np.ones((33, M.n)), np.ones((33, M.m)), np.full((33, M.nnz + 1), 7.0), 1000.0)
    lp.attach_qcqp(_Desc(M, nnz_coo=M.nnz + 1))
    lp.eval_qcqp(x)
    dE = lp.get_eval()[3]
    assert np.all(dE[:, -1] == 0.0)
    ref, bar = restate(M, x)
    assert np.all(np.abs(dE[:, :-1].astype(LD) - ref[3]) <= 1.01 * bar[3] + 1e-300)
    lp.close()


def _all_affine(P):
    """A QcqpModel whose j_str is exactly that of the AcopfModel P (one affine term per entry): a handle made for P
    accepts both evaluators."""
    r, c = P.j_str[:, 0] - 1, P.j_str[:, 1] - 1
    assert np.all(np.diff(r) >= 0)
    return QcqpModel(P.n, P.x_L, P.x_U, P.g_L, P.g_U, P.x0, obj_aff=([0], [1.0]), aff=(r, c, np.ones(len(r))))


def test_call_order_and_switching(gpu):
    from activesetmethods_b200.sublp import SubLp
    P = acopf.AcopfModel(acopf.case9())
    Q = _all_affine(P)
    assert np.array_equal(Q.j_str, P.j_str)
    lp = SubLp(P.n, P.m, P.j_str, P.x_L, P.x_U, P.g_L, P.g_U)
    lib, h = lp._lib, lp._h
    d = capi.dptr
    x = np.clip(P.x0, P.x_L, P.x_U)
    one, nu, out = np.ones(1), np.ones(P.m), np.zeros(1)

    def codes():
        return (lib.asm_slp_eval_qcqp(h, d(x), d(one), 0), lib.asm_slp_eval_acopf(h, d(x), d(one), 0))

    assert codes() == (capi.E_STATE, capi.E_STATE)
    assert lib.asm_slp_qcqp_trial(h, d(one), d(nu), None, 0, d(out)) == capi.E_STATE
    lp.attach_acopf(P)
    assert codes() == (capi.E_STATE, capi.OK)
    lp.attach_qcqp(Q)                            # detaches the ACOPF evaluator
    assert codes() == (capi.OK, capi.E_STATE)
    assert lib.asm_slp_acopf_trial(h, d(one), d(nu), None, 0, d(out)) == capi.E_STATE
    assert lib.asm_slp_acopf_branch_coef(h, d(np.zeros(12 * P.nl))) == capi.E_STATE
    # trial before a solve
    assert lib.asm_slp_qcqp_trial(h, d(one), d(nu), None, 0, d(out)) == capi.E_STATE
    lp.solve_extract()
    assert lib.asm_slp_qcqp_trial(h, d(one), d(nu), None, 0, d(out)) == capi.OK
    assert lib.asm_slp_qcqp_trial(h, d(one), d(nu), None, 1, d(out)) == capi.E_INVALID      # restoration needs base
    assert lib.asm_slp_eval_qcqp(h, None, d(one), 0) == capi.E_INVALID
    # the evaluation is the all-affine model's: E = sum of the row's columns, dE = 1
    f, df, E, dE = lp.get_eval()
    assert np.all(dE == 1.0) and f == x[0] and np.array_equal(df, np.eye(P.n)[0])
    lp.attach_acopf(P)                           # and back
    assert codes() == (capi.E_STATE, capi.OK)
    assert lib.asm_slp_qcqp_trial(h, d(one), d(nu), None, 0, d(out)) == capi.E_STATE
    lp.close()
