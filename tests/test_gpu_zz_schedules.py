"""The barrier engine's two schedules -- supernodal (default) and one column per level of the elimination tree
(ASM_IPM_SUPERNODE=1, read when a handle builds its engine, for batches and single LPs alike) -- factorise the same
matrices with different kernels (dense panels + chunked updates vs single-term updates) and must return the same LP
solutions.  Both are also run through test_gpu_lp_conformance.py / test_gpu_sublp.py by setting the variable for the
whole run."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _inputs(B):
    from activesetmethods_b200.examples import acopf
    net = acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"])
    mdls = [acopf.AcopfModel(acopf.perturb_loads(net, s + 1)) for s in range(B)]
    stack = lambda fn: np.array([fn(m) for m in mdls])
    x = stack(lambda m: np.clip(m.x0, m.x_L, m.x_U))
    d = dict(x=x, f=np.array([m.eval_f(xx) for m, xx in zip(mdls, x)]),
             df=np.array([m.eval_grad_f(xx, np.zeros(m.n)) for m, xx in zip(mdls, x)]),
             E=np.array([m.eval_g(xx, np.zeros(m.m)) for m, xx in zip(mdls, x)]),
             dE=np.array([m.eval_jac_g(xx, "eval", None, None, np.zeros(m.nnz)) for m, xx in zip(mdls, x)]),
             xL=stack(lambda m: m.x_L), xU=stack(lambda m: m.x_U), gL=stack(lambda m: m.g_L), gU=stack(lambda m: m.g_U))
    return mdls[0], d


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("fr", [False, True])
def test_schedules_agree(gpu, monkeypatch, B, fr):
    from activesetmethods_b200.sublp import SubLp
    m0, d = _inputs(B)
    sq = (lambda a: a[0]) if B == 1 else (lambda a: a)
    res = {}
    for name, width in (("supernodal", "16"), ("levels", "1")):
        monkeypatch.setenv("ASM_IPM_SUPERNODE", width)
        lp = SubLp(m0.n, m0.m, m0.j_str, sq(d["xL"]), sq(d["xU"]), sq(d["gL"]), sq(d["gU"]), batch=B, engine=4)
        out = lp.sub_optimize(sq(d["x"]), sq(d["f"]), sq(d["df"]), sq(d["E"]), sq(d["dE"]), 1000.0, fr)
        res[name] = dict(status=np.atleast_1d(out[5]).astype(int),
                         obj=np.array([i["objective"] for i in lp.last_info]), steps=lp.ipm_info()["levels"])
        lp.close()
    a, b = res["supernodal"], res["levels"]
    assert a["steps"] < b["steps"]                           # the schedules really are different
    assert np.array_equal(a["status"], b["status"]) and np.all(a["status"] == 0)
    # same LPs, same algorithm, different summation order: the objectives agree far inside the path's 1e-6 bar
    assert np.all(np.abs(a["obj"] - b["obj"]) <= 1e-6 * np.maximum(1.0, np.abs(b["obj"])))
