"""The long-double PDHG reference (tests/pdhg_reference.py) on the CPU: it solves the generator's LPs as HiGHS
does, its float64 twin stays inside the rounding bars the GPU tests use, and every case the GPU tests run keeps
each discrete decision far enough from its threshold that those tests can demand exact equality."""
import numpy as np
import pytest

import pdhg_reference as R
from oracle import slp_oracle as so


def test_long_double_is_extended():
    assert np.finfo(np.longdouble).eps < 1e-18


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reference_matches_highs(seed):
    pat, lp = R.make_lp(14, 11, 4, seed)
    ref = R.solve(pat, lp, dict(eps_rel=1e-8))
    for s in range(4):
        K = R.scipy_matrix(pat, lp, s)
        st, x, y, z, obj = so.HighsLp().solve(K.tocsc(), lp["c"][:, s], lp["c0"][s], lp["lb"][:, s], lp["ub"][:, s],
                                              lp["rl"][:, s], lp["ru"][:, s])
        assert st == so.OPTIMAL and ref["status"][s] == R.OPTIMAL
        assert abs(ref["objective"][s] - obj) <= 1e-8 * (1.0 + abs(ref["pobj"][s]) + abs(ref["dobj"][s])) * 10
        xs = ref["x"][:, s]
        assert np.all(xs >= lp["lb"][:, s]) and np.all(xs <= lp["ub"][:, s])


@pytest.mark.parametrize("seed", [0, 1])
def test_infeasible_variant(seed):
    pat, lp = R.make_lp(12, 10, 4, seed, infeasible=True)
    ref = R.solve(pat, lp, dict(max_iter=20000))
    assert (ref["status"] == R.INFEASIBLE).all()
    for s in range(4):
        K = R.scipy_matrix(pat, lp, s)
        st = so.HighsLp().solve(K.tocsc(), lp["c"][:, s], 0.0, lp["lb"][:, s], lp["ub"][:, s], lp["rl"][:, s],
                                lp["ru"][:, s])[0]
        assert st == so.INFEASIBLE


# (n, m, B, seed, infeasible): the drift cases; the GPU cases are of the same kind and size
DRIFT_CASES = [(12, 10, 4, 1, False), (12, 10, 4, 2, False), (20, 16, 8, 3, False), (12, 10, 4, 0, True),
               (16, 12, 6, 5, False), (40, 30, 4, 7, False)]


def test_float64_twin_inside_the_bars():
    """The bars are 10x the worst rounding drift of a double implementation of this exact operation order: the
    float64 run of the same code against the long-double one, over windows of 1 block to termination."""
    worst = {}
    cases = [(R.make_lp(n, m, B, seed, infeasible=inf), (1, 3, 64)) for n, m, B, seed, inf in DRIFT_CASES]
    cases.append((R.case("hybrid"), (64,)))       # spread conditioning
    for (pat, lp), periods in cases:
        B = lp["vals"].shape[1]
        for ce in periods:
            for nb in (1, 2, 3, 10, 40, None):
                P = dict(R.TEST_PARAMS, check_every=ce)
                if nb:
                    P["max_iter"] = nb * max(2, ce)
                a = R.solve(pat, lp, P)
                b = R.solve(pat, lp, P, dtype=np.float64)
                for key in ("status", "iterations", "restarts"):
                    assert np.array_equal(a[key], b[key]), (key, ce, nb)
                for s in range(B):
                    for key, v in R.compare(b, a, s, s, a["iterations"][s]).items():
                        worst[key] = max(worst.get(key, 0.0), v)
                for ta, tb in zip(a["trace"], b["trace"]):
                    ok = np.isfinite(ta["r"])
                    if ok.any():
                        d = np.abs(ta["r"][ok] - tb["r"][ok]) / np.maximum(ta["r"][ok], 1e-300)
                        v = float(np.max(d / (R.BARS["r"] * np.sqrt(np.maximum(1, ta["it"] + ta["j"] + 1)))))
                        worst["r"] = max(worst.get("r", 0.0), v)
    print("\nworst float64 drift / bar:", {k: f"{v:.3f}" for k, v in worst.items()})
    for key, v in worst.items():
        assert v <= (0.025 if key == "x" else 0.1), (key, v)      # each bar is at least 10x the drift, x's 40x
    assert set(worst) == set(R.BARS)
    # and not needlessly loose: the worst drift uses at least 1/100 of every bar but r's (r's cancellation is rare)
    assert all(v >= 0.01 for k, v in worst.items() if k != "r"), worst


def _full(name, ce):
    pat, lp = R.case(name)
    cap = R.K_MAX_STEPS if ce > R.K_MAX_STEPS else None
    return R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=ce), period_cap=cap)


@pytest.mark.parametrize("name,ce", [(n, ce) for n in R.CASES if R.FULL_RUN.get(n, True) for ce in R.CHECK_EVERY[n]])
def test_margins_of_the_gpu_cases(name, ce):
    """Every discrete decision of every check of every lane is at least 100x its quantity's bar from the
    threshold, at the bar of the run's longest lane: a change of rounding cannot flip it."""
    full = _full(name, ce)
    it = int(full["iterations"].max())
    assert full["margins"]
    for key, v in full["margins"].items():
        need = 100 * R.bar(R.margin_quantity(key), it)
        assert v >= need, (key, v, need)


@pytest.mark.parametrize("name,ce,nb,warm", [("wide", 4, 1, False), ("wide", 4, 2, False), ("big", 64, 1, False),
                                             ("big", 64, 2, False), ("b3", 64, 2, True), ("b1", 64, 2, True),
                                             ("infeasible", 64, 2, True)])
def test_margins_of_the_gpu_windows(name, ce, nb, warm):
    """The windows the GPU tests compare without a full cold run here: the grid-stride and streamed-matrix cases
    (two blocks only) and the set_start runs from R.random_start (the infeasible one with y left cold).  The
    warm starts from a GPU solution and the SLP sub-LPs have their margins asserted where they run."""
    pat, lp = R.case(name)
    start = R.random_start(name) if warm else None
    if name == "infeasible":
        start = (start[0], np.zeros_like(start[1]))
    ref = R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=ce, max_iter=nb * ce), warm=int(warm), start=start)
    it = int(ref["iterations"].max())
    for key, v in ref["margins"].items():
        need = 100 * R.bar(R.margin_quantity(key), it)
        assert v >= need, (key, v, need)


def test_hybrid_case_compacts_then_hands_over():
    """Engine 5 on the hybrid case (hand_over 0.3 of 100 LPs = 30): some check period ends with 31..64 LPs running
    (128 -> 64) and a later one with at most 30 (hand-over to the group kernel)."""
    full = _full("hybrid", 64)
    its = full["iterations"]
    live = [(its > b * 64).sum() for b in range(1, its.max() // 64 + 1)]
    assert any(30 < v <= 64 for v in live) and any(0 < v <= 30 for v in live), live


def test_check_every_one_behaves_as_two():
    pat, lp = R.case("b3")
    a = R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=1))
    b = R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=2))
    for key in ("status", "iterations", "restarts", "x", "y", "zl", "zu", "objective"):
        assert np.array_equal(a[key], b[key]), key


def test_three_blocks_are_a_prefix_of_five():
    pat, lp = R.case("b3")
    a = R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=3, max_iter=9))
    b = R.solve(pat, lp, dict(R.TEST_PARAMS, check_every=3, max_iter=15))
    assert len(a["trace"]) == 6 and len(b["trace"]) == 10
    for ta, tb in zip(a["trace"], b["trace"]):
        for key in ("k", "r", "omega", "flag", "status"):
            assert np.array_equal(ta[key], tb[key], equal_nan=True), key


def test_generator_covers_the_edges():
    pat, lp = R.make_lp(14, 11, 2, 1)
    lens = np.diff(pat.row_ptr)
    assert lens[-1] == 0 and 0.0 >= lp["rl"][-1, 0] and 0.0 <= lp["ru"][-1, 0]          # empty row holding 0
    assert np.bincount(pat.col_idx, minlength=pat.n)[-1] == 0                             # empty column
    assert {l % 4 for l in lens[lens > 0]} >= {1, 2, 3}                                   # spmv tails
    assert np.isinf(lp["lb"][0]).all() and np.isinf(lp["ub"][0]).all()                    # free column
    assert (lp["lb"][1] == lp["ub"][1]).all()                                              # fixed column
    assert np.isinf(lp["ub"][2]).all() and np.isinf(lp["lb"][3]).all()                    # one-sided columns
    assert np.isinf(lp["rl"]).any() and np.isinf(lp["ru"]).any() and (lp["rl"] == lp["ru"]).any()
    r2 = pat.col_idx[pat.row_ptr[2]:pat.row_ptr[3]]
    assert len(r2) != len(set(r2))                                                        # duplicated entry
    tiny = np.abs(lp["vals"][pat.row_of == pat.m - 2]).max()
    assert tiny < 1e-8 * np.abs(lp["vals"]).max()                                         # numerically empty row
