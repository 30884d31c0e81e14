"""Host-only checks of the barrier engine's symbolic analysis (csrc/kkt_symbolic.hpp) through asm_kkt_selftest: the
fill-reducing ordering, the pattern of L, the level schedule and the chunked fan-out term lists are exercised by
factorising a quasi-definite KKT matrix and solving one system ON THE HOST with exactly the lists and the summation
order the device kernels use; the answer is compared with scipy's sparse LU.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf, small_nlps


def _selftest(lib, K, dx, ew, rhs):
    K = sp.csr_matrix(K)
    K.sort_indices()
    m, n = K.shape
    rp = K.indptr.astype(np.int64)
    ci = K.indices.astype(np.int32)
    vals = np.ascontiguousarray(K.data, dtype=np.float64)
    sol = np.ascontiguousarray(rhs, dtype=np.float64).copy()
    stats = np.zeros(8, dtype=np.int64)
    rc = lib.asm_kkt_selftest(n, m, rp.ctypes.data_as(capi.c_int64_p), ci.ctypes.data_as(capi.c_int32_p),
                              capi.dptr(vals), capi.dptr(np.ascontiguousarray(dx, dtype=np.float64)),
                              capi.dptr(np.ascontiguousarray(ew, dtype=np.float64)), capi.dptr(sol),
                              stats.ctypes.data_as(capi.c_int64_p))
    capi.check(rc)
    return sol, dict(zip(("nnz_L", "terms", "levels", "f_steps", "w_steps", "b_steps", "longest_chunk", "chunks"),
                         (int(v) for v in stats)))


def _kkt(K, dx, ew):
    return sp.bmat([[-sp.diags(dx), K.T], [K, sp.diags(ew)]], format="csc")


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_pattern_against_sparse_lu(built_lib, seed):
    rng = np.random.default_rng(seed)
    m, n = 40 + 7 * seed, 55 + 3 * seed
    K = sp.random(m, n, density=0.08, random_state=seed, format="csr")
    K.data[:] = rng.standard_normal(K.nnz)
    dx = 10.0 ** rng.uniform(-6, 3, n)
    ew = 10.0 ** rng.uniform(-6, 3, m)
    rhs = rng.standard_normal(n + m)
    sol, st = _selftest(built_lib, K, dx, ew, rhs)
    ref = spla.spsolve(_kkt(K, dx, ew), rhs)
    assert np.linalg.norm(sol - ref) <= 1e-8 * np.linalg.norm(ref)
    assert st["nnz_L"] >= K.nnz and st["levels"] >= 1 and st["terms"] >= st["chunks"] >= 0


def test_empty_rows_and_columns(built_lib):
    """Rows / columns without entries are isolated nodes of the KKT graph: their pivots are the diagonal itself."""
    K = sp.csr_matrix(np.array([[1.0, 0.0, 2.0, 0.0], [0.0, 0.0, 0.0, 0.0], [0.0, 0.0, -1.0, 0.0]]))
    dx = np.array([1.0, 2.0, 3.0, 4.0])
    ew = np.array([0.5, 0.25, 2.0])
    rhs = np.arange(1.0, 8.0)
    sol, st = _selftest(built_lib, K, dx, ew, rhs)
    ref = spla.spsolve(_kkt(K, dx, ew), rhs)
    assert np.allclose(sol, ref, rtol=1e-12, atol=1e-12)


def test_acopf_kkt_with_barrier_like_diagonals(built_lib):
    """case118-sized ACOPF Jacobian, diagonals spread over 12 orders of magnitude as in the last Newton steps; one step
    of iterative refinement (what the engine does) brings the residual to round-off."""
    mdl = acopf.AcopfModel(acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"]))
    x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    dE = mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz))
    J = sp.coo_matrix((dE, (mdl.j_str[:, 0] - 1, mdl.j_str[:, 1] - 1)), shape=(mdl.m, mdl.n)).tocsr()
    J.sum_duplicates()
    rng = np.random.default_rng(5)
    dx = 10.0 ** rng.uniform(-8, 4, mdl.n)
    ew = 10.0 ** rng.uniform(-8, 4, mdl.m)
    rhs = rng.standard_normal(mdl.n + mdl.m)
    M = _kkt(J, dx, ew)
    sol, st = _selftest(built_lib, J, dx, ew, rhs)
    r = rhs - M @ sol
    corr, _ = _selftest(built_lib, J, dx, ew, r)
    sol2 = sol + corr
    assert np.linalg.norm(rhs - M @ sol2) <= 1e-10 * np.linalg.norm(rhs)
    # the fan-out schedule keeps the critical path of a step short: no chunk is longer than a few dozen terms
    assert st["longest_chunk"] <= 64
    assert st["nnz_L"] < 6 * J.nnz          # minimum degree keeps the fill small on network matrices


def test_toy_pattern(built_lib):
    pr = small_nlps.ToyNlp()
    J = sp.coo_matrix((np.arange(1.0, 7.0), (pr.j_str[:, 0] - 1, pr.j_str[:, 1] - 1)), shape=(pr.m, pr.n)).tocsr()
    dx = np.array([1e-8, 1e-8])
    ew = np.array([1.0, 1e-8, 1e-8, 3.0])
    rhs = np.array([1.0, -1.0, 0.5, 0.25, -2.0, 1.0])
    M = _kkt(J, dx, ew)
    sol, _ = _selftest(built_lib, J, dx, ew, rhs)
    ref = spla.spsolve(M, rhs)
    assert np.allclose(sol, ref, rtol=1e-5)        # pivots of 1e-8 without pivoting: seven digits ...
    for _ in range(2):                             # ... and the engine's two refinement passes recover the rest
        corr, _ = _selftest(built_lib, J, dx, ew, rhs - M @ sol)
        sol = sol + corr
    assert np.allclose(sol, ref, rtol=1e-10)


@pytest.mark.parametrize("width", ["1", "4", "16"])
def test_supernodes_dense_block(built_lib, monkeypatch, width):
    """A dense K makes the whole elimination tree one chain: with supernodes it is cut into panels of at most `width`
    columns (diagonal block + rows below, k_sn_factor / k_sn_solve on the device), each updating the next through the
    chunked term lists.  Same answer as without (width 1) and as scipy."""
    monkeypatch.setenv("ASM_IPM_SUPERNODE", width)
    rng = np.random.default_rng(11)
    m, n = 23, 31
    K = sp.csr_matrix(rng.standard_normal((m, n)))
    dx = 10.0 ** rng.uniform(-3, 3, n)
    ew = 10.0 ** rng.uniform(-3, 3, m)
    rhs = rng.standard_normal(n + m)
    sol, st = _selftest(built_lib, K, dx, ew, rhs)
    ref = spla.spsolve(_kkt(K, dx, ew), rhs)
    assert np.linalg.norm(sol - ref) <= 1e-9 * np.linalg.norm(ref)
    # the n column nodes are independent (level 0); the first of them and the m row nodes form one chain of m + 1
    # columns with nested patterns: a level each without supernodes, ceil((m + 1) / width) steps with them
    chain = m + 1
    assert st["levels"] == {"1": chain, "4": 1 + -(-chain // 4), "16": 1 + -(-chain // 16)}[width]


def test_supernodes_shorten_the_schedule(built_lib, monkeypatch):
    """case118-sized ACOPF KKT: the supernodal schedule has several times fewer steps and target updates, and the host
    mirror of the device numerics gives the same solution."""
    mdl = acopf.AcopfModel(acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"]))
    x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    dE = mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz))
    J = sp.coo_matrix((dE, (mdl.j_str[:, 0] - 1, mdl.j_str[:, 1] - 1)), shape=(mdl.m, mdl.n)).tocsr()
    J.sum_duplicates()
    rng = np.random.default_rng(7)
    dx = 10.0 ** rng.uniform(-2, 2, mdl.n)
    ew = 10.0 ** rng.uniform(-2, 2, mdl.m)
    rhs = rng.standard_normal(mdl.n + mdl.m)
    out = {}
    for width in ("1", "16"):
        monkeypatch.setenv("ASM_IPM_SUPERNODE", width)
        out[width] = _selftest(built_lib, J, dx, ew, rhs)
    (s1, st1), (s16, st16) = out["1"], out["16"]
    assert np.linalg.norm(s1 - s16) <= 1e-10 * np.linalg.norm(s1)
    assert st16["levels"] * 2 < st1["levels"]
    assert st16["chunks"] * 2 < st1["chunks"]
    assert st16["nnz_L"] == st1["nnz_L"]


@pytest.mark.parametrize("seed", range(8))
def test_supernodes_random_structures(built_lib, monkeypatch, seed):
    """Patterns that produce supernodes of every width, wide panels with and without rows below them, chains longer
    than one supernode and columns with several rows in one supernode (chunks in the backward substitution): block
    diagonal dense blocks coupled by a few dense rows, plus random sparse noise.  Every width gives scipy's answer."""
    rng = np.random.default_rng(100 + seed)
    blocks = [sp.csr_matrix(rng.standard_normal((int(rng.integers(2, 9)), int(rng.integers(2, 12)))))
              for _ in range(int(rng.integers(2, 6)))]
    K = sp.block_diag(blocks, format="csr")
    m0, n = K.shape
    coupling = sp.random(int(rng.integers(1, 5)), n, density=0.6, random_state=seed, format="csr")
    noise = sp.random(m0, n, density=0.02, random_state=seed + 50, format="csr")
    K = sp.vstack([K + noise, coupling], format="csr")
    K.data[:] = rng.standard_normal(K.nnz)
    m = K.shape[0]
    dx = 10.0 ** rng.uniform(-4, 2, n)
    ew = 10.0 ** rng.uniform(-4, 2, m)
    ew[rng.random(m) < 0.3] = 1e-8            # equality rows: only the regularisation on the diagonal
    rhs = rng.standard_normal(n + m)
    ref = spla.spsolve(_kkt(K, dx, ew), rhs)
    levels = {}
    for width in ("1", "2", "5", "16"):
        monkeypatch.setenv("ASM_IPM_SUPERNODE", width)
        sol, st = _selftest(built_lib, K, dx, ew, rhs)
        assert np.linalg.norm(sol - ref) <= 1e-7 * np.linalg.norm(ref), width
        levels[width] = st["levels"]
    # a supernode never starts later than the level of its last column: steps <= levels for every width
    assert max(levels["2"], levels["5"], levels["16"]) <= levels["1"]


def test_host_threads_do_not_change_the_lists(built_lib, monkeypatch):
    """The symbolic analysis builds its lists on several host threads; every thread writes to positions fixed
    beforehand, so the numeric result is bit-identical for any thread count."""
    mdl = acopf.AcopfModel(acopf.synthetic_network(*acopf.PEGASE_SHAPES["case118"]))
    x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    dE = mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz))
    J = sp.coo_matrix((dE, (mdl.j_str[:, 0] - 1, mdl.j_str[:, 1] - 1)), shape=(mdl.m, mdl.n)).tocsr()
    J.sum_duplicates()
    rng = np.random.default_rng(3)
    dx = 10.0 ** rng.uniform(-6, 2, mdl.n)
    ew = 10.0 ** rng.uniform(-6, 2, mdl.m)
    rhs = rng.standard_normal(mdl.n + mdl.m)
    out = []
    for threads in ("1", "2", "7"):
        monkeypatch.setenv("ASM_HOST_THREADS", threads)
        out.append(_selftest(built_lib, J, dx, ew, rhs))
    for sol, st in out[1:]:
        assert np.array_equal(sol, out[0][0])
        assert st == out[0][1]
