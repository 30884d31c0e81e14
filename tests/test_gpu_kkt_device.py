"""The barrier engine's numeric LDL' kernels on the device (k_sn_diag, k_sn_rows, k_ldl_factor, k_sn_solve, k_ldl_fwd,
k_ldl_diag, k_ldl_bwd), checked lane by lane through asm_kkt_device_selftest against high-precision references.

The LP-level tests cannot see a wrong Newton direction: the barrier method computes its residuals exactly and an
inexact direction only costs Newton steps.  Here every scenario of a batch gets its own matrix values, diagonals and
right-hand side, and each solution is judged on its own:
  * backward error of x in long double: normwise  |b - Mx|_inf / (|M|_inf |x|_inf + |b|_inf)  for well-scaled diagonals,
    componentwise  max_i |b - Mx|_i / (|M||x| + |b|)_i  for end-game diagonals (1e20 and 1e-8 on the diagonal make
    the normwise measure meaningless there), bounded relative to the host mirror asm_kkt_selftest;
  * forward error against scipy's sparse LU, relative to the mirror's own;
  * inertia (n negative, m positive pivots: the matrix is quasi-definite) and log|det| from the device's 1/d.
Scipy and the mirror run on a few lanes (0, 31, 32 and the last): the lanes at the edges of a warp and of blockIdx.y.
Run with -s to see the worst value of every check and the schedule statistics that show which kernel paths ran."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf

pytestmark = pytest.mark.gpu

LD = np.longdouble
STATS = ("nnz_L", "steps", "narrow", "wide", "narrow_split", "wide_multi", "longest_chunk", "capped", "launches_factor",
         "launches_solve")

# bars, calibrated on a B200 (profiles/r04_gpu_kkt_device.txt): each sits at most 10x above the worst value seen there
ETA_WELL = 2e-14          # normwise backward error, well-scaled diagonals
FWD_RATIO = 10.0          # forward error vs scipy <= FWD_RATIO * the mirror's + FWD_ABS
FWD_ABS = 1e-15
ETA_RATIO = 10.0          # end game: componentwise backward error <= ETA_RATIO * the mirror's
LOGDET_REL = 1e-14        # |log|det| - splu| <= LOGDET_REL * max(1, |log|det||), well-scaled diagonals
LOGDET_REL_ENDGAME = 5e-6 # the same in the end game, where pivots of 1e-8 next to 1e20 carry few correct digits


class Kkt:
    """M = [-diag(dx) K'; K diag(ew)] for a batch of scenarios sharing the CSR pattern of K: rows of M in CSR order,
    the values of every scenario gathered from (vals, dx, ew) by one permutation."""

    def __init__(self, K):
        K = sp.csr_matrix(K)
        K.sort_indices()
        self.m, self.n = K.shape
        n, m = self.n, self.m
        self.N = n + m
        self.nnz = K.nnz
        self.rp = K.indptr.astype(np.int64)
        self.ci = K.indices.astype(np.int32)
        ri = np.repeat(np.arange(m), np.diff(K.indptr))
        rows = np.concatenate([np.arange(n), self.ci, n + ri, n + np.arange(m)])
        cols = np.concatenate([np.arange(n), n + ri, self.ci, n + np.arange(m)])
        self.order = np.lexsort((cols, rows))
        self.rows, self.cols = rows[self.order], cols[self.order]
        self.indptr = np.searchsorted(self.rows, np.arange(self.N + 1))

    def data(self, vals, dx, ew):
        return np.concatenate([-dx, vals, vals, ew], axis=1)[:, self.order]

    def matrix(self, d):
        return sp.csr_matrix((d, self.cols, self.indptr), shape=(self.N, self.N))

    def backward_errors(self, data, x, b, chunk=64):
        """(normwise, componentwise) backward error of every row of x, residuals in long double"""
        nw, cw = [], []
        for c0 in range(0, len(x), chunk):
            d = data[c0:c0 + chunk].astype(LD)
            xs, bs = x[c0:c0 + chunk].astype(LD), b[c0:c0 + chunk].astype(LD)
            prod = d * xs[:, self.cols]
            r = np.abs(bs - np.add.reduceat(prod, self.indptr[:-1], axis=1))
            den = np.add.reduceat(np.abs(prod), self.indptr[:-1], axis=1) + np.abs(bs)
            mnorm = np.add.reduceat(np.abs(d), self.indptr[:-1], axis=1).max(axis=1)
            nw.append(r.max(axis=1) / (mnorm * np.abs(xs).max(axis=1) + np.abs(bs).max(axis=1)))
            cw.append(np.where(den > 0, r / np.where(den > 0, den, 1), 0).max(axis=1))
        return np.concatenate(nw).astype(np.float64), np.concatenate(cw).astype(np.float64)

    def residual(self, data, x, b):
        """b - Mx in long double, rounded to float64 (the right-hand side of a refinement step)"""
        prod = data.astype(LD) * x.astype(LD)[:, self.cols]
        return (b.astype(LD) - np.add.reduceat(prod, self.indptr[:-1], axis=1)).astype(np.float64)


def device(lib, kkt, vals, dx, ew, rhs, active=None):
    B = len(rhs)
    sol = np.ascontiguousarray(rhs, dtype=np.float64).copy()
    invp = np.zeros((B, kkt.N))
    stats = np.zeros(10, dtype=np.int64)
    act = None if active is None else np.ascontiguousarray(active, dtype=np.int32)
    rc = lib.asm_kkt_device_selftest(
        kkt.n, kkt.m, kkt.rp.ctypes.data_as(capi.c_int64_p), kkt.ci.ctypes.data_as(capi.c_int32_p), B,
        capi.dptr(np.ascontiguousarray(vals, dtype=np.float64)), capi.dptr(np.ascontiguousarray(dx, dtype=np.float64)),
        capi.dptr(np.ascontiguousarray(ew, dtype=np.float64)),
        None if act is None else act.ctypes.data_as(capi.c_int32_p), capi.dptr(sol), capi.dptr(invp), 0,
        stats.ctypes.data_as(capi.c_int64_p))
    capi.check(rc)
    return sol, invp, dict(zip(STATS, (int(v) for v in stats)))


def mirror(lib, kkt, vals, dx, ew, rhs):
    """asm_kkt_selftest: the host execution of the same lists, one scenario"""
    sol = np.ascontiguousarray(rhs, dtype=np.float64).copy()
    rc = lib.asm_kkt_selftest(kkt.n, kkt.m, kkt.rp.ctypes.data_as(capi.c_int64_p),
                              kkt.ci.ctypes.data_as(capi.c_int32_p), capi.dptr(np.ascontiguousarray(vals)),
                              capi.dptr(np.ascontiguousarray(dx)), capi.dptr(np.ascontiguousarray(ew)), capi.dptr(sol),
                              None)
    capi.check(rc)
    return sol


def ref_lanes(B):
    return sorted({s for s in (0, 31, 32, B - 1) if s < B})


def fwd_err(x, ref):
    return float(np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-300))


def check(lib, name, kkt, vals, dx, ew, rhs, sol, invp, stats, endgame=False, active=None, refine=False):
    """every check of the module on one device run; prints the worst values.  Returns them."""
    B = len(rhs)
    live = np.ones(B, bool) if active is None else np.asarray(active) != 0
    # without pivoting or regularisation an end-game matrix can break down (a pivot cancels to zero): the host mirror
    # does on 5 of the 64 case1354pegase end-game lanes, and rounding decides which ones.  Such lanes are left out
    broken = live & ~(np.isfinite(sol).all(axis=1) & np.isfinite(invp).all(axis=1))
    assert not broken.any() or endgame, (name, np.nonzero(broken)[0])
    assert broken.sum() <= B // 8, (name, broken.sum())
    live &= ~broken
    data = kkt.data(vals, dx, ew)
    nw, cw = kkt.backward_errors(data, sol, rhs)
    worst = {"eta_norm": float(nw[live].max()), "eta_comp": float(cw[live].max()), "broken lanes": int(broken.sum())}
    # inertia, every live lane: n negative and m positive pivots
    neg = (invp[live] < 0).sum(axis=1)
    pos = (invp[live] > 0).sum(axis=1)
    assert np.all(neg == kkt.n) and np.all(pos == kkt.m), (name, neg, pos)
    if not endgame:
        assert worst["eta_norm"] <= ETA_WELL, (name, worst)
    fr, er, lr, rr = [], [], [], []
    for s in ref_lanes(B):
        if not live[s]:
            continue
        M = kkt.matrix(data[s]).tocsc()
        lu = spla.splu(M)
        ref = lu.solve(rhs[s])
        xm = mirror(lib, kkt, vals[s], dx[s], ew[s], rhs[s])
        if not np.isfinite(xm).all():   # the mirror breaks down where the device does not: nothing to compare with
            continue
        f_dev, f_mir = fwd_err(sol[s], ref), fwd_err(xm, ref)
        fr.append(f_dev / (FWD_RATIO * f_mir + FWD_ABS))
        assert f_dev <= FWD_RATIO * f_mir + FWD_ABS, (name, s, f_dev, f_mir)
        logdet = float(np.log(np.abs(lu.U.diagonal())).sum())
        ld_dev = float(-np.log(np.abs(invp[s])).sum())
        lr.append(abs(ld_dev - logdet) / max(1.0, abs(logdet)))
        assert lr[-1] <= (LOGDET_REL_ENDGAME if endgame else LOGDET_REL), (name, s, ld_dev, logdet)
        if endgame:
            _, cm = kkt.backward_errors(data[s:s + 1], xm[None], rhs[s:s + 1])
            er.append(cw[s] / cm[0])
            assert cw[s] <= ETA_RATIO * cm[0], (name, s, cw[s], cm[0])
        if refine:   # one refinement step each, the correction solved by the device entry / by the mirror
            r = kkt.residual(data[s:s + 1], sol[s:s + 1], rhs[s:s + 1])
            c, _, _ = device(lib, kkt, vals[s:s + 1], dx[s:s + 1], ew[s:s + 1], r)
            x2 = sol[s] + c[0]
            rm = kkt.residual(data[s:s + 1], xm[None], rhs[s:s + 1])
            xm2 = xm + mirror(lib, kkt, vals[s], dx[s], ew[s], rm[0])
            _, c2 = kkt.backward_errors(data[s:s + 1], x2[None], rhs[s:s + 1])
            _, cm2 = kkt.backward_errors(data[s:s + 1], xm2[None], rhs[s:s + 1])
            rr.append(c2[0] / cm2[0])
            assert c2[0] <= ETA_RATIO * cm2[0], (name, s, c2[0], cm2[0])
    worst["fwd/bar"] = max(fr, default=0.0)
    worst["logdet_rel"] = max(lr, default=0.0)
    if endgame:
        worst["eta_comp/mirror"] = max(er, default=0.0)
    if refine:
        worst["refined/mirror"] = max(rr, default=0.0)
    print(f"\n[{name}] B {B}: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()) + " | " +
          " ".join(f"{k} {v}" for k, v in stats.items()))
    return worst


# ---- inputs --------------------------------------------------------------------------------------------------------
def draw(kkt, B, seed, endgame=False, base=None):
    """per-scenario values: K entries (scaled copies of `base` when given), diagonals, right-hand sides"""
    rng = np.random.default_rng(seed)
    if base is None:
        vals = rng.standard_normal((B, kkt.nnz))
    else:
        vals = base[None, :] * rng.uniform(0.5, 1.5, (B, kkt.nnz))
    if endgame:
        dx = 10.0 ** rng.uniform(-8, 4, (B, kkt.n))
        ew = 10.0 ** rng.uniform(-8, 4, (B, kkt.m))
        ew[rng.random((B, kkt.m)) < 0.3] = 1e-8
        dx[rng.random((B, kkt.n)) < 0.02] = 1e20
    else:
        dx = 10.0 ** rng.uniform(-2, 2, (B, kkt.n))
        ew = 10.0 ** rng.uniform(-2, 2, (B, kkt.m))
    rhs = rng.standard_normal((B, kkt.N))
    return vals, dx, ew, rhs


def random_pattern(seed):   # the patterns of test_kkt_symbolic.test_random_pattern_against_sparse_lu
    m, n = 40 + 7 * seed, 55 + 3 * seed
    return sp.random(m, n, density=0.08, random_state=seed, format="csr")


def block_structure(seed):   # the patterns of test_kkt_symbolic.test_supernodes_random_structures
    rng = np.random.default_rng(100 + seed)
    blocks = [sp.csr_matrix(rng.standard_normal((int(rng.integers(2, 9)), int(rng.integers(2, 12)))))
              for _ in range(int(rng.integers(2, 6)))]
    K = sp.block_diag(blocks, format="csr")
    m0, n = K.shape
    coupling = sp.random(int(rng.integers(1, 5)), n, density=0.6, random_state=seed, format="csr")
    noise = sp.random(m0, n, density=0.02, random_state=seed + 50, format="csr")
    return sp.vstack([K + noise, coupling], format="csr")


def dense_blocks(ms, extra):
    """block-diagonal dense m x (m + extra) blocks: each is one chain of m + 1 columns along the elimination tree, cut
    into panels of the supernode width from its first column, so a width-w chain's first panel has m + 1 - w rows below
    its diagonal block and the next ones w fewer each"""
    return sp.block_diag([np.ones((m, m + extra)) for m in ms], format="csr")


# narrow (w = 4) first panels with nr = 0, 1, 31, 32, 33, 70 rows below them; wide (w = 16) ones with 0, 1, 15, 16, 17, 40
DENSE_NARROW = [nr + 3 for nr in (0, 1, 31, 32, 33, 70)]
DENSE_WIDE = [nr + 15 for nr in (0, 1, 15, 16, 17, 40)]


def pattern(kind):
    return {"random": lambda: random_pattern(1), "blocks": lambda: block_structure(3),
            "dense_narrow": lambda: dense_blocks(DENSE_NARROW, 2), "dense_wide": lambda: dense_blocks(DENSE_WIDE, 3),
            "dense_57x60": lambda: sp.block_diag([np.ones((57, 60)), np.ones((41, 45))], format="csr")}[kind]()


def acopf_jacobian(case):
    mdl = acopf.AcopfModel(acopf.synthetic_network(*acopf.PEGASE_SHAPES[case]))
    x = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    dE = mdl.eval_jac_g(x, "eval", None, None, np.zeros(mdl.nnz))
    J = sp.coo_matrix((dE, (mdl.j_str[:, 0] - 1, mdl.j_str[:, 1] - 1)), shape=(mdl.m, mdl.n)).tocsr()
    J.sum_duplicates()
    J.sort_indices()
    return J


# ---- 1. supernode widths and panel paths ---------------------------------------------------------------------------
KINDS = ["random", "blocks", "dense_narrow", "dense_wide", "dense_57x60"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("width", ["1", "2", "4", "5", "16"])
def test_widths_and_panel_paths(gpu, monkeypatch, width, kind):
    monkeypatch.setenv("ASM_IPM_SUPERNODE", width)
    kkt = Kkt(pattern(kind))
    vals, dx, ew, rhs = draw(kkt, 40, seed=100 * KINDS.index(kind) + int(width))
    sol, invp, st = device(gpu, kkt, vals, dx, ew, rhs)
    check(gpu, f"width {width} {kind}", kkt, vals, dx, ew, rhs, sol, invp, st)
    w = int(width)
    if w == 1:
        assert st["narrow"] == st["wide"] == 0
    if kind.startswith("dense"):
        if w in (2, 4):
            assert st["narrow"] > 0 and st["narrow_split"] > 0 and st["wide"] == 0, st
        if w in (5, 16):
            assert st["wide"] > 0 and st["wide_multi"] > 0, st
        assert st["longest_chunk"] > 4, st   # chunks longer than one pass of four terms
        if kind != "dense_57x60":
            assert st["longest_chunk"] % 4 != 0, st   # ... and a partial last pass
    if kind == "blocks" and w > 1:
        assert st["narrow"] + st["wide"] > 0, st


# ---- 2. batch shapes -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 2, 31, 32, 33, 64, 65, 100])
def test_batch_shapes(gpu, monkeypatch, B):
    """B = 1 takes the thread-per-item path; 33 and 65 have padding lanes; 64 and up more than one blockIdx.y"""
    monkeypatch.setenv("ASM_IPM_SUPERNODE", "16")
    kkt = Kkt(pattern("dense_narrow"))
    vals, dx, ew, rhs = draw(kkt, B, seed=200 + B)
    sol, invp, st = device(gpu, kkt, vals, dx, ew, rhs)
    assert st["narrow"] > 0 and st["wide"] > 0 and st["wide_multi"] > 0, st
    check(gpu, f"batch {B}", kkt, vals, dx, ew, rhs, sol, invp, st)


# ---- 3. ACOPF Jacobians with end-game diagonals --------------------------------------------------------------------
@pytest.mark.parametrize("case,B", [("case118", 33), ("case1354pegase", 64), ("case1354pegase", 1)])
def test_acopf_endgame(gpu, case, B):
    J = acopf_jacobian(case)
    kkt = Kkt(J)
    vals, dx, ew, rhs = draw(kkt, B, seed=300 + B, endgame=True, base=J.data)
    sol, invp, st = device(gpu, kkt, vals, dx, ew, rhs)
    assert st["narrow"] > 0 and st["wide"] > 0, st
    check(gpu, f"{case} end game", kkt, vals, dx, ew, rhs, sol, invp, st, endgame=True, refine=True)


# ---- 4. grid-stride loops ------------------------------------------------------------------------------------------
def test_grid_stride_loops(gpu):
    """case118 at B = 1024: 32 blockIdx.y rows leave 148 blocks per step, and the widest steps loop"""
    J = acopf_jacobian("case118")
    kkt = Kkt(J)
    vals, dx, ew, rhs = draw(kkt, 1024, seed=400, base=J.data)
    sol, invp, st = device(gpu, kkt, vals, dx, ew, rhs)
    assert st["capped"] > 0, st
    check(gpu, "case118 grid stride", kkt, vals, dx, ew, rhs, sol, invp, st)


# ---- 5. lane independence ------------------------------------------------------------------------------------------
@pytest.fixture
def batch100(monkeypatch):
    monkeypatch.setenv("ASM_IPM_SUPERNODE", "16")
    kkt = Kkt(pattern("dense_narrow"))
    return kkt, draw(kkt, 100, seed=500)


def test_permuted_scenarios_come_back_permuted(gpu, batch100):
    kkt, (vals, dx, ew, rhs) = batch100
    sol, invp, _ = device(gpu, kkt, vals, dx, ew, rhs)
    p = np.random.default_rng(501).permutation(100)
    sol_p, invp_p, _ = device(gpu, kkt, vals[p], dx[p], ew[p], rhs[p])
    assert np.array_equal(sol_p, sol[p]) and np.array_equal(invp_p, invp[p])


def test_masked_lanes(gpu, batch100):
    kkt, (vals, dx, ew, rhs) = batch100
    sol, invp, _ = device(gpu, kkt, vals, dx, ew, rhs)
    active = np.ones(100, np.int32)
    masked = [0, 31, 32, 63, 99]
    active[masked] = 0
    sol_m, invp_m, st = device(gpu, kkt, vals, dx, ew, rhs, active=active)
    assert np.array_equal(sol_m[masked], rhs[masked])
    live = active != 0
    assert np.array_equal(sol_m[live], sol[live]) and np.array_equal(invp_m[live], invp[live])
    check(gpu, "masked", kkt, vals, dx, ew, rhs, sol_m, invp_m, st, active=active)


def test_single_lp_path_agrees_with_the_batch(gpu, batch100):
    kkt, (vals, dx, ew, rhs) = batch100
    sol, _, _ = device(gpu, kkt, vals, dx, ew, rhs)
    k = 57
    one, _, _ = device(gpu, kkt, vals[k:k + 1], dx[k:k + 1], ew[k:k + 1], rhs[k:k + 1])
    ref = spla.splu(kkt.matrix(kkt.data(vals, dx, ew)[k]).tocsc()).solve(rhs[k])
    xm = mirror(gpu, kkt, vals[k], dx[k], ew[k], rhs[k])
    diff = fwd_err(one[0], sol[k])
    print(f"\n[B = 1 vs batch lane {k}] difference {diff:.2e}, bit-identical {np.array_equal(one[0], sol[k])}")
    assert diff <= FWD_RATIO * fwd_err(xm, ref) + FWD_ABS


# ---- 6. reproducibility --------------------------------------------------------------------------------------------
def test_two_calls_give_identical_bits(gpu, batch100):
    kkt, (vals, dx, ew, rhs) = batch100
    a = device(gpu, kkt, vals, dx, ew, rhs)
    b = device(gpu, kkt, vals, dx, ew, rhs)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_pdl_does_not_change_the_bits(gpu, batch100, monkeypatch):
    """a read placed before pdl_wait() would see the previous step's data only with programmatic dependent launches"""
    kkt, (vals, dx, ew, rhs) = batch100
    a = device(gpu, kkt, vals, dx, ew, rhs)
    monkeypatch.setenv("ASM_NO_PDL", "1")
    b = device(gpu, kkt, vals, dx, ew, rhs)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- 7. edges ------------------------------------------------------------------------------------------------------
EDGES = {
    "no rows": sp.csr_matrix((0, 5)),
    "empty rows and columns": sp.csr_matrix(np.array([[1.0, 0.0, 2.0, 0.0], [0.0, 0.0, 0.0, 0.0],
                                                      [0.0, 0.0, -1.0, 0.0]])),
    "one column": sp.csr_matrix(np.ones((3, 1))),
    "one dense row": sp.vstack([sp.csr_matrix(np.ones((1, 40))), sp.random(12, 40, density=0.1, random_state=9)],
                               format="csr"),
}


@pytest.mark.parametrize("edge", list(EDGES))
@pytest.mark.parametrize("B", [1, 33])
def test_edges(gpu, edge, B):
    kkt = Kkt(EDGES[edge])
    vals, dx, ew, rhs = draw(kkt, B, seed=700 + B)
    sol, invp, st = device(gpu, kkt, vals, dx, ew, rhs)
    check(gpu, f"edge {edge}", kkt, vals, dx, ew, rhs, sol, invp, st)
