"""The SLP layer's device kernels, lane by lane at full batch width, against exact and long-double references.

Nothing downstream notices an error in these kernels: a wrong bound built by k_slp_cols / k_slp_rows / k_fr_rows /
k_fr_vals is a different LP that the engine solves correctly, k_extract's output goes straight to the driver, and the
reductions (k_viol, k_kt, k_row_norms, k_compl, k_merit, k_dot, k_final) and the ACOPF evaluator (k_acopf_*) decide
termination, step acceptance and nu.  So every output is checked here for every lane, at the batch widths and sizes
where the launch geometry of util.cuh (geo_for, pad_batch, restated below and asserted per shape) takes its capped,
grid-stride and multi-block paths:
  * LP data, both phases, bit-exact (==, and the signbit of the step bounds) against a vectorised restatement of
    oracle.SubLp.build, which is itself compared with SubLp.build on the lanes at the edges of a warp and of blockIdx.y;
  * the read-back, bit-exact against a restatement of k_extract on the raw LP solution of asm_slp_get_lp, with masked
    lanes; and each raw solution primal-feasible for its own lane's LP data;
  * norm_violations (p = inf bit-exact), kt_residuals, norm_complementarity, row_norms, merit_phi, merit_derivative and
    acopf_trial against long double (np.longdouble, 64-bit mantissa on x86-64);
  * the ACOPF evaluator, f, df, E and dE in j_str order, against a long-double restatement of its formulas;
  * lane independence: a permutation of the scenarios permutes the outputs bit for bit, a repeated call is
    bit-identical, and shared bounds passed as per-scenario arrays give the shared-bounds results bit for bit.

Rounding-error bars are a priori, not calibrated.  With u = 2^-53, an output that the device sums as
S = sum_i t_i obeys, to first order,
    |S_device - S| <= (k + d) u sum_i |t_i|,
k = the roundings inside one term t_i (nvcc contracts a*b + c into an FMA by default, so a product that feeds a sum
costs no rounding of its own and is still counted once here), d = the longest addition chain of the reduction:
ceil(count / (grid.x * rows per block)) per thread (rows per block: 256 for one LP, 8 warps for a batch), then the
block's combine (5 shuffle levels for one LP, then 8 warps), then ceil(nbx / 128) per thread of final_reduce and its
7 tree levels.  The bar goes through a final sqrt as half the relative error plus one rounding, and through a division
as the sum of relative errors plus one rounding.  Evaluator entries get a per-entry bar from the magnitudes of their
terms: 10 u of the magnitude covers the products and sums of one Ohm row or Jacobian entry, including sincos's error;
CUDA 12.9's Programming Guide lists double sincos at 2 ulp (full range), i.e. 4 u relative.  In trial mode every
variable x + alpha p carries u (|x + alpha p| + |alpha p|) (one rounding, or two without an FMA), propagated through
the entry's partial derivatives; va_f - va_t uses absolute terms.  The long-double references carry their own error
(2^-64 per operation, pairwise sums), added to each bar.  Any dropped or misplaced term larger than its bar fails.
Run with -s to see the worst err/bar of every check and the geometry each shape reaches."""
import math
import time

import numpy as np
import pytest
import scipy.sparse as sp

from activesetmethods_b200 import capi
from activesetmethods_b200.examples import acopf
from oracle import slp_oracle as so
from test_oracle_pins import case3_network

pytestmark = pytest.mark.gpu

LD = np.longdouble
U = 2.0 ** -53
U_LD = float(np.finfo(LD).eps) / 2
ETA = 2.0 ** -1074          # smallest subnormal: an underflowing product or square is off by at most this much
THREADS, WARPS, MAX_BX, FINAL_THREADS = 256, 8, 148 * 8, 128
EQ, RANGE, LOWER, UPPER = 0, 1, 2, 3
SKIPPED = 5
WORST = {}


# ---- launch geometry of util.cuh ----------------------------------------------------------------------------
def pad_batch(b):
    return 1 if b <= 1 else (32 if b <= 32 else (b + 63) // 64 * 64)


def geo_for(count, B):
    """(grid.x, grid.y, items per block per sweep)"""
    if B == 1:
        return max(1, min(-(-count // THREADS), MAX_BX)), 1, THREADS
    gy = B // 32
    cap = max(1, min(MAX_BX * 2 // gy, MAX_BX))
    return max(1, min(-(-count // WARPS), cap)), gy, WARPS


def per_thread(count, B):
    gx, _, rpb = geo_for(count, B)
    return -(-max(count, 0) // (gx * rpb))


def chain(per, B, nbx):
    """longest addition chain of block_reduce_store + final_reduce after `per` items of one thread"""
    return per + (5 if B == 1 else 0) + WARPS + -(-nbx // FINAL_THREADS) + 7


def note(name, ratio):
    ratio = float(ratio)
    WORST[name] = max(WORST.get(name, 0.0), ratio)


def check_bar(name, got, ref, bar):
    got = np.asarray(got, dtype=LD)
    ref = np.asarray(ref, dtype=LD)
    bar = np.asarray(bar, dtype=LD) + U_LD * 64 * np.abs(ref) + 1e6 * ETA
    err = np.abs(got - ref)
    assert np.all(np.isfinite(got) == np.isfinite(ref)), name
    fin = np.isfinite(ref)
    assert np.all(got[~fin] == ref[~fin]), name
    err, bar = err[fin], np.broadcast_to(bar, ref.shape)[fin]
    bad = err > bar
    ratio = np.where(bar > 0, err / np.where(bar > 0, bar, 1), np.where(err > 0, np.inf, 0))
    note(name, ratio.max(initial=0.0))
    assert not bad.any(), (name, np.flatnonzero(bad)[:5], err[bad][:5], bar[bad][:5])


def bit_equal(name, got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    same = (got == ref) | (np.isnan(got) & np.isnan(ref)) if got.dtype.kind == "f" else got == ref
    assert same.all(), (name, np.argwhere(~same)[:5], got[~same][:5], ref[~same][:5])
    note(name + " (bit-exact: 0 = equal)", 0.0)


def report(tag, t0):
    print(f"\n[{tag}] {time.time() - t0:.1f} s")
    for k in sorted(WORST):
        print(f"    {k:58s} worst err/bar {WORST[k]:.3g}")
    WORST.clear()


# ---- problems ---------------------------------------------------------------------------------------------------
class Nlp:
    def __init__(self, name, n, m, j_str, x_L, x_U, g_L, g_U, model=None):
        self.name, self.n, self.m, self.model = name, n, m, model
        self.j_str = np.asarray(j_str, dtype=np.int64).reshape(-1, 2)
        self.x_L, self.x_U, self.g_L, self.g_U = (np.asarray(a, dtype=float) for a in (x_L, x_U, g_L, g_U))


def make_nlp(name):
    if name in ("case9", "case3", "case118", "case1354"):
        net = {"case9": acopf.case9, "case3": case3_network}.get(name)
        net = net() if net else acopf.synthetic_network(*acopf.PEGASE_SHAPES["case1354pegase" if name == "case1354"
                                                                               else name])
        mdl = acopf.AcopfModel(net)
        return Nlp(name, mdl.n, mdl.m, mdl.j_str, mdl.x_L, mdl.x_U, mdl.g_L, mdl.g_U, mdl)
    if name == "banded":
        # one band per row plus a duplicate of every third diagonal entry: nnz_coo > 1184 * 256 = 303 104, so the
        # single-LP grid is capped and every Map<false> loop takes a second sweep
        n = m = 320_000
        i = np.arange(m)
        dup = i[::3]
        j = np.concatenate([np.stack([i, i], 1), np.stack([i, (i + 1) % n], 1), np.stack([dup, dup], 1)]) + 1
        return Nlp(name, n, m, j, *four_class_bounds(n, m))
    if name == "m0":
        return Nlp(name, 3, 0, np.zeros((0, 2)), [-1.0, -np.inf, 0.0], [1.0, 2.0, np.inf], [], [])
    if name == "one":
        return Nlp(name, 1, 1, [[1, 1], [1, 1]], [-1.0], [2.0], [-0.5], [0.75])
    if name == "classes":
        j = [[1, 1], [1, 2], [2, 2], [2, 3], [3, 3], [3, 4], [4, 4], [4, 1], [2, 2], [1, 1]]
        return Nlp(name, 4, 4, j, *four_class_bounds(4, 4))
    raise KeyError(name)


def four_class_bounds(n, m):
    """rows cycle through ==, range, >=, <=; columns through finite, lower only, upper only, free"""
    k = np.arange(m) % 4
    gl = np.where(k == 0, 0.25, np.where(k == 1, -1.0, np.where(k == 2, -0.5, -np.inf)))
    gu = np.where(k == 0, 0.25, np.where(k == 1, 1.5, np.where(k == 2, np.inf, 0.5)))
    c = np.arange(n) % 4
    xl = np.where(c == 0, -1.0, np.where(c == 1, -2.0, -np.inf))
    xu = np.where(c == 0, 1.0, np.where(c == 2, 3.0, np.inf))
    return xl, xu, gl, gu


def lane_bounds(nlp, B, per):
    """[B, n] / [B, m] bounds; per-scenario ones differ per lane and keep every row class"""
    xl, xu, gl, gu = (np.broadcast_to(a, (B, len(a))).copy() for a in (nlp.x_L, nlp.x_U, nlp.g_L, nlp.g_U))
    if not per:
        return xl, xu, gl, gu
    fac = 1.0 + 0.02 * ((np.arange(B) * 7919) % 13 - 6) / 6.0
    xl, xu = xl * fac[:, None], xu * fac[:, None]          # +-inf stay, finite bounds scale, order kept
    if nlp.model is not None:
        mdl = nlp.model
        r = mdl.r_bal
        for s in range(B):
            net = acopf.perturb_loads(mdl.net, s + 1)
            gl[s, r:r + 2 * mdl.nb:2] = gu[s, r:r + 2 * mdl.nb:2] = -net.pd
            gl[s, r + 1:r + 2 * mdl.nb:2] = gu[s, r + 1:r + 2 * mdl.nb:2] = -net.qd
    else:
        gl, gu = gl * fac[:, None], gu * fac[:, None]
    return xl, xu, gl, gu


def pick(lo, hi, rng):
    """values strictly inside, exactly on, 1 ulp outside and far outside [lo, hi] (componentwise, per lane)"""
    shape = lo.shape
    r = rng.random(shape)
    with np.errstate(invalid="ignore"):
        inside = np.where(np.isfinite(lo) & np.isfinite(hi), lo + (hi - lo) * (0.05 + 0.9 * r),
                          np.where(np.isfinite(lo), lo + r + 0.01, np.where(np.isfinite(hi), hi - r - 0.01, 2 * r - 1)))
    mode = rng.integers(0, 7, shape)
    v = inside.copy()
    lf, hf = np.isfinite(lo), np.isfinite(hi)
    v = np.where((mode == 1) & lf, lo, v)
    v = np.where((mode == 2) & hf, hi, v)
    v = np.where((mode == 3) & lf, np.nextafter(lo, -np.inf), v)
    v = np.where((mode == 4) & hf, np.nextafter(hi, np.inf), v)
    v = np.where((mode == 5) & lf, lo - 10.0 * (1.0 + np.abs(np.where(lf, lo, 0))), v)
    v = np.where((mode == 6) & hf, hi + 10.0 * (1.0 + np.abs(np.where(hf, hi, 0))), v)
    return v


DELTAS = np.array([1000.0, 1e-6, 0.0, 5e-324])


def adversarial_inputs(nlp, bounds, B, rng):
    xl, xu, gl, gu = bounds
    n, m, nz = nlp.n, nlp.m, len(nlp.j_str)
    x = pick(xl, xu, rng)
    E = pick(gl, gu, rng)
    df = rng.standard_normal((B, n))
    df[rng.random((B, n)) < 0.2] = 0.0
    dE = rng.standard_normal((B, nz)) * 10.0 ** rng.integers(-3, 4, (B, nz))
    z = rng.random((B, nz))
    dE[z < 0.1] = 0.0
    dE[(z >= 0.1) & (z < 0.2)] = -0.0
    return dict(x=x, f=rng.standard_normal(B), df=df, E=E, dE=dE, delta=DELTAS[np.arange(B) % 4])


# ---- restatement of the handle's LP data (oracle.SubLp.build, device layout) ------------------------------------
class Layout:
    """row classes, slack columns, range rows and the restoration pattern, as SlpHandle::create / build_fr lay them
    out (the reference layout of asm_slp_sizes)"""

    def __init__(self, nlp):
        n, m = nlp.n, nlp.m
        gl, gu = nlp.g_L, nlp.g_U
        self.n, self.m = n, m
        self.pat = so.JacobianPattern(m, n, nlp.j_str)
        self.cls = np.where(gl == gu, EQ, np.where(np.isfinite(gl) & np.isfinite(gu), RANGE,
                                                   np.where(np.isfinite(gl), LOWER, UPPER))).astype(np.int64)
        two = (self.cls == EQ) | (self.cls == RANGE)
        nsl = 1 + two
        self.s1 = n + np.concatenate([[0], np.cumsum(nsl)[:-1]]).astype(np.int64) if m else np.zeros(0, np.int64)
        self.s2 = np.where(two, self.s1 + 1, -1)
        self.adj = np.flatnonzero(self.cls == RANGE)
        self.ncol_fr, self.nrow_fr = n + int(nsl.sum()), m + len(self.adj)
        rp = self.pat.row_ptr
        rowlen = np.diff(rp)
        self.rowlen = rowlen
        self.collen = np.bincount(self.pat.cols, minlength=n)
        # restoration CSR: row i = J row i, +s1 (-s1 for <= rows), -s2 for == rows; extra row a = J row adj[a], -s2
        jrow = np.repeat(np.arange(m), rowlen)
        seq = np.arange(self.pat.nnz) - rp[jrow]
        ea = np.repeat(np.arange(len(self.adj)), rowlen[self.adj])
        ek = np.concatenate([np.arange(rp[i], rp[i + 1]) for i in self.adj]) if len(self.adj) else np.zeros(0, int)
        eq = np.flatnonzero(self.cls == EQ)
        rows = np.concatenate([jrow, np.arange(m), eq, m + ea, m + np.arange(len(self.adj))])
        seqs = np.concatenate([seq, rowlen, rowlen[eq] + 1, ek - rp[self.adj][ea] if len(ek) else ek,
                               rowlen[self.adj]])
        cols = np.concatenate([self.pat.cols, self.s1, self.s2[eq], self.pat.cols[ek], self.s2[self.adj]])
        src = np.concatenate([np.arange(self.pat.nnz), np.where(self.cls == UPPER, -2, -1), np.full(len(eq), -2),
                              ek, np.full(len(self.adj), -2)])
        o = np.lexsort((seqs, rows))
        self.fr_cols, self.fr_src = cols[o].astype(np.int32), src[o]
        self.fr_rp = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=self.nrow_fr))]).astype(np.int64)

    def assemble(self, dE):
        """compute_jacobian_matrix for every lane: ((0.0 + v1) + v2) + ... in j_str order"""
        J = np.zeros((len(dE), self.pat.nnz))
        for r in range(self.pat.max_rank + 1):
            sel = self.pat.rank == r
            J[:, self.pat.slot[sel]] = J[:, self.pat.slot[sel]] + dE[:, sel]
        return J

    def lp_data(self, inp, bounds, fr):
        """the raw LP arrays of every lane, in the device's layout"""
        xl, xu, gl, gu = bounds
        n, m = self.n, self.m
        x, E, delta = inp["x"], inp["E"], inp["delta"][:, None]
        J = self.assemble(inp["dE"])
        plb = np.maximum(-delta, xl - x)
        pub = np.minimum(delta, xu - x)
        plb = np.where(plb == 0.0, 0.0, plb)                 # tol_error = 0 only normalises -0.0
        pub = np.where(pub == 0.0, 0.0, pub)
        cls = self.cls
        if not fr:
            lo, up = gl - E, gu - E
            return dict(vals=J, c=inp["df"].copy(), c0=inp["f"].copy(), lb=plb, ub=pub,
                        rl=np.where(cls == UPPER, -np.inf, lo),
                        ru=np.where(cls == EQ, lo, np.where(cls == LOWER, np.inf, up)))
        B = len(x)
        viol = np.where(E > gu, gu - E, np.where(E < gl, gl - E, 0.0))
        bs = E - np.abs(viol)
        lo, up = gl - bs, gu - bs
        rl = np.concatenate([np.where(cls == UPPER, -np.inf, lo), np.full((B, len(self.adj)), -np.inf)], 1)
        ru = np.concatenate([np.where(cls == EQ, lo, np.where(cls == UPPER, up, np.inf)), up[:, self.adj]], 1)
        lb = np.zeros((B, self.ncol_fr))
        ub = np.full((B, self.ncol_fr), np.inf)
        lb[:, :n], ub[:, :n] = plb, pub
        two = self.s2 >= 0
        neg = viol < 0
        # the device snaps -viol = -0.0 to +0.0 (pos_zero); the oracle keeps -0.0 there
        lb[:, self.s1] = np.where(two, np.where(neg, 0.0, np.where(viol == 0, 0.0, -viol)),
                                  np.where(viol == 0, 0.0, -np.abs(viol)))
        t = np.flatnonzero(two)
        lb[:, self.s2[t]] = np.where(neg[:, t], viol[:, t], 0.0)
        c = np.zeros((B, self.ncol_fr))
        c[:, n:] = 1.0
        src = self.fr_src
        vals = np.where(src >= 0, J[:, np.maximum(src, 0)], np.where(src == -1, 1.0, -1.0))
        return dict(vals=vals, c=c, c0=np.zeros(B), lb=lb, ub=ub, rl=rl, ru=ru)


def oracle_pin(lay, nlp, inp, bounds, fr, dev, s):
    """the restatement's lane s against oracle.SubLp.build itself"""
    xl, xu, gl, gu = (b[s] for b in bounds)
    ref = so.SubLp(lay.pat, gl, gu, xl, xu, engine=object())
    vals = lay.pat.assemble(inp["dE"][s])
    K, cost, off, lb, ub, rl, ru = ref.build(vals, inp["df"][s], inp["f"][s], inp["E"][s], inp["x"][s],
                                             inp["delta"][s], fr)
    n, m = lay.n, lay.m
    bit_equal("pin: p-column lb", dev["lb"][:n], lb[:n])
    bit_equal("pin: p-column ub", dev["ub"][:n], ub[:n])
    bit_equal("pin: p-column bound signbits", np.signbit(np.r_[dev["lb"][:n], dev["ub"][:n]]),
              np.signbit(np.r_[lb[:n], ub[:n]]))
    if not fr:
        Kd = sp.csr_matrix((dev["vals"], lay.pat.cols, lay.pat.row_ptr), shape=(m, n))
        assert (Kd - K[:m, :n]).count_nonzero() == 0
        bit_equal("pin: objective", dev["c"], cost[:n])
        assert dev["c0"] == off
        bit_equal("pin: rl", dev["rl"], rl[:m])
        # range rows are two-sided on the device, the oracle's row plus its extra <= row
        ru_o = ru[:m].copy()
        ru_o[lay.adj] = ru[m:]
        bit_equal("pin: ru", dev["ru"], ru_o)
        return
    Kd = sp.csr_matrix((dev["vals"], lay.fr_cols, lay.fr_rp), shape=K.shape)
    # scipy's sparse + in build() drops exact zeros: compare as (row, col) -> value maps, absent = 0.0
    assert (Kd - K).count_nonzero() == 0
    for key, o in (("lb", lb), ("ub", ub), ("rl", rl), ("ru", ru)):
        bit_equal("pin: restoration " + key, dev[key], o)
    bit_equal("pin: restoration objective", dev["c"], cost)
    zero = dev["lb"][n:] == 0                        # slack bounds: +0.0 on the device (oracle: -0.0 where viol = 0)
    assert not np.signbit(dev["lb"][n:][zero]).any()


# ---- the C ABI ----------------------------------------------------------------------------------------------------
def new_handle(nlp, bounds, B, per, **kw):
    from activesetmethods_b200.sublp import SubLp
    xl, xu, gl, gu = bounds if per else (nlp.x_L, nlp.x_U, nlp.g_L, nlp.g_U)
    lp = SubLp(nlp.n, nlp.m, nlp.j_str, xl, xu, gl, gu, batch=B, **kw)
    lp._squeeze = False
    return lp


def get_lp(lp, s, solution):
    lib, h = lp._lib, lp._h
    cols, rows, st = np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int32)
    nnz = np.zeros(1, np.int64)
    i32, i64, d = capi.c_int32_p, capi.c_int64_p, capi.dptr
    capi.check(lib.asm_slp_get_lp(h, s, cols.ctypes.data_as(i32), rows.ctypes.data_as(i32), nnz.ctypes.data_as(i64),
                                  *[None] * 14))
    nc, nr, nz = int(cols[0]), int(rows[0]), int(nnz[0])
    o = dict(row_ptr=np.zeros(nr + 1, np.int64), col_idx=np.zeros(nz, np.int32), vals=np.zeros(nz), c=np.zeros(nc),
             c0=np.zeros(1), lb=np.zeros(nc), ub=np.zeros(nc), rl=np.zeros(nr), ru=np.zeros(nr))
    if solution:
        o.update(x=np.zeros(nc), y=np.zeros(nr), dual_lb=np.zeros(nc), dual_ub=np.zeros(nc))
    g = lambda k: d(o[k]) if k in o else None   # noqa: E731
    capi.check(lib.asm_slp_get_lp(h, s, None, None, None, o["row_ptr"].ctypes.data_as(i64),
                                  o["col_idx"].ctypes.data_as(i32), g("vals"), g("c"), g("c0"), g("lb"), g("ub"),
                                  g("rl"), g("ru"), g("x"), g("y"), g("dual_lb"), g("dual_ub"),
                                  st.ctypes.data_as(i32) if solution else None))
    o["c0"] = o["c0"][0]
    o["status"] = int(st[0])
    return o


def read_lanes(lp, B, solution):
    out = [get_lp(lp, s, solution) for s in range(B)]
    return {k: np.array([o[k] for o in out]) for k in out[0]}


def check_lp_data(name, lay, nlp, inp, bounds, fr, dev):
    B = len(inp["x"])
    ref = lay.lp_data(inp, bounds, fr)
    if fr:
        bit_equal(name + " restoration row_ptr", dev["row_ptr"][0], lay.fr_rp)
        bit_equal(name + " restoration col_idx", dev["col_idx"][0], lay.fr_cols)
    else:
        bit_equal(name + " normal row_ptr", dev["row_ptr"][0], lay.pat.row_ptr)
        bit_equal(name + " normal col_idx", dev["col_idx"][0], lay.pat.cols.astype(np.int32))
    for k in ("vals", "c", "c0", "lb", "ub", "rl", "ru"):
        bit_equal(f"{name} LP {k} ({'restoration' if fr else 'normal'})", dev[k], ref[k])
    n = lay.n
    assert not np.signbit(dev["lb"][:, :n][dev["lb"][:, :n] == 0]).any()
    assert not np.signbit(dev["ub"][:, :n][dev["ub"][:, :n] == 0]).any()
    for s in sorted({0, 31, 32, 33, 63, 64, B - 1} & set(range(B))):
        oracle_pin(lay, nlp, inp, bounds, fr, {k: v[s] for k, v in dev.items()}, s)


# ---- long-double references of the reductions ------------------------------------------------------------------
def chunks(B, size=64):
    return [slice(a, min(a + size, B)) for a in range(0, B, size)]


def ldsum(a, axis=-1):
    return np.sum(np.asarray(a, dtype=LD), axis=axis)


def viol_terms(E, gl, gu, x, xl, xu):
    E, x = E.astype(LD), x.astype(LD)
    tr = np.where(E > gu, E - gu, np.where(E < gl, gl - E, 0))
    tc = np.where(x > xu, x - xu, np.where(x < xl, xl - x, 0))
    return np.concatenate([tr, tc], 1)


def check_reductions(name, lp, lay, inp, bounds, fr, J, rng):
    """norm_violations, kt_residuals, norm_complementarity, row_norms and merit_phi at the update's point; returns the
    device outputs (for the lane-independence checks)"""
    xl, xu, gl, gu = bounds
    n, m, Bu = lay.n, lay.m, len(inp["x"])
    B = pad_batch(Bu)
    E, x = inp["E"], inp["x"]
    out = {}
    # norm_violations: host E / x for p = 1, the update's for p = 2 and inf
    gv = geo_for(max(n, m), B)
    d = chain(per_thread(m, B) + per_thread(n, B), B, gv[0])
    t = np.abs(viol_terms(E, gl, gu, x, xl, xu))
    # the inf-norm in float64, the device's own arithmetic: max, fabs and one subtraction per term
    t64 = np.concatenate([np.where(E > gu, E - gu, np.where(E < gl, gl - E, 0.0)),
                          np.where(x > xu, x - xu, np.where(x < xl, xl - x, 0.0))], 1)
    for pn in (np.inf, 1, 2):
        got = np.atleast_1d(lp.norm_violations(E if pn == 1 else None, x if pn == 1 else None, pn))
        out[f"viol{pn}"] = got
        if pn == np.inf:
            bit_equal(name + " norm_violations inf", got, np.abs(t64).max(axis=1, initial=0.0))
        elif pn == 1:
            check_bar(name + " norm_violations 1", got, ldsum(t), (1 + d) * U * ldsum(t))
        else:
            S = ldsum(t * t)
            barS = (3 + d) * U * S
            check_bar(name + " norm_violations 2", got, np.sqrt(S), sqrt_bar(S, barS))
    # row norms
    rn = np.asarray(lp.row_norms()).reshape(Bu, m)
    out["row_norms"] = rn
    rn_ref = np.sqrt(ldsum_rows(J, lay))
    check_bar(name + " row_norms", rn, rn_ref, (lay.rowlen / 2 + 1) * U * rn_ref)
    # kt residuals
    lam = rng.standard_normal((Bu, m)) * (rng.random((Bu, m)) > 0.2)
    mu_u = -rng.random((Bu, n)) * (rng.random((Bu, n)) > 0.5)
    mu_l = rng.random((Bu, n)) * (rng.random((Bu, n)) > 0.5)
    got = np.atleast_1d(lp.kt_residuals(lam, mu_u, mu_l))
    out["kt"] = got
    ref, bar = kt_ref(lay, J, inp["df"], lam, mu_u, mu_l, B)
    check_bar(name + " kt_residuals", got, ref, bar)
    # complementarity
    got = np.atleast_1d(lp.norm_complementarity(lam))
    out["compl"] = got
    ineq = gl != gu
    with np.errstate(invalid="ignore"):
        A = np.where(ineq, np.abs(np.minimum(E.astype(LD) - gl, gu - E.astype(LD)) * lam), 0).max(axis=1, initial=0)
    L = ldsum(np.where(ineq, lam.astype(LD) ** 2, 0))
    dc = chain(per_thread(m, B), B, geo_for(m, B)[0])
    den = 1 + np.sqrt(L)
    eps_den = np.sqrt(L) / den * ((1 + dc) / 2 * U + U) + U
    ref = A / den
    check_bar(name + " norm_complementarity", got, ref, ref * (3 * U + eps_den))
    # merit phi at E_trial with the handle's slacks (zero before any solve)
    nu = np.abs(rng.standard_normal((Bu, m))) * (rng.random((Bu, m)) > 0.2)
    Et = E + 1e-3 * rng.standard_normal((Bu, m))
    base = rng.standard_normal(Bu)
    alpha = rng.uniform(0.05, 1.0, Bu)
    got = np.atleast_1d(lp.merit_phi(base, Et, nu, alpha, fr))
    out["phi"] = got
    ref, bar = merit_ref(lay, bounds, E, Et, nu, np.zeros((Bu, m, 2)), alpha, base, fr, B)
    check_bar(f"{name} merit_phi ({'restoration' if fr else 'normal'})", got, ref, bar)
    out["inputs"] = (lam, mu_u, mu_l, nu, Et, base, alpha)
    return out


def sqrt_bar(S, barS):
    """first-order bar of sqrt(S) from a bar of S, plus the rounding of sqrt"""
    S = np.asarray(S, dtype=LD)
    barS = barS + 1e6 * ETA     # underflow of up to 1e6 squares
    rs = np.sqrt(S)
    return np.minimum(np.where(rs > 0, barS / (2 * np.where(rs > 0, rs, 1)), np.inf), np.sqrt(barS)) + U * rs


def ldsum_rows(J, lay):
    """sum of squares of every row of every lane, long double"""
    B, m = len(J), lay.m
    out = np.zeros((B, m), dtype=LD)
    nonempty = lay.rowlen > 0
    if lay.pat.nnz == 0:
        return out
    starts = lay.pat.row_ptr[:-1][nonempty]
    for c in chunks(B):
        v = J[c].astype(LD)
        out[c, :][:, nonempty] = np.add.reduceat(v * v, starts, axis=1)
    return out


def kt_ref(lay, J, df, lam, mu_u, mu_l, B):
    n, m, Bu = lay.n, lay.m, len(df)
    order = np.argsort(lay.pat.cols, kind="stable")
    cp = np.concatenate([[0], np.cumsum(lay.collen)])
    nonempty = lay.collen > 0
    rows = lay.pat.rows[order]
    a = np.zeros((Bu, n), dtype=LD)
    aa = np.zeros((Bu, n), dtype=LD)
    for c in chunks(Bu):
        if lay.pat.nnz == 0:
            break
        prod = J[c][:, order].astype(LD) * lam[c][:, rows].astype(LD)
        t = np.zeros((prod.shape[0], n), dtype=LD)
        t[:, nonempty] = np.add.reduceat(prod, cp[:-1][nonempty], axis=1)
        a[c] = t
        t = np.zeros((prod.shape[0], n), dtype=LD)
        t[:, nonempty] = np.add.reduceat(np.abs(prod), cp[:-1][nonempty], axis=1)
        aa[c] = t
    dfl = df.astype(LD)
    r = dfl - a - mu_u - mu_l
    T = np.abs(dfl) + aa + np.abs(mu_u) + np.abs(mu_l)
    gr, gc = geo_for(m, B), geo_for(n, B)
    nbx = max(gr[0], gc[0])
    d = chain(per_thread(n, B), B, nbx)
    R = ldsum(r * r)
    barR = U * ldsum((2 * (lay.collen + 4) + 1 + d) * T * T)
    sR = np.sqrt(R)
    D = ldsum(dfl * dfl)
    sD = np.sqrt(D)
    rn = np.sqrt(ldsum_rows(J, lay))
    M = (np.abs(lam) * rn).max(axis=1, initial=0) if m else np.zeros(Bu, dtype=LD)
    scalar = np.maximum(np.maximum(1, sD), M)
    dscal = np.maximum(sD * ((1 + d) / 2 * U + U), M * ((lay.rowlen.max(initial=0) / 2 + 2) * U))
    ref = sR / scalar
    bar = sqrt_bar(R, barR) / scalar + ref * dscal / scalar + U * ref
    return ref, bar


def merit_terms(lay, bounds, E, Et, pslack, alpha, fr):
    """(per-row violation term, its magnitude bound, slack sums) of k_merit in long double"""
    xl, xu, gl, gu = bounds
    lhs = Et.astype(LD)
    mag = np.abs(lhs)
    if fr:
        El = E.astype(LD)
        viol = np.maximum(0, np.maximum(El - gu, gl - El))
        s1, s2 = pslack[:, :, 0].astype(LD), pslack[:, :, 1].astype(LD)
        al = alpha.astype(LD)[:, None]
        cls = lay.cls
        sh = np.where((cls == EQ) | (cls == RANGE), s1 - s2, np.where(cls == LOWER, s1, -s1))
        lhs = lhs - viol + al * sh
        mag = mag + np.abs(El) + np.abs(al) * (np.abs(s1) + np.abs(s2))
    gfin = np.where(np.isfinite(gl), np.abs(gl), 0) + np.where(np.isfinite(gu), np.abs(gu), 0)
    v = np.maximum(0, np.maximum(lhs - gu, gl - lhs))
    return v, mag + 2 * gfin, (ldsum(pslack[:, :, 0] + pslack[:, :, 1].astype(LD)) if fr else None)


def merit_ref(lay, bounds, E, Et, nu, pslack, alpha, base, fr, B, Et_bar=None, nbx=None):
    m = lay.m
    v, mag, S = merit_terms(lay, bounds, E, Et, pslack, alpha, fr)
    nul = nu.astype(LD)
    RA = ldsum(nul * v)
    d = chain(per_thread(m, B), B, nbx or geo_for(m, B)[0])
    bar = (8 + d) * U * ldsum(nul * mag)
    if Et_bar is not None:
        bar = bar + ldsum(nul * Et_bar)
    ref = base.astype(LD) + RA
    if fr:
        al = alpha.astype(LD)
        bar = bar + np.abs(al) * (1 + d) * U * ldsum(np.abs(pslack).sum(axis=2))
        ref = ref + al * S
        bar = bar + 3 * U * (np.abs(base) + np.abs(al * S) + np.abs(RA))
    else:
        bar = bar + U * (np.abs(base) + np.abs(RA))
    return ref, bar


# ---- k_extract restated -----------------------------------------------------------------------------------------
def extract_ref(lay, raw, x, bounds, fr):
    xl, xu = bounds[0], bounds[1]
    n, m = lay.n, lay.m
    st = raw["status"]
    ok = (st == 0)[:, None]
    p = np.where(ok, raw["x"][:, :n], 0.0)
    mu_u = np.where(ok, raw["dual_ub"][:, :n], 0.0)
    mu_l = np.where(ok, raw["dual_lb"][:, :n], 0.0)
    mu_u = np.where(p < xu - x, 0.0, mu_u)
    mu_l = np.where(p > xl - x, 0.0, mu_l)
    lam = np.where(ok, raw["y"][:, :m], 0.0)
    slack = np.zeros((len(st), m, 2))
    if fr:
        lam[:, lay.adj] = np.where(ok, lam[:, lay.adj] + raw["y"][:, m:], 0.0)
        slack[:, :, 0] = np.where(ok, raw["x"][:, lay.s1], 0.0)
        two = np.flatnonzero(lay.s2 >= 0)
        slack[:, two, 1] = np.where(ok, raw["x"][:, lay.s2[two]], 0.0)
    return p, lam, mu_u, mu_l, slack, np.where(st < 0, 3, st).astype(np.int32)


def primal_feasibility(lay, raw, fr):
    """worst violation of each optimal lane's raw solution of its own LP, relative to 1 + the largest finite bound
    and row activity |K||x| of that lane (the engine's tolerance is relative to the LP's norms; a solution stored in
    another lane's slot violates by a share of the data that differs between lanes)"""
    ok = raw["status"] == 0
    worst = 0.0
    rp, ci = raw["row_ptr"][0], raw["col_idx"][0]
    fin = lambda b: np.abs(b[np.isfinite(b)]).max(initial=0.0)   # noqa: E731
    for s in np.flatnonzero(ok):
        K = sp.csr_matrix((raw["vals"][s], ci, rp), shape=(len(raw["rl"][s]), len(raw["lb"][s])))
        xs = raw["x"][s]
        Kx = K @ xs
        act = abs(K) @ np.abs(xs)
        scale = 1.0 + max(fin(raw["rl"][s]), fin(raw["ru"][s]), fin(raw["lb"][s]), fin(raw["ub"][s]),
                          act.max(initial=0.0))
        v = max(np.max(raw["rl"][s] - Kx, initial=0.0), np.max(Kx - raw["ru"][s], initial=0.0),
                np.max(raw["lb"][s] - xs, initial=0.0), np.max(xs - raw["ub"][s], initial=0.0)) / scale
        worst = max(worst, v)
    note(f"raw LP solution primal infeasibility / 1e-6 ({'restoration' if fr else 'normal'})", worst / 1e-6)
    assert worst <= 1e-6, worst
    return int(ok.sum())


# ---- the ACOPF evaluator restated in long double ----------------------------------------------------------------
class AcopfRef:
    def __init__(self, mdl):
        self.m = mdl
        cf = mdl._cf
        self.coef = [np.asarray(cf[k], dtype=LD) for k in ("a_pf", "b_pf", "c_pf", "a_qf", "b_qf", "c_qf", "a_pt",
                                                             "b_pt", "c_pt", "a_qt", "b_qt", "c_qt")]
        self.bal_rows = mdl._bal_rows - mdl.r_bal
        self.bal_cols = mdl._bal_cols
        self.shunt = np.isnan(mdl._bal_coef)
        self.bal_len = np.bincount(self.bal_rows, minlength=2 * mdl.nb)

    def evaluate(self, X, dX=None, plain=True):
        """f, E, dE (plain only), df, and their bars at X[b, n] (long double, exact inputs); dX: the absolute error
        of each variable (trial mode)"""
        mdl, net = self.m, self.m.net
        nb, ng, nl, nd = mdl.nb, mdl.ng, mdl.nl, mdl.nd
        b = len(X)
        dX = np.zeros_like(X) if dX is None else dX
        var = lambda o, i: (X[:, o + i], dX[:, o + i])   # noqa: E731
        f_, t_ = net.f_bus, net.t_bus
        (vaf, dvaf), (vat, dvat) = var(mdl.o_va, f_), var(mdl.o_va, t_)
        (vf, dvf), (vt, dvt) = var(mdl.o_vm, f_), var(mdl.o_vm, t_)
        br = np.arange(nl)
        flows = [var(mdl.o_p, br), var(mdl.o_q, br), var(mdl.o_p, nl + br), var(mdl.o_q, nl + br)]
        d = vaf - vat
        Dd = U * np.abs(d) + dvaf + dvat
        cs, sn = np.cos(d), np.sin(d)
        vv = vf * vt
        E = np.zeros((b, mdl.m), dtype=LD)
        Eb = np.zeros((b, mdl.m), dtype=LD)
        E[:, mdl.r_angmax:mdl.r_angmax + nl] = d
        E[:, mdl.r_angmin:mdl.r_angmin + nl] = d
        Eb[:, mdl.r_angmax:mdl.r_angmax + nl] = Eb[:, mdl.r_angmin:mdl.r_angmin + nl] = Dd
        E[:, mdl.r_ref], Eb[:, mdl.r_ref] = var(mdl.o_va, net.ref_bus)
        if nd:
            l1 = np.asarray(net.dc_loss1, dtype=LD)
            (pf, dpf), (pt, dpt) = var(mdl.o_pdc, np.arange(nd)), var(mdl.o_pdc, nd + np.arange(nd))
            E[:, mdl.r_dc:mdl.r_dc + nd] = (1 - l1) * pf + pt
            Eb[:, mdl.r_dc:mdl.r_dc + nd] = 3 * U * (np.abs((1 - l1) * pf) + np.abs(pt)) + np.abs(1 - l1) * dpf + dpt
        for side in (0, 1):
            (p, dp), (q, dq) = flows[2 * side], flows[2 * side + 1]
            r = mdl.r_thermal + 2 * br + side
            E[:, r] = p * p + q * q
            Eb[:, r] = 2 * U * (p * p + q * q) + 2 * np.abs(p) * dp + 2 * np.abs(q) * dq
        # balance rows: sum of +-1 coefficients times their column, then the shunt term
        cf = np.where(self.shunt, 0.0, mdl._bal_coef).astype(LD)
        xs = X[:, self.bal_cols]
        acc = np.zeros((b, 2 * nb), dtype=LD)
        mag = np.zeros((b, 2 * nb), dtype=LD)
        dacc = np.zeros((b, 2 * nb), dtype=LD)
        np.add.at(acc.T, self.bal_rows, (cf * xs).T)
        np.add.at(mag.T, self.bal_rows, (np.abs(cf) * np.abs(xs)).T)
        np.add.at(dacc.T, self.bal_rows, (np.abs(cf) * dX[:, self.bal_cols]).T)
        vm, dvm = X[:, mdl.o_vm:mdl.o_vm + nb], dX[:, mdl.o_vm:mdl.o_vm + nb]
        gs, bs = np.asarray(net.gs, dtype=LD), np.asarray(net.bs, dtype=LD)
        sh = np.empty((b, 2 * nb), dtype=LD)
        sh[:, 0::2], sh[:, 1::2] = gs * vm * vm, -bs * vm * vm
        dsh = np.empty((b, 2 * nb), dtype=LD)
        dsh[:, 0::2], dsh[:, 1::2] = 2 * np.abs(gs * vm) * dvm, 2 * np.abs(bs * vm) * dvm
        rb = slice(mdl.r_bal, mdl.r_bal + 2 * nb)
        E[:, rb] = acc + sh
        Eb[:, rb] = (self.bal_len + 3) * U * (mag + np.abs(sh)) + dacc + dsh
        # Ohm rows
        c = self.coef
        cm = [np.abs(c[3 * r + 1]) + np.abs(c[3 * r + 2]) for r in range(4)]
        for r in range(4):
            a_, b_, c_ = c[3 * r], c[3 * r + 1], c[3 * r + 2]
            own, oth, down, doth = (vf, vt, dvf, dvt) if r < 2 else (vt, vf, dvt, dvf)
            sg = 1 if r < 2 else -1
            expr = a_ * own * own + b_ * vv * cs + sg * c_ * vv * sn
            p, dp = flows[r]
            rows = mdl.r_ohm + 4 * br + r
            E[:, rows] = p - expr
            magr = np.abs(p) + np.abs(a_) * own * own + cm[r] * np.abs(vv)
            Eb[:, rows] = (10 * U * magr + dp + (2 * np.abs(a_ * own) + cm[r] * np.abs(oth)) * down
                           + cm[r] * np.abs(own) * doth + cm[r] * np.abs(vv) * Dd)
        pg, dpg = X[:, mdl.o_pg:mdl.o_pg + ng], dX[:, mdl.o_pg:mdl.o_pg + ng]
        c2, c1, c0 = (np.asarray(a, dtype=LD) for a in (net.cost2, net.cost1, net.cost0))
        f = ldsum(c2 * pg * pg + c1 * pg + c0)
        fb = (ng + 4) * U * ldsum(np.abs(c2) * pg * pg + np.abs(c1 * pg) + np.abs(c0)) + \
            ldsum((2 * np.abs(c2 * pg) + np.abs(c1)) * dpg)
        out = dict(f=f, fb=fb, E=E, Eb=Eb)
        if not plain:
            return out
        df = np.zeros((b, mdl.n), dtype=LD)
        dfb = np.zeros((b, mdl.n), dtype=LD)
        df[:, mdl.o_pg:mdl.o_pg + ng] = 2 * c2 * pg + c1
        dfb[:, mdl.o_pg:mdl.o_pg + ng] = 2 * U * (np.abs(2 * c2 * pg) + np.abs(c1))
        # Jacobian in j_str order; bar 0 = bit-exact entry
        J = np.zeros((b, mdl.nnz), dtype=LD)
        Jb = np.zeros((b, mdl.nnz), dtype=LD)
        k = 0
        for _ in range(2):
            J[:, k:k + 2 * nl:2], J[:, k + 1:k + 2 * nl:2] = 1, -1
            k += 2 * nl
        J[:, k] = 1
        k += 1
        if nd:
            J[:, k:k + 2 * nd:2] = (1.0 - np.asarray(net.dc_loss1))     # float64 on both sides
            J[:, k + 1:k + 2 * nd:2] = 1
            k += 2 * nd
        for j, (p, _) in enumerate(flows):
            J[:, k + j:k + 4 * nl:4] = 2 * p
        k += 4 * nl
        J[:, k:k + mdl._nnz_bal] = np.where(self.shunt, 0, mdl._bal_coef)
        for pos, i, is_q in mdl._bal_shunt:
            J[:, k + pos] = (-2 * bs[i] if is_q else 2 * gs[i]) * vm[:, i]
            Jb[:, k + pos] = U * np.abs(J[:, k + pos])
        k += mdl._nnz_bal
        for r in range(4):
            a_, b_, c_ = c[3 * r], c[3 * r + 1], c[3 * r + 2]
            sg = 1 if r < 2 else -1
            cross = b_ * cs + sg * c_ * sn
            k0 = k + 20 * br + 5 * r
            J[:, k0] = 1
            if r < 2:
                J[:, k0 + 1] = -(2 * a_ * vf + cross * vt)
                J[:, k0 + 2] = -(cross * vf)
                m1, m2 = 2 * np.abs(a_ * vf) + cm[r] * np.abs(vt), cm[r] * np.abs(vf)
            else:
                J[:, k0 + 1] = -(cross * vt)
                J[:, k0 + 2] = -(2 * a_ * vt + cross * vf)
                m1, m2 = cm[r] * np.abs(vt), 2 * np.abs(a_ * vt) + cm[r] * np.abs(vf)
            dd = vv * (-b_ * sn + sg * c_ * cs)
            J[:, k0 + 3], J[:, k0 + 4] = -dd, dd
            ud = U * np.abs(d)
            for j, mg in ((1, m1), (2, m2), (3, cm[r] * np.abs(vv)), (4, cm[r] * np.abs(vv))):
                Jb[:, k0 + j] = mg * (10 * U + ud)
        out.update(df=df, dfb=dfb, dE=J, dEb=Jb)
        return out


def check_eval(name, ref_fn, mdl, x, got, lanes_pin):
    """device (f, df, E, dE) of plain evaluations at x against the long-double restatement, in chunks of lanes"""
    f, df, E, dE = got
    Bu = len(x)
    for c in chunks(Bu):
        r = ref_fn.evaluate(x[c].astype(LD))
        check_bar(name + " evaluator f", f[c], r["f"], r["fb"])
        for key, bkey, g in (("df", "dfb", df), ("E", "Eb", E), ("dE", "dEb", dE)):
            exact = r[bkey] == 0
            if key == "E":
                # angle rows and the reference row are single operations on the inputs: bit-exact in float64
                exact[:] = False
                for s0 in (mdl.r_angmax, mdl.r_angmin):
                    exact[:, s0:s0 + mdl.nl] = True
                exact[:, mdl.r_ref] = True
                xx = x[c]
                ang = xx[:, mdl.o_va + mdl.net.f_bus] - xx[:, mdl.o_va + mdl.net.t_bus]
                bit_equal(name + " evaluator E angle rows", g[c][:, mdl.r_angmax:mdl.r_angmax + mdl.nl], ang)
                bit_equal(name + " evaluator E angle rows", g[c][:, mdl.r_angmin:mdl.r_angmin + mdl.nl], ang)
                bit_equal(name + " evaluator E reference row", g[c][:, mdl.r_ref], xx[:, mdl.o_va + mdl.net.ref_bus])
            elif key == "dE":
                pf = x[c][:, mdl.o_p:mdl.o_p + 2 * mdl.nl]
                qf = x[c][:, mdl.o_q:mdl.o_q + 2 * mdl.nl]
                k = 4 * mdl.nl + 1 + 2 * mdl.nd
                nl = mdl.nl
                for j, v in enumerate((pf[:, :nl], qf[:, :nl], pf[:, nl:], qf[:, nl:])):
                    bit_equal(name + " evaluator dE thermal 2 p", g[c][:, k + j:k + 4 * nl:4], 2.0 * v)
                bit_equal(name + " evaluator dE constants", g[c][exact], r[key][exact].astype(np.float64))
            else:
                bit_equal(name + f" evaluator {key} exact entries", g[c][exact], r[key][exact].astype(np.float64))
            check_bar(name + f" evaluator {key}", g[c][~exact], r[key][~exact], r[bkey][~exact])
    for s in lanes_pin:
        # the restatement against the float64 model (numpy's sin / cos, separate products)
        r = ref_fn.evaluate(x[s:s + 1].astype(LD))
        for key, host in (("E", mdl.eval_g(x[s], np.zeros(mdl.m))),
                          ("dE", mdl.eval_jac_g(x[s], "eval", None, None, np.zeros(mdl.nnz))),
                          ("df", mdl.eval_grad_f(x[s], np.zeros(mdl.n)))):
            rr = r[key][0].astype(np.float64)
            assert np.max(np.abs(rr - host) / (1 + np.abs(host)), initial=0) <= 1e-12, (name, key, s)
        assert abs(float(r["f"][0]) - mdl.eval_f(x[s])) <= 1e-12 * (1 + abs(mdl.eval_f(x[s])))


# ---- tests --------------------------------------------------------------------------------------------------------
DATA_CASES = [("case9", 1, False), ("case9", 2, False), ("case9", 33, False), ("case9", 33, True),
              ("case3", 33, False), ("case118", 100, False), ("case118", 1000, True), ("case1354", 1000, False),
              ("case1354", 1000, True), ("banded", 1, False), ("m0", 1, False), ("m0", 33, True), ("one", 1, False),
              ("one", 33, True), ("classes", 1, False), ("classes", 33, True)]


def geometry_claims(nlp, Bu):
    B = pad_batch(Bu)
    n, m, nz = nlp.n, nlp.m, len(nlp.j_str)
    gc, gr = geo_for(n, B), geo_for(m, B)
    loops = lambda cnt: per_thread(cnt, B) > 1                 # noqa: E731
    claims = dict(B=B, grid_y=gr[1], grid_x_rows=gr[0], row_loop=loops(m), col_loop=loops(n), coo_loop=loops(nz))
    if nlp.name == "case9":
        assert B == {1: 1, 2: 32, 33: 64}[Bu] and gr[1] == {1: 1, 2: 1, 33: 2}[Bu]
    if nlp.name in ("case118", "case1354") and Bu >= 1000:
        assert B == 1024 and gr[0] == 74 and loops(m) and loops(n)
    if nlp.name == "case1354":
        assert loops(2 * nlp.model.nb) and loops(nlp.model.nl)     # k_acopf_bus / k_acopf_branch sweep again
    if nlp.name == "banded":
        assert B == 1 and nz > MAX_BX * THREADS and loops(nz) and loops(n) and loops(m)
    return claims


@pytest.mark.parametrize("name,Bu,per", DATA_CASES)
def test_lp_data_and_reductions(gpu, name, Bu, per):
    """LP data of both phases bit-exact, the reductions within their bars, and lane independence, at adversarial
    inputs (no solve)."""
    t0 = time.time()
    nlp = make_nlp(name)
    claims = geometry_claims(nlp, Bu)
    rng = np.random.default_rng(Bu * 7 + per)
    lay = Layout(nlp)
    bounds = lane_bounds(nlp, Bu, per)
    inp = adversarial_inputs(nlp, bounds, Bu, rng)
    lp = new_handle(nlp, bounds, Bu, per)
    assert (lp.lp_cols, lp.lp_rows) == (lay.ncol_fr, lay.nrow_fr)
    J = lay.assemble(inp["dE"])
    perm = rng.permutation(Bu)
    shared_as_per = None if per or Bu == 1 else new_handle(nlp, bounds, Bu, True)
    for fr in (False, True):
        lp.update(inp["x"], inp["f"], inp["df"], inp["E"], inp["dE"], inp["delta"], fr)
        dev = read_lanes(lp, Bu, False)
        check_lp_data(name, lay, nlp, inp, bounds, fr, dev)
        out = check_reductions(name, lp, lay, inp, bounds, fr, J, np.random.default_rng(5))
        lam, mu_u, mu_l, nu, Et, base, alpha = out.pop("inputs")
        again = replay(lp, inp, fr, lam, mu_u, mu_l, nu, Et, base, alpha, None)
        for k in out:
            bit_equal(f"repeat call {k}", again[k], out[k])
        if Bu > 1:
            pl = lambda a: a[perm]                               # noqa: E731
            pin = {k: (v[perm] if np.ndim(v) else v) for k, v in inp.items()}
            if per:
                lpp = new_handle(nlp, tuple(b[perm] for b in bounds), Bu, True)
            else:
                lpp = lp
            got = replay(lpp, pin, fr, pl(lam), pl(mu_u), pl(mu_l), pl(nu), pl(Et), pl(base), pl(alpha), None)
            for k in out:
                bit_equal(f"permuted lanes {k}", got[k], out[k][perm])
            if lpp is not lp:
                lpp.close()
            if shared_as_per is not None:
                got = replay(shared_as_per, inp, fr, lam, mu_u, mu_l, nu, Et, base, alpha, None)
                for k in out:
                    bit_equal(f"shared bounds as per-scenario arrays {k}", got[k], out[k])
                bit_equal("shared bounds as per-scenario arrays: LP lb",
                          np.array([get_lp(shared_as_per, s, False)["lb"] for s in (0, Bu - 1)]), dev["lb"][[0, Bu - 1]])
    lp.close()
    if shared_as_per is not None:
        shared_as_per.close()
    print(f"\n    geometry {claims}")
    report(f"{name} B={Bu} {'per-scenario' if per else 'shared'} bounds", t0)


def replay(lp, inp, fr, lam, mu_u, mu_l, nu, Et, base, alpha, _):
    """every reduction of check_reductions on `lp` after an update with `inp`; device outputs only"""
    lp.update(inp["x"], inp["f"], inp["df"], inp["E"], inp["dE"], inp["delta"], fr)
    Bu = len(inp["x"])
    out = {}
    for pn in (np.inf, 1, 2):
        out[f"viol{pn}"] = np.atleast_1d(lp.norm_violations(inp["E"] if pn == 1 else None,
                                                            inp["x"] if pn == 1 else None, pn))
    out["row_norms"] = np.asarray(lp.row_norms()).reshape(Bu, -1)
    out["kt"] = np.atleast_1d(lp.kt_residuals(lam, mu_u, mu_l))
    out["compl"] = np.atleast_1d(lp.norm_complementarity(lam))
    out["phi"] = np.atleast_1d(lp.merit_phi(base, Et, nu, alpha, fr))
    return out


SOLVE_CASES = [("case9", 1, False, (0, 1)), ("case9", 2, False, (0, 1)), ("case9", 33, True, (0, 1)),
               ("case3", 33, False, (0, 1)), ("case118", 100, False, (0, 1)), ("case118", 1000, True, (0, 1)),
               ("case1354", 1000, False, (0,))]


def acopf_point(mdl, Bu, rng):
    """points inside the box, varied per lane; the reference angle sits at 0 on every other lane"""
    lo = np.where(np.isfinite(mdl.x_L), mdl.x_L, -0.3)
    hi = np.where(np.isfinite(mdl.x_U), mdl.x_U, 0.3)
    x0 = np.clip(mdl.x0, mdl.x_L, mdl.x_U)
    w = rng.uniform(0.0, 0.05, (Bu, 1))
    x = (1 - w) * x0 + w * rng.uniform(lo, hi, (Bu, mdl.n))
    x[::2, mdl.o_va + mdl.net.ref_bus] = 0.0
    return x


@pytest.mark.parametrize("name,Bu,per,phases", SOLVE_CASES)
def test_evaluator_solve_readback(gpu, name, Bu, per, phases):
    """device ACOPF evaluation (plain) against long double; the LP data it feeds; a masked solve; the read-back against
    k_extract restated on the raw solution; merit_derivative and acopf_trial (trial evaluation + merit) against
    long double; lane independence of the evaluator and repeat calls."""
    t0 = time.time()
    nlp = make_nlp(name)
    mdl = nlp.model
    claims = geometry_claims(nlp, Bu)
    B = pad_batch(Bu)
    rng = np.random.default_rng(100 + Bu)
    lay = Layout(nlp)
    bounds = lane_bounds(nlp, Bu, per)
    lp = new_handle(nlp, bounds, Bu, per)
    lp.attach_acopf(mdl)
    ref_fn = AcopfRef(mdl)
    x = acopf_point(mdl, Bu, rng)
    delta = np.where(np.arange(Bu) % 3 == 2, 0.05, 1000.0)
    pins = sorted({0, 32, Bu - 1} & set(range(Bu)))
    mask = None
    if Bu >= 33:
        mask = np.ones(Bu, dtype=bool)
        mask[[0, 32, Bu - 1]] = False
    for fr in phases:
        lp.set_active(None)
        lp.eval_acopf(x, delta, fr)
        f, df, E, dE = lp.get_eval()
        check_eval(name, ref_fn, mdl, x, (f, df, E, dE), pins if fr == phases[0] else [])
        inp = dict(x=x, f=f, df=df, E=E, dE=dE, delta=delta)
        check_lp_data(name, lay, nlp, inp, bounds, fr, read_lanes(lp, Bu, False))
        lp.set_active(mask)
        lp.solve()
        raw = read_lanes(lp, Bu, True)
        if mask is not None:
            assert np.all(raw["status"][~mask] == SKIPPED)
        solved = primal_feasibility(lay, raw, fr)
        print(f"\n    {name} {'restoration' if fr else 'normal'}: raw statuses {np.unique(raw['status'], return_counts=True)}")
        assert solved >= 1, (fr, np.unique(raw["status"], return_counts=True))
        p, lam, mu_u, mu_l, slack, st = lp.extract()
        ref = extract_ref(lay, raw, x, bounds, fr)
        for k, g, r in zip(("p", "lambda", "mult_x_U", "mult_x_L", "p_slack", "status"),
                           (p, lam, mu_u, mu_l, slack, st), ref):
            bit_equal(f"extract {k} ({'restoration' if fr else 'normal'})", g, r)
        if mask is not None:
            assert np.all(st[~mask] == SKIPPED) and not p[~mask].any() and not lam[~mask].any()
        # merit_derivative
        nu = np.abs(rng.standard_normal((Bu, lay.m))) * (rng.random((Bu, lay.m)) > 0.2)
        got = np.atleast_1d(lp.merit_derivative(nu, fr))
        bit_equal("merit_derivative repeat call", np.atleast_1d(lp.merit_derivative(nu, fr)), got)
        zero = np.zeros(Bu)
        nbx = max(geo_for(lay.m, B)[0], geo_for(lay.n, B)[0])
        Ra, Rbar = merit_ref(lay, bounds, E, E, nu, slack, zero, zero, fr, B, nbx=nbx)
        if fr:
            S = ldsum(slack[:, :, 0] + slack[:, :, 1].astype(LD))
            dm = chain(per_thread(lay.m, B), B, nbx)
            ref = S - Ra
            bar = Rbar + (1 + dm) * U * ldsum(np.abs(slack).sum(axis=2)) + U * np.abs(ref)
        else:
            dd = chain(per_thread(lay.n, B), B, nbx)
            prod = df.astype(LD) * p
            ref = ldsum(prod) - Ra
            bar = Rbar + (1 + dd) * U * ldsum(np.abs(prod)) + U * np.abs(ref)
        check_bar(f"{name} merit_derivative ({'restoration' if fr else 'normal'})", got, ref, bar)
        # acopf_trial: f and g at x + alpha p on the device, then the merit
        alpha = rng.uniform(0.05, 1.0, Bu)
        base = np.abs(rng.standard_normal(Bu))
        got = np.atleast_1d(lp.acopf_trial(alpha, nu, base if fr else None, fr))
        bit_equal("acopf_trial repeat call", np.atleast_1d(lp.acopf_trial(alpha, nu, base if fr else None, fr)), got)
        refs, bars = [], []
        for c in chunks(Bu):
            xl, al, pl = x[c].astype(LD), alpha[c].astype(LD)[:, None], p[c].astype(LD)
            xt = xl + al * pl
            r = ref_fn.evaluate(xt, U * (np.abs(xt) + np.abs(al * pl)), plain=False)
            sub = tuple(b[c] for b in bounds)
            if fr:
                rr, bb = merit_ref(lay, sub, E[c], r["E"], nu[c], slack[c], alpha[c], base[c], True, B, r["Eb"])
            else:
                rr, bb = merit_ref(lay, sub, E[c], r["E"], nu[c], slack[c], alpha[c], np.zeros(len(xl)), False, B,
                                   r["Eb"])
                rr = rr + r["f"]
                bb = bb + r["fb"] + U * (np.abs(r["f"]) + np.abs(rr))
            refs.append(rr)
            bars.append(bb)
        check_bar(f"{name} acopf_trial ({'restoration' if fr else 'normal'})", got, np.concatenate(refs),
                  np.concatenate(bars))
    # lane independence of the evaluator: permuted points give permuted outputs, bit for bit
    if Bu > 1:
        perm = rng.permutation(Bu)
        lp.set_active(None)
        lp.eval_acopf(x, delta, False)
        first = lp.get_eval()
        lp.eval_acopf(x[perm], delta[perm], False)
        for k, a, b in zip(("f", "df", "E", "dE"), lp.get_eval(), first):
            bit_equal(f"evaluator permuted lanes {k}", a, b[perm])
    lp.close()
    print(f"\n    geometry {claims}")
    report(f"{name} B={Bu} {'per-scenario' if per else 'shared'} bounds, solve", t0)


def test_readback_after_pdhg_hybrid(gpu):
    """engine 5 compacts the running LPs and scatters them back: every lane's raw solution must be feasible for its
    own LP and the read-back must be k_extract's restatement of it (case9, 160 scenarios, normal phase)."""
    t0 = time.time()
    nlp = make_nlp("case9")
    mdl = nlp.model
    Bu = 160
    lay = Layout(nlp)
    bounds = lane_bounds(nlp, Bu, True)
    lp = new_handle(nlp, bounds, Bu, True, eps_rel=1e-7, engine=5)
    lp.attach_acopf(mdl)
    x = acopf_point(mdl, Bu, np.random.default_rng(7))
    lp.eval_acopf(x, 1000.0, False)
    lp.solve()
    raw = read_lanes(lp, Bu, True)
    assert primal_feasibility(lay, raw, False) == Bu
    got = lp.extract()
    for k, g, r in zip(("p", "lambda", "mult_x_U", "mult_x_L", "p_slack", "status"), got,
                       extract_ref(lay, raw, x, bounds, False)):
        bit_equal(f"extract after engine 5 {k}", g, r)
    lp.close()
    report("case9 B=160 engine 5", t0)


@pytest.mark.parametrize("Bu", [1, 33])
def test_readback_range_rows(gpu, Bu):
    """the four row classes (the ACOPF models have no range rows): k_extract sums the dual of a range row's extra <= row
    into lambda in restoration; read-back bit-exact against the raw solution, the raw solution feasible, and
    merit_derivative in long double, both phases"""
    t0 = time.time()
    nlp = make_nlp("classes")
    lay = Layout(nlp)
    rng = np.random.default_rng(Bu)
    bounds = lane_bounds(nlp, Bu, Bu > 1)
    B = pad_batch(Bu)
    inp = adversarial_inputs(nlp, bounds, Bu, rng)
    lo, hi = bounds[0], bounds[1]
    with np.errstate(invalid="ignore"):
        inp["x"] = np.where(np.isfinite(lo) & np.isfinite(hi), 0.5 * (lo + hi), np.where(np.isfinite(lo), lo + 0.5,
                                                                                         np.where(np.isfinite(hi), hi - 0.5, 0.0)))
    inp["dE"] = rng.uniform(0.5, 2.0, inp["dE"].shape) * rng.choice([-1.0, 1.0], inp["dE"].shape)
    inp["delta"] = np.where(np.arange(Bu) % 2, 0.5, 1000.0)
    lp = new_handle(nlp, bounds, Bu, Bu > 1)
    extra_dual = 0
    for fr in (False, True):
        lp.update(inp["x"], inp["f"], inp["df"], inp["E"], inp["dE"], inp["delta"], fr)
        lp.solve()
        raw = read_lanes(lp, Bu, True)
        check_lp_data("classes", lay, nlp, inp, bounds, fr, raw)
        solved = primal_feasibility(lay, raw, fr)
        print(f"\n    classes {'restoration' if fr else 'normal'}: raw statuses "
              f"{np.unique(raw['status'], return_counts=True)}")
        if fr:
            assert solved == Bu
            extra_dual = int(np.count_nonzero(raw["y"][:, lay.m:]))
        got = lp.extract()
        ref = extract_ref(lay, raw, inp["x"], bounds, fr)
        for k, g, r in zip(("p", "lambda", "mult_x_U", "mult_x_L", "p_slack", "status"), got, ref):
            bit_equal(f"extract {k} ({'restoration' if fr else 'normal'})", g, r)
        p, slack = got[0], got[4]
        nu = np.abs(rng.standard_normal((Bu, lay.m)))
        zero = np.zeros(Bu)
        nbx = max(geo_for(lay.m, B)[0], geo_for(lay.n, B)[0])
        Ra, Rbar = merit_ref(lay, bounds, inp["E"], inp["E"], nu, slack, zero, zero, fr, B, nbx=nbx)
        d = chain(per_thread(lay.n if not fr else lay.m, B), B, nbx)
        if fr:
            S = ldsum(slack[:, :, 0] + slack[:, :, 1].astype(LD))
            ref, bar = S - Ra, Rbar + (1 + d) * U * ldsum(np.abs(slack).sum(axis=2))
        else:
            prod = inp["df"].astype(LD) * p
            ref, bar = ldsum(prod) - Ra, Rbar + (1 + d) * U * ldsum(np.abs(prod))
        check_bar(f"classes merit_derivative ({'restoration' if fr else 'normal'})",
                  np.atleast_1d(lp.merit_derivative(nu, fr)), ref, bar + U * np.abs(ref))
    if Bu > 1:
        assert extra_dual > 0      # some extra <= row is active, so its dual reaches lambda
    lp.close()
    report(f"classes B={Bu} range rows, solve", t0)
