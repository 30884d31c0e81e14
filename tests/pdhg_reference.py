"""The PDHG engines' solve restated in numpy at a chosen precision (``np.longdouble`` by default).

This follows the code operation by operation, not the algorithm in general: ``LpSolver::precondition`` (Ruiz
passes on the previous pass's scales, one Pock-Chambolle 1-norm pass, the ``tiny_rel`` test on the original
coefficients), the norms of ``k_prepare_*``, ``pdhg_start``, the cold / warm start of ``k_prepare_finish``, the
block schedule of ``enqueue_block`` (steps 0 and steps-1 of a block are check steps), the check terms and the
decision of ``pdhg.cuh`` (``pdhg_decide``), ``k_apply`` with the Halpern weight of ``k_store_kstep`` and
``k_finalize``.  The streaming kernels, the group kernel and the row-partitioned kernels all compute this
iteration; they differ only in the order of their sums.

Vectors are element-major ``[len, B]`` like the device's; every lane is one LP on the shared pattern.  Besides the
solution the run records, per check, k, r, omega and each decision, and for every discrete decision how far its
quantity was from the threshold (``margins``).  The tests demand exact equality of the discrete outcomes only
where those margins clear the rounding bars (``BARS``) by a wide factor.

``tools/pdhg_proto.py`` is a different prototype (check schedule, PID gains, no finalize); it is not this file.
"""
from __future__ import annotations

import numpy as np

OPTIMAL, INFEASIBLE, ITERATION_LIMIT, NUMERICAL_ERROR = 0, 1, 3, 4
K_TINY_REL = 1e-8          # lp_solver.cuh kTinyRel
K_MAX_STEPS = 256          # pdhg_group.cuh kMaxSteps: the group kernel's cap of check_every

# asm_lp_default_params
PARAMS = dict(eps_rel=1e-8, eps_infeas=1e-9, max_iter=2_000_000, check_every=64, ruiz_iters=10,
              restart_sufficient=0.2, restart_necessary=0.8, restart_artificial=0.36,
              pid_kp=0.5, pid_ki=0.0, pid_kd=0.0, weight_balance=0.0, tiny_rel=0.0)

# Rounding bars of a double implementation of this operation order, times sqrt(iterations of the window): the drift
# of a nonexpansive iteration grows like a random walk, not linearly (measured: per-iteration normalisation makes
# long windows' bars 30x looser than their drift).  Each is about 10x the worst float64-vs-longdouble drift over the
# generator's cases; tests/test_pdhg_reference_cpu.py pins them.  x, y, the bound duals: infinity norm of the
# difference over the infinity norm of the reference; pres / dres / gap: absolute difference over 1 + nq_un,
# 1 + nc_un, 1 + |pobj| + |dobj| (or the value, when larger); r: relative (near convergence r is a norm of
# differences of nearly equal iterates, so its relative drift is the largest of all).  x alone is set at 40x: on the
# device (FMA-contracted, other summation orders) its drift reached 0.88 of a 10x bar (NVIDIA B200), too little
# headroom for a compiler change.
BARS = dict(x=2e-13, y=7e-12, zl=7e-12, zu=7e-12, pres=1.5e-14, dres=2e-13, gap=2e-13, r=1e-8)


def bar(quantity, iterations):
    return BARS[quantity] * np.sqrt(max(1, int(iterations)))


class Pattern:
    """CSR pattern (duplicates allowed) and the CSC order the device builds from it (LpSolver::init): columns
    ascending, rows ascending within a column; ``csc_src`` maps a CSC position to its CSR position."""

    def __init__(self, n, m, row_ptr, col_idx):
        self.n, self.m = int(n), int(m)
        self.row_ptr = np.asarray(row_ptr, dtype=np.int64)
        self.col_idx = np.asarray(col_idx, dtype=np.int64)
        self.nnz = int(self.row_ptr[-1])
        self.row_of = np.repeat(np.arange(self.m), np.diff(self.row_ptr))
        self.csc_src = np.argsort(self.col_idx, kind="stable")
        self.row_idx = self.row_of[self.csc_src]
        self.col_ptr = np.concatenate([[0], np.cumsum(np.bincount(self.col_idx, minlength=self.n))]).astype(np.int64)


def _seg(ufunc, vals, ptr, empty=0.0):
    """ufunc-reduce consecutive segments [ptr[i], ptr[i+1]) of vals along axis 0; empty segments give `empty`."""
    out = np.full((len(ptr) - 1,) + vals.shape[1:], empty, dtype=vals.dtype)
    nz = np.flatnonzero(ptr[1:] > ptr[:-1])
    if nz.size:
        out[nz] = ufunc.reduceat(vals, ptr[nz], axis=0)
    return out


def _support(x, l, u):
    """pdhg_support: l x for x > 0, u x for x < 0, else 0."""
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(x > 0, l * x, np.where(x < 0, u * x, 0.0))


class _Margins:
    """Smallest relative distance of each decision's quantity from its threshold, over all checks and lanes."""

    def __init__(self):
        self.m = {}

    def add(self, name, value, thr, scale=None):
        scale = abs(thr) if scale is None else scale
        if not np.isfinite(value) or not np.isfinite(thr) or scale == 0:
            return
        d = float(abs(value - thr) / scale)
        self.m[name] = min(self.m.get(name, np.inf), d)


def _decide(st, s, P, q, jit, steps, dt, mg):
    """pdhg_decide for lane s (scalars of dtype dt); returns restart_flag (0 Halpern, 1 restart, 2 freeze)."""
    one = dt(1.0)
    omega, eta, sb, sc = st["omega"][s], st["eta"][s], st["sb"][s], st["sc"][s]
    tau, sigma = eta / omega, eta * omega
    k = int(st["k0"][s]) + jit + 1
    total = int(st["total"][s]) + jit + 1
    r2 = q["dx2"] / tau - dt(2.0) * q["dyadx"] + q["dy2"] / sigma
    r = np.sqrt(max(r2, dt(0.0)))
    # r^2 is a difference of terms of size rs2: its rounding error is relative to rs2, not to r^2
    rs2 = q["dx2"] / tau + dt(2.0) * abs(q["dyadx"]) + q["dy2"] / sigma
    unit = one / (sb * sc)
    pobj = q["pobj"] * unit
    dobj = (q["dobj_row"] + q["dobj_col"]) * unit
    pres, dres = np.sqrt(q["pres2"]), np.sqrt(q["dres2"])
    gap = abs(pobj - dobj)
    st["pobj"][s], st["dobj"][s], st["pres"][s], st["dres"][s], st["gap"][s] = pobj, dobj, pres, dres, gap
    eps = dt(P["eps_rel"])
    dp, dd, dg = one + st["nq_un"][s], one + st["nc_un"][s], one + abs(pobj) + abs(dobj)
    mg.add("opt_pres", pres, eps * dp, dp)
    mg.add("opt_dres", dres, eps * dd, dd)
    mg.add("opt_gap", gap, eps * dg, dg)
    status = -1
    if pres <= eps * dp and dres <= eps * dd and gap <= eps * dg:
        status = OPTIMAL
    if status < 0:
        nr = q["ray_max"] / sc
        if nr > 0:
            robj = (q["ray_row"] + q["ray_col"]) * unit / nr
            kty = q["kty_max"] / sc / nr
            thr = dt(P["eps_infeas"]) * max(one, kty)
            mg.add("farkas", robj, thr)
            if robj > thr:
                status = INFEASIBLE
    if not (r == r) or not (pobj == pobj):
        status = NUMERICAL_ERROR
    restart = 0
    if status < 0:
        if k == 1:
            st["r0"][s] = r
            st["rs2_0"][s] = rs2
        elif jit + 1 == steps:
            r0 = st["r0"][s]
            bs, bn = dt(P["restart_sufficient"]) * r0, dt(P["restart_necessary"]) * r0
            mg.add("restart_sufficient", r, bs)
            if r <= bs:
                restart = 1
            else:
                mg.add("restart_necessary", r, bn)
                if r <= bn:
                    mg.add("restart_r_prev", r, st["r_prev"][s])
                if r <= bn and r > st["r_prev"][s]:
                    restart = 1
                # integer arithmetic against a double: exactly what the device computes
                elif float(k) >= P["restart_artificial"] * float(total):
                    restart = 1
        st["r_prev"][s] = r
        st["rs2_prev"][s] = rs2
        if restart:
            ddx, ddy = np.sqrt(q["dxa2"]), np.sqrt(q["dya2"])
            rp, rd = pres / dp, dres / dd
            if P["weight_balance"] > 0:
                if rp > 0 and rd > 0:
                    omega = np.exp(np.log(omega) + dt(P["weight_balance"]) * np.log(rp / rd))
            else:
                mg.add("weight_ddx", ddx, dt(1e-16))
                mg.add("weight_ddy", ddy, dt(1e-16))
                if ddx > dt(1e-16) and ddy > dt(1e-16):
                    e = np.log(omega * ddx / ddy)
                    st["e_sum"][s] += e
                    dlog = -(dt(P["pid_kp"]) * e + dt(P["pid_ki"]) * st["e_sum"][s] +
                             dt(P["pid_kd"]) * (e - st["e_prev"][s]))
                    omega = np.exp(np.log(omega) + dlog)
                    st["e_prev"][s] = e
            w0 = st["omega0"][s]
            mg.add("weight_low", omega, w0 * dt(1e-16))
            mg.add("weight_high", omega, w0 * dt(1e16))
            if not (omega > w0 * dt(1e-16) and omega < w0 * dt(1e16)):
                omega = w0
                st["e_sum"][s] = 0
                st["e_prev"][s] = 0
            st["omega"][s] = omega
            st["restarts"][s] += 1
            st["r_prev"][s] = dt(np.inf)
    flag = restart
    if jit + 1 == steps:
        st["total"][s] += steps
        st["k0"][s] = 0 if restart else st["k0"][s] + steps
    if status >= 0:
        st["total"][s] = total
        st["status"][s] = status
        flag = 2
    return flag, k, r, rs2


def solve(pat, lp, params=None, dtype=np.longdouble, warm=0, start=None, start_ok=None, period_cap=None):
    """Run the PDHG solve of every lane of `lp` on `pat`.

    lp: dict of float64 arrays vals [nnz, B], c, lb, ub [n, B], rl, ru [m, B], optional c0 [B].
    warm: 0 cold, 1 (x, y), 2 y only, from start = (xo [n, B], yo [m, B]) in unscaled units, on the lanes where
    start_ok is true (all when None).  period_cap: the group kernel's cap of check_every (K_MAX_STEPS).
    Returns a dict: per-lane info (status, iterations, restarts, objective, dual_objective, pres, dres, gap,
    nq_un, nc_un), x, y, zl, zu [len, B], `trace` (one dict per check) and `margins`."""
    P = dict(PARAMS)
    P.update(params or {})
    dt = dtype
    f = lambda a: np.asarray(a, dtype=dt)
    vals, c, lb, ub, rl, ru = (f(lp[k]) for k in ("vals", "c", "lb", "ub", "rl", "ru"))
    n, m, B = pat.n, pat.m, vals.shape[1]
    c0 = np.zeros(B) if lp.get("c0") is None else np.asarray(lp["c0"], dtype=np.float64)
    mg = _Margins()
    rp, cp, ci, ri, src = pat.row_ptr, pat.col_ptr, pat.col_idx, pat.row_idx, pat.csc_src
    zero, one = dt(0.0), dt(1.0)

    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        # ---- preconditioning (LpSolver::precondition)
        absv = np.abs(vals)
        tiny_rel = P["tiny_rel"] if P["tiny_rel"] > 0 else K_TINY_REL
        gmax = absv.max(axis=0) * dt(tiny_rel / K_TINY_REL) if pat.nnz else np.zeros(B, dt)
        tiny = dt(K_TINY_REL) * gmax
        row_a0 = _seg(np.maximum, absv, rp)
        col_a0 = _seg(np.maximum, absv[src], cp)
        for a0, name in ((row_a0, "tiny_row"), (col_a0, "tiny_col")):
            for s in range(B):
                keep = a0[:, s] > 0
                if keep.any() and tiny[s] > 0:
                    mg.add(name, float(np.min(np.abs(np.log(a0[keep, s] / tiny[s])))), 0.0, 1.0)
        dr, dc = np.ones((m, B), dt), np.ones((n, B), dt)
        ruiz = int(P["ruiz_iters"])
        for it in range(ruiz + 1):
            red = np.add if it == ruiz else np.maximum      # last pass: Pock-Chambolle 1-norms
            t = np.abs(vals * dr[pat.row_of] * dc[ci])
            ra = _seg(red, t, rp)
            ca = _seg(red, t[src], cp)
            sr = np.where((ra > 0) & (row_a0 > tiny), one / np.sqrt(ra), one)
            scf = np.where((ca > 0) & (col_a0 > tiny), one / np.sqrt(ca), one)
            dr, dc = dr * sr, dc * scf                     # both sides of a pass use the previous scales
        A = vals * dr[pat.row_of] * dc[ci]
        AT = A[src]
        # ---- k_prepare_cols / k_prepare_rows / pdhg_start
        cs = c * dc
        lbs, ubs = lb / dc, ub / dc
        c2, cun2 = (cs * cs).sum(axis=0), (c * c).sum(axis=0)
        rls, rus = rl * dr, ru * dr
        fl, fu = np.isfinite(rl), np.isfinite(ru) & (ru != rl)
        q2 = np.where(fl, rls * rls, zero).sum(axis=0) + np.where(fu, rus * rus, zero).sum(axis=0)
        qun2 = np.where(fl, rl * rl, zero).sum(axis=0) + np.where(fu, ru * ru, zero).sum(axis=0)
        sb = one / (np.sqrt(q2) + one)
        sc = one / (np.sqrt(c2) + one)
        ncs, nqs = np.sqrt(c2) * sc, np.sqrt(q2) * sb
        omega = np.where((ncs > 0) & (nqs > 0), ncs / nqs, one)
        st = dict(omega=omega.copy(), omega0=omega.copy(), eta=np.full(B, dt(0.998)), sb=sb, sc=sc,
                  nq_un=np.sqrt(qun2), nc_un=np.sqrt(cun2), r0=np.zeros(B, dt), r_prev=np.full(B, dt(np.inf)),
                  rs2_0=np.zeros(B, dt), rs2_prev=np.zeros(B, dt), e_sum=np.zeros(B, dt), e_prev=np.zeros(B, dt), pobj=np.zeros(B, dt), dobj=np.zeros(B, dt),
                  pres=np.full(B, dt(np.inf)), dres=np.full(B, dt(np.inf)), gap=np.full(B, dt(np.inf)),
                  total=np.zeros(B, np.int64), k0=np.zeros(B, np.int64), restarts=np.zeros(B, np.int64),
                  status=np.full(B, -1, np.int64))
        # ---- k_prepare_finish
        cs = cs * sc
        lbs, ubs = lbs * sb, ubs * sb
        rls, rus = rls * sb, rus * sb
        wl = np.full(B, bool(warm)) if start_ok is None else (np.asarray(start_ok, bool) & bool(warm))
        xo, yo = (np.zeros((n, B)), np.zeros((m, B))) if start is None else start
        x = np.where(wl & (warm == 1), f(xo) / dc * sb, zero)
        x = np.minimum(np.maximum(x, lbs), ubs)
        y = np.where(wl, f(yo) / dr * sc, zero)
        y = np.where(np.isfinite(rl), y, np.minimum(y, zero))
        y = np.where(np.isfinite(ru), y, np.maximum(y, zero))
        xa, ya = x.copy(), y.copy()
        xp_l, rc_l, yp_l = x.copy(), np.zeros((n, B), dt), y.copy()
        fin_lb, fin_ub = np.isfinite(lbs), np.isfinite(ubs)
        fixed = lbs == ubs
        inf_rl, inf_ru = ~np.isfinite(rls), ~np.isfinite(rus)

        def aty(w):       # CSC pass: A'w
            return _seg(np.add, AT * w[ri], cp)

        def ax(w):        # CSR pass: A w
            return _seg(np.add, A * w[ci], rp)

        def dual_step(a, y, sigma):
            t = a - y * (one / sigma)
            return np.where(t < rls, sigma * (rls - t), np.where(t > rus, sigma * (rus - t), zero))

        # ---- the block schedule of enqueue_block / the group kernel
        steps = max(2, int(P["check_every"]))
        if period_cap:
            steps = min(steps, period_cap)
        trace = []
        it = 0
        while it < P["max_iter"] and (st["status"] < 0).any():
            for j in range(steps):
                live = st["status"] < 0
                if not live.any():
                    break
                kk = st["k0"] + j + 1
                w = kk.astype(dt) / (kk.astype(dt) + one)       # pdhg_halpern_weight; k_store_kstep's k
                tau, sigma = st["eta"] / st["omega"], st["eta"] * st["omega"]
                g = cs - aty(y)
                v = x - tau * g
                xpv = np.minimum(np.maximum(v, lbs), ubs)
                xb = 2 * xpv - x
                if 0 < j < steps - 1:
                    xn = w * xb + (one - w) * xa
                    ypv = dual_step(ax(xb), y, sigma)
                    yn = w * (2 * ypv - y) + (one - w) * ya
                    x = np.where(live, xn, x)
                    y = np.where(live, yn, y)
                    continue
                # check step: the terms of pdhg.cuh, the decision, k_apply
                q = dict(dx2=((xpv - x) ** 2).sum(0), dxa2=((xpv - xa) ** 2).sum(0), pobj=(cs * xpv).sum(0))
                a, axx = ax(xb), ax(x)
                ypv = dual_step(a, y, sigma)
                dy, da = ypv - y, ypv - ya
                adx, axp = dt(0.5) * (a - axx), dt(0.5) * (a + axx)
                viol = np.where(axp < rls, rls - axp, np.where(axp > rus, axp - rus, zero)) * (one / st["sb"]) / dr
                q.update(dy2=(dy * dy).sum(0), dyadx=(dy * adx).sum(0), dya2=(da * da).sum(0),
                         pres2=(viol * viol).sum(0), dobj_row=_support(ypv, rls, rus).sum(0))
                rc = cs - aty(ypv)
                at_l, at_u = fin_lb & (xpv <= lbs), fin_ub & (xpv >= ubs)
                rpos = np.where(at_l, np.maximum(rc, zero), zero)
                rneg = np.where(at_u, np.minimum(rc, zero), zero)
                res = (rc - rpos - rneg) * (one / st["sc"]) / dc
                dcol = np.where(rpos > 0, lbs * rpos, zero) + np.where(rneg < 0, ubs * rneg, zero)
                q.update(dres2=(res * res).sum(0), dobj_col=dcol.sum(0))
                d = ypv - y
                d = np.where(inf_rl, np.minimum(d, zero), d)
                d = np.where(inf_ru, np.maximum(d, zero), d)
                atr = aty(d)
                q.update(ray_row=_support(d, rls, rus).sum(0), ray_max=np.abs(d * dr).max(0),
                         ray_col=_support(-atr, lbs, ubs).sum(0), kty_max=np.abs(atr / dc).max(0))
                # clamp ties feed the discrete at-bound tests of pdhg_rc_terms and k_finalize
                scale = np.maximum(one, np.abs(xpv).max(0))
                # g == 0 exactly (a column without cost or live rows) leaves x where it is in any arithmetic
                tie = ~fixed & (g != 0)
                gapl = np.where(fin_lb & tie, np.abs(v - lbs), dt(np.inf))
                gapu = np.where(fin_ub & tie, np.abs(v - ubs), dt(np.inf))
                cm = np.minimum(gapl, gapu).min(0) / scale
                rec = dict(j=j, it=it, k=np.full(B, -1), r=np.full(B, np.nan), rs2=np.full(B, np.nan),
                           omega=np.full(B, np.nan), flag=np.full(B, -1), status=np.full(B, -1))
                flags = np.zeros(B, np.int64)
                for s in np.flatnonzero(live):
                    mg.add("clamp", float(cm[s]), 0.0, 1.0)
                    qs = {key: val[s] for key, val in q.items()}
                    flags[s], rec["k"][s], r, rs2 = _decide(st, s, P, qs, j, steps, dt, mg)
                    rec["r"][s], rec["rs2"][s] = float(r), float(rs2)
                    rec["omega"][s], rec["flag"][s] = float(st["omega"][s]), flags[s]
                    rec["status"][s] = st["status"][s]
                trace.append(rec)
                hal = live & (flags == 0)
                frz = live & (flags > 0)
                xh = w * xb + (one - w) * xa
                yh = w * (2 * ypv - y) + (one - w) * ya
                x = np.where(hal, xh, np.where(frz, xpv, x))
                xa = np.where(frz, xpv, xa)
                y = np.where(hal, yh, np.where(frz, ypv, y))
                ya = np.where(frz, ypv, ya)
                xp_l = np.where(live, xpv, xp_l)
                rc_l = np.where(live, rc, rc_l)
                yp_l = np.where(live, ypv, yp_l)
            it += steps
        # ---- k_finalize
        status = np.where(st["status"] < 0, ITERATION_LIMIT, st["status"])
        at_l, at_u = fin_lb & (xp_l <= lbs), fin_ub & (xp_l >= ubs)
        xo = np.where(at_l, lb, np.where(at_u, ub, xp_l * dc * (one / st["sb"])))
        rcu = rc_l * (one / st["sc"]) / dc
        zl = np.where(at_l, np.maximum(rcu, zero), zero)
        zu = np.where(at_u, np.minimum(rcu, zero), zero)
        yo = yp_l * dr * (one / st["sc"])
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    return dict(status=status, iterations=st["total"].copy(), restarts=st["restarts"].copy(),
                objective=f64(st["pobj"]) + c0, dual_objective=f64(st["dobj"]) + c0, pres=f64(st["pres"]),
                dres=f64(st["dres"]), gap=f64(st["gap"]), pobj=f64(st["pobj"]), dobj=f64(st["dobj"]),
                nq_un=f64(st["nq_un"]), nc_un=f64(st["nc_un"]), x=f64(xo), y=f64(yo), zl=f64(zl), zu=f64(zu),
                trace=trace, margins=dict(mg.m), steps=steps)


def lane(lp, s):
    """Lane s of a batch as a one-lane batch."""
    return {k: (None if v is None else (v[s:s + 1] if k == "c0" else v[:, s:s + 1])) for k, v in lp.items()}


def lanes(lp, idx):
    idx = np.asarray(idx)
    return {k: (None if v is None else (v[idx] if k == "c0" else v[:, idx])) for k, v in lp.items()}


# =================================== LP generator ================================================================
def make_lp(n, m, B, seed, infeasible=False, max_row=9, spread=0.0):
    """A batch of B LPs on one pattern (per-lane values), feasible by construction around an interior x0.

    Row lengths 1..max_row (so the 4-, 2- and 1-term tails of spmv_row / spmv_row2 all occur); equality, range,
    lower-only and upper-only rows; row m-1 empty with bounds containing 0, row m-2 numerically empty (values
    1e-12 of the rest, below tiny_rel); column 0 free (pinned through the equality row 0), 1 fixed, 2 lower-only
    (cost > 0), 3 upper-only (cost < 0), n-1 empty (boxed); one duplicated (row, col) entry in row 2.
    infeasible: row 1 (boxed columns only) asks for more than its box allows; column 0 gets a box.
    spread > 0: lane s's matrix values are multiplied by (1 + spread * u) entrywise with u in [-1, 1] drawn
    with a lane-dependent spread, which spreads the conditioning (and the iteration counts) over the batch."""
    assert n >= 8 and m >= 5
    rng = np.random.default_rng(seed)
    special = {0, 2, 3, n - 1}
    boxed = np.array([j for j in range(n) if j not in special])
    inner = np.array([j for j in range(n - 1)])
    cols = []
    for i in range(m):
        if i == m - 1:
            cols.append(np.array([], np.int64))
            continue
        L = int(rng.integers(1, max_row + 1))
        if i in (0, 1):
            L = max(L, 2)
            pick = np.sort(rng.choice(boxed, size=min(L, len(boxed)), replace=False))
            if i == 0:
                pick = np.concatenate([[0], pick])
        else:
            pick = np.sort(rng.choice(inner, size=min(L, len(inner)), replace=False))
        if i == 2:
            pick = np.concatenate([pick[:1], pick])      # duplicated (row, col) entry
        cols.append(pick.astype(np.int64))
    row_ptr = np.concatenate([[0], np.cumsum([len(p) for p in cols])]).astype(np.int64)
    col_idx = np.concatenate(cols).astype(np.int64)
    pat = Pattern(n, m, row_ptr, col_idx)
    nnz = pat.nnz
    vals = rng.uniform(0.2, 2.0, (nnz, B)) * rng.choice([-1.0, 1.0], (nnz, B))
    if spread > 0:
        lane_s = spread * np.linspace(0.0, 1.0, B)
        vals *= 1.0 + lane_s * rng.uniform(-1.0, 1.0, (nnz, B)) * 0.9
        vals *= 10.0 ** (lane_s * rng.uniform(-1.0, 1.0, (nnz, B)))
    vals[pat.row_of == m - 2] *= 1e-12                    # numerically empty row
    x0 = rng.uniform(-1.0, 1.0, (n, B))
    lb = x0 - rng.uniform(0.5, 2.0, (n, B))
    ub = x0 + rng.uniform(0.5, 2.0, (n, B))
    lb[0], ub[0] = -np.inf, np.inf
    lb[1] = ub[1] = x0[1]
    ub[2] = np.inf
    lb[3] = -np.inf
    c = rng.standard_normal((n, B))
    c[2] = np.abs(c[2]) + 0.5
    c[3] = -np.abs(c[3]) - 0.5
    Kx0 = _seg(np.add, vals * x0[col_idx], row_ptr)
    kind = rng.integers(0, 4, m)                          # 0 equality, 1 range, 2 lower only, 3 upper only
    kind[0], kind[1], kind[m - 2], kind[m - 1] = 0, 1, 1, 1
    lo_gap, up_gap = rng.uniform(0.1, 1.0, (m, B)), rng.uniform(0.1, 1.0, (m, B))
    rl = np.where(kind[:, None] == 3, -np.inf, np.where(kind[:, None] == 0, Kx0, Kx0 - lo_gap))
    ru = np.where(kind[:, None] == 2, np.inf, np.where(kind[:, None] == 0, Kx0, Kx0 + up_gap))
    rl[m - 1], ru[m - 1] = -1.0, 2.0                      # empty row, bounds contain 0
    if infeasible:
        # a free column stops the Farkas test (its ray entry must vanish exactly): box it
        lb[0], ub[0] = x0[0] - 5.0, x0[0] + 5.0
        k0, k1 = row_ptr[1], row_ptr[2]
        v, j = vals[k0:k1], col_idx[k0:k1]
        rl[1] = np.maximum(v * lb[j], v * ub[j]).sum(axis=0) + 1.0
        ru[1] = np.inf
    c0 = rng.standard_normal(B)
    return pat, dict(vals=vals, c=c, lb=lb, ub=ub, rl=rl, ru=ru, c0=c0)


def scipy_matrix(pat, lp, s):
    """Lane s's matrix with duplicates summed (for HiGHS)."""
    import scipy.sparse as sp
    K = sp.csr_matrix((lp["vals"][:, s].copy(), pat.col_idx.copy(), pat.row_ptr.copy()), shape=(pat.m, pat.n))
    K.sum_duplicates()
    return K


def compare(got, ref, s_got, s_ref, iterations):
    """err / bar of every continuous quantity of one lane: x, y, zl, zu by the infinity norm relative to the
    reference's; pres, dres, gap against the termination test's denominators (or the value, when larger)."""
    out = {}
    for key in ("x", "y", "zl", "zu"):
        a, b = np.asarray(got[key])[:, s_got], np.asarray(ref[key])[:, s_ref]
        den = max(np.max(np.abs(b), initial=0.0), 1e-300)
        out[key] = float(np.max(np.abs(a - b), initial=0.0) / den) / bar(key, iterations)
    dens = dict(pres=1.0 + ref["nq_un"][s_ref], dres=1.0 + ref["nc_un"][s_ref],
                gap=1.0 + abs(ref["pobj"][s_ref]) + abs(ref["dobj"][s_ref]))
    for key, den in dens.items():
        den = max(den, abs(ref[key][s_ref]))      # far from the threshold (diverging iterates) the value's own size
        out[key] = float(abs(got[key][s_got] - ref[key][s_ref]) / den) / bar(key, iterations)
    return out


# =================================== the cases of the GPU tests ===================================================
# name -> make_lp arguments; the GPU file (tests/test_gpu_pdhg_engines.py) runs each with the listed check periods
# over the windows of `windows`, and tests/test_pdhg_reference_cpu.py asserts their margins clear the bars
CASES = {
    "b1": dict(n=12, m=10, B=1, seed=1),
    "b3": dict(n=12, m=10, B=3, seed=2),
    "b33": dict(n=14, m=11, B=33, seed=3),
    "b64": dict(n=14, m=11, B=64, seed=4),
    "b100": dict(n=12, m=10, B=100, seed=5),
    "infeasible": dict(n=12, m=10, B=4, seed=0, infeasible=True),
    "group5": dict(n=30, m=24, B=5, seed=6),
    "hybrid": dict(n=16, m=12, B=100, seed=18, spread=0.4),
    # n, m > 592: geo_for caps the grid of a 1024-wide batch, so every kernel loops grid-stride
    "wide": dict(n=700, m=650, B=1024, seed=8),
    # too large for a group of one block to keep the matrix in shared memory: values streamed from L2
    "big": dict(n=1200, m=1200, B=1, seed=9),
}
# (b33 and b100 at check periods 1 and 3 check every lane ~400 times: some check lands within the bars of a
# threshold; b64 covers those periods on k_primal2 / k_dual2)
CHECK_EVERY = {"b1": (1, 3, 64), "b3": (1, 3, 64), "b33": (64,), "b64": (1, 3, 64), "b100": (64,),
               "infeasible": (64,), "group5": (64, 300), "hybrid": (64,), "wide": (4,), "big": (64,)}
FULL_RUN = {"wide": False, "big": False}   # the reference would be too slow to run these to termination
# the tests' tolerance: at 1e-8 the bars (6e-10 of the denominators at 1000 iterations, times the factor 100 the
# margins must clear) are 6 % of the threshold itself, and some check of a 100-lane batch lands that close
TEST_PARAMS = dict(eps_rel=1e-6)


def case(name):
    kw = dict(CASES[name])
    n, m, B, seed = kw.pop("n"), kw.pop("m"), kw.pop("B"), kw.pop("seed")
    return make_lp(n, m, B, seed, **kw)


def random_start(name, seed=5):
    """A start (x [n, B], y [m, B]) for set_start: uniform in [-1, 1], so some y entries have the wrong sign for
    one-sided rows and must be projected."""
    pat, lp = case(name)
    rng = np.random.default_rng(seed)
    B = lp["vals"].shape[1]
    return rng.uniform(-1.0, 1.0, (pat.n, B)), rng.uniform(-1.0, 1.0, (pat.m, B))


def windows(full, steps):
    """Block counts to stop at: 1, 2, 3, the block of the first restart and the one after it (from the full run's
    trace); None = run to termination."""
    out = [1, 2, 3]
    for rec in full["trace"]:
        if (rec["flag"] == 1).any():
            b = rec["it"] // steps + 1
            out += [b, b + 1]
            break
    return sorted(set(out)) + [None]


def margin_quantity(name):
    """The bar a decision margin is measured against."""
    if name.startswith("opt_"):
        return name[4:]
    if name.startswith("restart_"):
        return "r"
    if name in ("farkas",) or name.startswith("weight_"):
        return "y"
    return "x"
