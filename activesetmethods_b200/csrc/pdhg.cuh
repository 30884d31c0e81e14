// The arithmetic of restarted, reflected Halpern PDHG, written once for its three schedules: the streaming kernels
// (lp_solver.cuh), the persistent group kernel (pdhg_group.cuh) and the row-partitioned kernels (lp_dist.cuh).
// The operators take and return scalars; each schedule keeps its own layout, loops and reduction order.  Engine 5
// hands a running LP from the streaming kernels to the group kernel, and the row-partitioned run is checked
// against the single-GPU iteration count: both rely on every schedule computing the same doubles here.
#pragma once
#include "util.cuh"

namespace asmb {

struct ScenState {
    double omega, omega0, eta, sb, sc;
    double nq_un, nc_un;
    double r0, r_prev, e_sum, e_prev;
    double pobj, dobj, pres, dres, gap;
    long long total;
    int k0;
    int restarts;
    int status;        // -1 while running, else ASM_LP_*
    int restart_flag;  // set by pdhg_decide, consumed by the apply step
};

struct DevParams {
    double eps_rel, eps_infeas;
    double b_suf, b_nec, b_art;
    double kp, ki, kd;
    double balance;
    int verbose;
};

// reduction slots of a check
enum {
    Q_DX2 = 0,   // sum (xp - x)^2
    Q_DXA2,      // sum (xp - xa)^2
    Q_POBJ,      // sum cs * xp
    Q_DY2,       // sum (yp - y)^2
    Q_DYADX,     // sum dy * A dx
    Q_DYA2,      // sum (yp - ya)^2
    Q_PRES2,     // unscaled primal residual^2
    Q_DOBJ_ROW,  // row part of the dual objective (scaled units)
    Q_DRES2,     // unscaled dual residual^2
    Q_DOBJ_COL,  // column part of the dual objective (scaled units)
    Q_RAY_ROW,   // Farkas: sum rl*ray+ + ru*ray-   (scaled units)
    Q_RAY_MAX,   // max |ray * dr|
    Q_RAY_COL,   // Farkas: box support of -(A'ray)
    Q_KTY_MAX,   // max |(A'ray)_j / dc_j|
    Q_COUNT
};
// bit i set: slot i is summed over the row side (else the column side); is a max (else a sum)
constexpr unsigned kQRows = (1u << Q_DY2) | (1u << Q_DYADX) | (1u << Q_DYA2) | (1u << Q_PRES2) | (1u << Q_DOBJ_ROW) |
                            (1u << Q_RAY_ROW) | (1u << Q_RAY_MAX);
constexpr unsigned kQMax = (1u << Q_RAY_MAX) | (1u << Q_KTY_MAX);

// ---- one iteration ---------------------------------------------------------------------------------------------
// Halpern weight of step k (k = 1, 2, ... since the last restart)
__device__ __forceinline__ double pdhg_halpern_weight(int k) { return (double)k / ((double)k + 1.0); }
// Halpern update towards the anchor: w r + (1 - w) anchor
__device__ __forceinline__ double pdhg_halpern(double w, double r, double anchor) { return w * r + (1.0 - w) * anchor; }
// reflection of the step z -> p: 2 p - z
__device__ __forceinline__ double pdhg_reflect(double p, double z) { return 2.0 * p - z; }
// primal step: projection of x - tau g on [lo, up], g = c - A'y
__device__ __forceinline__ double pdhg_primal_step(double x, double g, double tau, double lo, double up) {
    return fmin(fmax(x - tau * g, lo), up);
}
// dual step: with t = A xbar - y / sigma, yp = sigma (proj_[l,u](t) - t)
__device__ __forceinline__ double pdhg_dual_step(double a, double y, double sigma, double isig, double l, double u) {
    const double t = a - y * isig;
    return t < l ? sigma * (l - t) : (t > u ? sigma * (u - t) : 0.0);
}

// ---- check terms -----------------------------------------------------------------------------------------------
// support of [l, u] in direction x: l x for x > 0, u x for x < 0 (the unused side may be infinite)
__device__ __forceinline__ double pdhg_support(double x, double l, double u) {
    return x > 0.0 ? l * x : (x < 0.0 ? u * x : 0.0);
}
// column: move and primal objective of the step x -> xp (anchor xa, cost c)
__device__ __forceinline__ void pdhg_col_terms(double xp, double x, double xa, double c, double &dx2, double &dxa2,
                                               double &pobj) {
    const double dx = xp - x, da = xp - xa;
    dx2 += dx * dx;
    dxa2 += da * da;
    pobj += c * xp;
}
// row: move of the step y -> yp (anchor ya), dy' A dx, violation of A xp in unscaled units, row part of the dual
// objective; a = A xbar and ax = A x, so A dx = (a - ax) / 2 and A xp = (a + ax) / 2
__device__ __forceinline__ void pdhg_row_terms(double yp, double y, double ya, double a, double ax, double l, double u,
                                               double inv_sb, double dr, double &dy2, double &dyadx, double &dya2,
                                               double &pres2, double &dobj) {
    const double dy = yp - y, da = yp - ya;
    const double adx = 0.5 * (a - ax);
    const double axp = 0.5 * (a + ax);
    dy2 += dy * dy;
    dyadx += dy * adx;
    dya2 += da * da;
    const double viol = (axp < l ? l - axp : (axp > u ? axp - u : 0.0)) * inv_sb / dr;
    pres2 += viol * viol;
    dobj += pdhg_support(yp, l, u);
}
// reduced cost rc at xp: dual residual in unscaled units and column part of the dual objective; reduced costs count
// as multipliers only where the iterate sits on a finite bound
__device__ __forceinline__ void pdhg_rc_terms(double rc, double xp, double l, double u, double inv_sc, double dc,
                                              double &dres2, double &dobj) {
    const double rpos = (isfinite(l) && xp <= l) ? fmax(rc, 0.0) : 0.0;
    const double rneg = (isfinite(u) && xp >= u) ? fmin(rc, 0.0) : 0.0;
    const double res = (rc - rpos - rneg) * inv_sc / dc;
    dres2 += res * res;
    dobj += (rpos > 0.0 ? l * rpos : 0.0) + (rneg < 0.0 ? u * rneg : 0.0);
}
// Farkas ray from the iterate difference d = yp - y, projected on the sign cone of the infinite sides
__device__ __forceinline__ double pdhg_ray(double d, double l, double u) {
    if (!isfinite(l)) d = fmin(d, 0.0);
    if (!isfinite(u)) d = fmax(d, 0.0);
    return d;
}
// ray terms of a row (ray entry d) and of a column (a = (A'ray)_j): support of the bounds, largest unscaled entry
__device__ __forceinline__ void pdhg_ray_row_terms(double d, double l, double u, double dr, double &sum, double &mx) {
    sum += pdhg_support(d, l, u);
    mx = fmax(mx, fabs(d * dr));
}
__device__ __forceinline__ void pdhg_ray_col_terms(double a, double l, double u, double dc, double &sum, double &mx) {
    sum += pdhg_support(-a, l, u);  // support of the box in direction -(A'ray)
    mx = fmax(mx, fabs(a / dc));
}

// ---- start state and check decision ----------------------------------------------------------------------------
// scalars of the scaled problem from |c|^2 and |q|^2, scaled and unscaled (q: the finite row bounds)
__device__ __forceinline__ ScenState pdhg_start(double c2, double cun2, double q2, double qun2) {
    ScenState st;
    st.sb = 1.0 / (sqrt(q2) + 1.0);
    st.sc = 1.0 / (sqrt(c2) + 1.0);
    const double nc = sqrt(c2) * st.sc, nq = sqrt(q2) * st.sb;
    st.omega = (nc > 0.0 && nq > 0.0) ? nc / nq : 1.0;
    st.omega0 = st.omega;
    st.eta = 0.998;  // ||A||_2 <= 1 after Pock-Chambolle (alpha = 1) scaling
    st.nq_un = sqrt(qun2);
    st.nc_un = sqrt(cun2);
    st.r0 = 0.0;
    st.r_prev = INFINITY;
    st.e_sum = 0.0;
    st.e_prev = 0.0;
    st.pobj = st.dobj = 0.0;
    st.pres = st.dres = st.gap = INFINITY;
    st.total = 0;
    st.k0 = 0;
    st.restarts = 0;
    st.status = -1;
    st.restart_flag = 0;
    return st;
}

// one line of the check decision (kept out of line: its argument buffer would otherwise add to the callers' frames)
__device__ __noinline__ void pdhg_trace(const char *tag, long long total, int k, double pres, double dres, double gap,
                                        double pobj, double r, double omega, int restarts, int restart, double robj,
                                        double rrow, double rcol, double kty, double nr) {
    printf("[%s] it %lld k %d pres %.3e dres %.3e gap %.3e pobj %.10e r %.3e w %.3e restarts %d%s | ray: obj %.3e "
           "(row %.3e col %.3e) kty %.3e norm %.3e\n", tag, total, k, pres, dres, gap, pobj, r, omega, restarts,
           restart ? " R" : "", robj, rrow, rcol, kty, nr);
}

// Every scalar decision of the check at step jit of a block of `steps` iterations, from the completed sums q[Q_COUNT]:
// termination (optimal, infeasible, numerical error), restart, primal weight, and the k0 / total bookkeeping.
// restart_flag: 0 Halpern step, 1 restart, 2 freeze at (xp, yp).  With P.verbose, a non-null `tag` prints one line.
__device__ inline void pdhg_decide(ScenState &st, const DevParams &P, const double *q, int jit, int steps,
                                   const char *tag) {
    const double tau = st.eta / st.omega, sigma = st.eta * st.omega;
    const int k = st.k0 + jit + 1;
    const long long total = st.total + jit + 1;
    const double r2 = q[Q_DX2] / tau - 2.0 * q[Q_DYADX] + q[Q_DY2] / sigma;
    const double r = sqrt(fmax(r2, 0.0));
    const double unit = 1.0 / (st.sb * st.sc);
    const double pobj = q[Q_POBJ] * unit;
    const double dobj = (q[Q_DOBJ_ROW] + q[Q_DOBJ_COL]) * unit;
    const double pres = sqrt(q[Q_PRES2]), dres = sqrt(q[Q_DRES2]);
    const double gap = fabs(pobj - dobj);
    st.pobj = pobj;
    st.dobj = dobj;
    st.pres = pres;
    st.dres = dres;
    st.gap = gap;
    int status = -1;
    if (pres <= P.eps_rel * (1.0 + st.nq_un) && dres <= P.eps_rel * (1.0 + st.nc_un) &&
        gap <= P.eps_rel * (1.0 + fabs(pobj) + fabs(dobj)))
        status = ASM_LP_OPTIMAL;
    double robj = 0.0, kty = 0.0, nr = 0.0;
    if (status < 0) {
        // Farkas certificate: ray'rl+ + ray'ru- - max_box (K'ray)'x > 0  (all terms carry 1/(sb sc);
        // normalise by ||ray||_inf in unscaled units = Q_RAY_MAX / sc)
        nr = q[Q_RAY_MAX] / st.sc;
        if (nr > 0.0) {
            robj = (q[Q_RAY_ROW] + q[Q_RAY_COL]) * unit / nr;
            kty = q[Q_KTY_MAX] / st.sc / nr;
            if (robj > P.eps_infeas * fmax(1.0, kty)) status = ASM_LP_INFEASIBLE;
        }
    }
    if (!(r == r) || !(pobj == pobj)) status = ASM_LP_NUMERICAL_ERROR;
    int restart = 0;
    if (status < 0) {
        if (k == 1) {
            st.r0 = r;
        } else if (jit + 1 == steps) {
            if (r <= P.b_suf * st.r0)
                restart = 1;
            else if (r <= P.b_nec * st.r0 && r > st.r_prev)
                restart = 1;
            else if ((double)k >= P.b_art * (double)total)
                restart = 1;
        }
        st.r_prev = r;
        if (restart) {
            // primal weight: PID controller on log(omega * |dx| / |dy|); the default gains (0.5, 0, 0) are the
            // PDLP rule omega <- sqrt(omega * |dy| / |dx|).  Degenerate moves or a runaway weight fall back to
            // the initial one.
            const double ddx = sqrt(q[Q_DXA2]), ddy = sqrt(q[Q_DYA2]);
            const double rp = pres / (1.0 + st.nq_un), rd = dres / (1.0 + st.nc_un);
            if (P.balance > 0.0) {
                // residual balancing: a larger weight shortens the primal step and lengthens the dual one, which
                // drives the primal residual down faster -- move the weight towards equal relative residuals
                if (rp > 0.0 && rd > 0.0) st.omega = exp(log(st.omega) + P.balance * log(rp / rd));
            } else if (ddx > 1e-16 && ddy > 1e-16) {
                const double e = log(st.omega * ddx / ddy);
                st.e_sum += e;
                const double dlog = -(P.kp * e + P.ki * st.e_sum + P.kd * (e - st.e_prev));
                st.omega = exp(log(st.omega) + dlog);
                st.e_prev = e;
            }
            if (!(st.omega > st.omega0 * 1e-16 && st.omega < st.omega0 * 1e16)) {
                st.omega = st.omega0;
                st.e_sum = 0.0;
                st.e_prev = 0.0;
            }
            st.restarts += 1;
            st.r_prev = INFINITY;
        }
    }
    if (P.verbose && tag)
        pdhg_trace(tag, total, k, pres, dres, gap, pobj, r, st.omega, st.restarts, restart, robj, q[Q_RAY_ROW] * unit,
                   q[Q_RAY_COL] * unit, kty, nr);
    st.restart_flag = restart;
    if (jit + 1 == steps) {
        st.total += steps;
        st.k0 = restart ? 0 : st.k0 + steps;
    }
    if (status >= 0) {
        st.total = total;
        st.status = status;
        st.restart_flag = 2;
    }
}

// ---- host ------------------------------------------------------------------------------------------------------
inline DevParams dev_params(const asm_lp_params &P) {
    DevParams dp;
    dp.eps_rel = P.eps_rel;
    dp.eps_infeas = P.eps_infeas;
    dp.b_suf = P.restart_sufficient;
    dp.b_nec = P.restart_necessary;
    dp.b_art = P.restart_artificial;
    dp.kp = P.pid_kp;
    dp.ki = P.pid_ki;
    dp.kd = P.pid_kd;
    dp.balance = P.weight_balance;
    dp.verbose = P.verbose;
    return dp;
}
// the report of one finished LP; c0 is the objective constant
inline void lp_info(const ScenState &st, double c0, asm_lp_info &info) {
    info.status = st.status;
    info.restarts = st.restarts;
    info.iterations = st.total;
    info.objective = st.pobj + c0;
    info.dual_objective = st.dobj + c0;
    info.primal_residual = st.pres;
    info.dual_residual = st.dres;
    info.gap = st.gap;
}

}  // namespace asmb
