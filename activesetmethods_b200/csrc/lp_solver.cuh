// Restarted, reflected Halpern PDHG for   min c'x  s.t.  rl <= Kx <= ru,  lb <= x <= ub   on sm_100a.
//
// This is the component that stands where GLPK's simplex stands in the reference
// (MOI.optimize!(qp.model), /root/reference/src/algorithms/subproblem.jl:490).  Algorithm (literature,
// SURVEY.md App. F): Ruiz + Pock-Chambolle diagonal preconditioning, bound/objective rescaling, PDHG with
// reflection and Halpern anchoring, fixed-point-error restarts (sufficient / necessary / artificial),
// PID-controlled primal weight, KKT termination in the unscaled space, Farkas-ray infeasibility test.
//
// Kernels (all hand-written; B = batch, vectors element-major v[i*B+s]):
//   k_primal<CHECK>   CSC pass  A'y fused with the primal box projection, reflection and Halpern step
//   k_dual<CHECK>     CSR pass  A xbar fused with the dual prox and Halpern step
//   k_dual_resid      CSC pass  A'y+ for reduced costs / dual residual / dual objective   (check only)
//   k_ray_rows/cols   Farkas certificate pieces                                          (check only)
//   k_decide          one block per LP: deterministic second-stage reductions, then pdhg_decide (pdhg.cuh):
//                     termination, restart, PID
//   k_apply           restart or Halpern update after a check
//   k_ruiz_* / k_build_scaled / k_prepare_* / k_finalize   preconditioning and (un)scaling
// A solve launches a CUDA graph of `check_every` iterations per host round trip; the only host<->device
// traffic inside the loop is the 4-byte active counter.
#pragma once
#include <chrono>
#include <cstdlib>
#include <map>
#include <memory>

#include "pdhg.cuh"

namespace asmb {

constexpr int kPartialSlots = 16;  // rows of the partial buffer: Q_COUNT here, I_COUNT in ipm.cuh
// preparation slots (reuse the same partial buffer)
enum { P_C2 = 0, P_CUN2, P_Q2, P_QUN2, P_COUNT };

struct LpView {
    int n, m, B;
    int nbx_rows, nbx_cols;
    const int *row_ptr, *col_idx, *col_ptr, *row_idx, *csc_src;
    // unscaled data
    const double *vals, *c, *lb, *ub, *rl, *ru;
    // scaled data
    double *A, *AT, *dr, *dc, *sr, *scf, *cs, *lbs, *ubs, *rls, *rus;
    // iterates
    double *x, *xa, *xp, *xbar, *gy, *gyp;
    double *y, *ya, *yp, *ray;
    // results (unscaled)
    double *xo, *yo, *dlo, *dup;
    double *partials;
    const double *gmax;  // per LP: max |K_ij| (rows / columns below kTinyRel * gmax are treated as empty by the scaling)
    ScenState *state;
    const DevParams *prm;
    int *n_active;
};

// =================================== preconditioning ======================================================
// A row (column) whose largest coefficient is below kTinyRel times the largest of the matrix is numerically empty
// (SLP produces them: the gradient of p^2 + q^2 <= s^2 at p, q ~ 1e-11).  Equilibrating it would multiply its
// right-hand side by ~1e10 and wreck the bound / objective balance of the whole LP, so it keeps scale 1.
constexpr double kTinyRel = 1e-8;
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_absmax(LpView v, int64_t nnz) {
    Map<BATCH> mp;
    const int B = v.B;
    double acc[1] = {0.0};
    for (int64_t k = mp.first; k < nnz; k += mp.stride) acc[0] = fmax(acc[0], fabs(v.vals[k * B + mp.s]));
    block_reduce_store<BATCH, 1>(acc, 1u, v.partials, 0, B);
}
// out = matrix maximum times (tiny_rel / kTinyRel): the scaling kernels compare against kTinyRel * out
__global__ void __launch_bounds__(kFinalThreads) k_final_max(const double *partials, int nbx, int B, double *out,
                                                              double rel) {
    const double q = final_reduce(partials, 0, nbx, B, blockIdx.x, true);
    if (threadIdx.x == 0) out[blockIdx.x] = q * rel;
}
template <bool BATCH, bool SUM>
__global__ void __launch_bounds__(kThreads) k_ruiz_rows(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const double tiny = kTinyRel * v.gmax[mp.s];
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const double dri = v.dr[i * B + mp.s];
        double a = 0.0, a0 = 0.0;
        for (int k = v.row_ptr[i]; k < v.row_ptr[i + 1]; ++k) {
            const double val = v.vals[(int64_t)k * B + mp.s];
            double t = fabs(val * dri * v.dc[(int64_t)v.col_idx[k] * B + mp.s]);
            a = SUM ? a + t : fmax(a, t);
            a0 = fmax(a0, fabs(val));
        }
        v.sr[i * B + mp.s] = (a > 0.0 && a0 > tiny) ? 1.0 / sqrt(a) : 1.0;
    }
}
template <bool BATCH, bool SUM>
__global__ void __launch_bounds__(kThreads) k_ruiz_cols(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const double tiny = kTinyRel * v.gmax[mp.s];
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const double dcj = v.dc[j * B + mp.s];
        double a = 0.0, a0 = 0.0;
        for (int k = v.col_ptr[j]; k < v.col_ptr[j + 1]; ++k) {
            const double val = v.vals[(int64_t)v.csc_src[k] * B + mp.s];
            double t = fabs(val * v.dr[(int64_t)v.row_idx[k] * B + mp.s] * dcj);
            a = SUM ? a + t : fmax(a, t);
            a0 = fmax(a0, fabs(val));
        }
        v.scf[j * B + mp.s] = (a > 0.0 && a0 > tiny) ? 1.0 / sqrt(a) : 1.0;
    }
}
__global__ void k_mul_inplace(double *__restrict__ a, const double *__restrict__ b, int64_t n) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
        a[t] *= b[t];
}
__global__ void k_fill(double *__restrict__ a, double val, int64_t n) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
        a[t] = val;
}
// scaled matrix in both orders; the product is formed identically so A and AT hold the same doubles
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_build_scaled_csr(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const double dri = v.dr[i * B + mp.s];
        for (int k = v.row_ptr[i]; k < v.row_ptr[i + 1]; ++k)
            v.A[(int64_t)k * B + mp.s] = v.vals[(int64_t)k * B + mp.s] * dri * v.dc[(int64_t)v.col_idx[k] * B + mp.s];
    }
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_build_scaled_csc(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const double dcj = v.dc[j * B + mp.s];
        for (int k = v.col_ptr[j]; k < v.col_ptr[j + 1]; ++k)
            v.AT[(int64_t)k * B + mp.s] =
                v.vals[(int64_t)v.csc_src[k] * B + mp.s] * v.dr[(int64_t)v.row_idx[k] * B + mp.s] * dcj;
    }
}

// first pass over the vectors: diagonal scaling + the norms that define sb, sc, omega0 and the
// termination denominators
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_prepare_cols(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    double acc[2] = {0.0, 0.0};
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double d = v.dc[e], cj = v.c[e];
        const double c0 = cj * d;
        v.cs[e] = c0;
        v.lbs[e] = v.lb[e] / d;
        v.ubs[e] = v.ub[e] / d;
        acc[0] += c0 * c0;
        acc[1] += cj * cj;
    }
    block_reduce_store<BATCH, 2>(acc, 0u, v.partials, P_C2, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_prepare_rows(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    double q2 = 0.0, qun2 = 0.0;
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        const double d = v.dr[e], l = v.rl[e], u = v.ru[e];
        const double ls = l * d, us = u * d;
        v.rls[e] = ls;
        v.rus[e] = us;
        if (isfinite(l)) {
            q2 += ls * ls;
            qun2 += l * l;
        }
        if (isfinite(u) && u != l) {
            q2 += us * us;
            qun2 += u * u;
        }
    }
    double acc[2] = {q2, qun2};
    block_reduce_store<BATCH, 2>(acc, 0u, v.partials, P_Q2, B);
}
// one block per scenario: scalars of the scaled problem
__global__ void __launch_bounds__(kFinalThreads) k_init_state(LpView v) {
    const int s = blockIdx.x, B = v.B;
    double c2 = final_reduce(v.partials, P_C2, v.nbx_cols, B, s, false);
    double cun2 = final_reduce(v.partials, P_CUN2, v.nbx_cols, B, s, false);
    double q2 = final_reduce(v.partials, P_Q2, v.nbx_rows, B, s, false);
    double qun2 = final_reduce(v.partials, P_QUN2, v.nbx_rows, B, s, false);
    if (threadIdx.x == 0) v.state[s] = pdhg_start(c2, cun2, q2, qun2);
}
// second pass: bound/objective rescaling and the starting point (x0, y0 are unscaled warm starts or 0)
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_prepare_finish(LpView v, int warm_all, const int *__restrict__ prev_ok) {
    Map<BATCH> mp;
    const int B = v.B;
    // a scenario is warm-started only from an OPTIMAL previous solve or a start the caller set (LpSolver::start_ok):
    // after INFEASIBLE the stored duals are a growing Farkas direction, after an iteration limit an unconverged point
    const int warm = (warm_all && (!prev_ok || prev_ok[mp.s])) ? warm_all : 0;
    const double sb = v.state[mp.s].sb, sc = v.state[mp.s].sc;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        v.cs[e] *= sc;
        const double l = v.lbs[e] * sb, u = v.ubs[e] * sb;
        v.lbs[e] = l;
        v.ubs[e] = u;
        double x0 = warm == 1 ? v.xo[e] / v.dc[e] * sb : 0.0;   // warm == 2: duals only
        x0 = fmin(fmax(x0, l), u);
        v.x[e] = x0;
        v.xa[e] = x0;
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        v.rls[e] *= sb;
        v.rus[e] *= sb;
        double y0 = warm ? v.yo[e] / v.dr[e] * sc : 0.0;
        if (!isfinite(v.rl[e])) y0 = fmin(y0, 0.0);
        if (!isfinite(v.ru[e])) y0 = fmax(y0, 0.0);
        v.y[e] = y0;
        v.ya[e] = y0;
    }
}

// =================================== PDHG iteration ========================================================
// sum_k val[k] * vec[idx[k]] over [k0, k1) of one scenario lane, four entries in flight at a time; the adds keep
// the sequential order, so the result is bit-identical to the plain loop.
__device__ __forceinline__ double spmv_row(const double *__restrict__ val, const int *__restrict__ idx,
                                           const double *__restrict__ vec, int k0, int k1, int B, int s) {
    double a = 0.0;
    int k = k0;
    for (; k + 4 <= k1; k += 4) {
        const int i0 = idx[k], i1 = idx[k + 1], i2 = idx[k + 2], i3 = idx[k + 3];
        const double a0 = val[(int64_t)k * B + s], a1 = val[(int64_t)(k + 1) * B + s],
                     a2 = val[(int64_t)(k + 2) * B + s], a3 = val[(int64_t)(k + 3) * B + s];
        const double x0 = vec[(int64_t)i0 * B + s], x1 = vec[(int64_t)i1 * B + s], x2 = vec[(int64_t)i2 * B + s],
                     x3 = vec[(int64_t)i3 * B + s];
        a += a0 * x0;
        a += a1 * x1;
        a += a2 * x2;
        a += a3 * x3;
    }
    if (k + 2 <= k1) {
        const int i0 = idx[k], i1 = idx[k + 1];
        const double a0 = val[(int64_t)k * B + s], a1 = val[(int64_t)(k + 1) * B + s];
        const double x0 = vec[(int64_t)i0 * B + s], x1 = vec[(int64_t)i1 * B + s];
        a += a0 * x0;
        a += a1 * x1;
        k += 2;
    }
    if (k < k1) a += val[(int64_t)k * B + s] * vec[(int64_t)idx[k] * B + s];
    return a;
}

// Primal half: g = cs - A'y ; xp = proj_box(x - tau g) ; xbar = 2 xp - x ; Halpern x <- w xbar + (1-w) xa.
// CHECK: keep xp, g and xbar, leave x untouched (k_apply finishes the step after the restart decision).
template <bool BATCH, bool CHECK>
__global__ void __launch_bounds__(kThreads) k_primal(LpView v, int jit) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const bool live = st->status < 0;
    const double tau = live ? st->eta / st->omega : 0.0;
    const double w = pdhg_halpern_weight(st->k0 + jit + 1);
    double acc[3] = {0.0, 0.0, 0.0};
    if (live) {
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            const int k1 = v.col_ptr[j + 1];
            int k = v.col_ptr[j];
            // the column's own operands first: their loads overlap the gather chain below (the kernel is bound by
            // bytes in flight per SM, not by issue)
            const double cj = v.cs[e], xv = v.x[e], lo = v.lbs[e], up = v.ubs[e];
            const double xav = CHECK ? 0.0 : v.xa[e];
            const double a = spmv_row(v.AT, v.row_idx, v.y, k, k1, B, mp.s);
            const double g = cj - a;
            const double xpv = pdhg_primal_step(xv, g, tau, lo, up);
            const double xb = pdhg_reflect(xpv, xv);
            v.xbar[e] = xb;
            if (CHECK) {
                v.xp[e] = xpv;
                v.gy[e] = g;
                pdhg_col_terms(xpv, xv, v.xa[e], cj, acc[0], acc[1], acc[2]);
            } else {
                v.x[e] = pdhg_halpern(w, xb, xav);
            }
        }
    }
    if (CHECK) block_reduce_store<BATCH, 3>(acc, 0u, v.partials, Q_DX2, B);
}

// Dual half: t = A xbar - y/sigma ; yp = sigma (proj_[rl,ru](t) - t) ; Halpern y <- w (2 yp - y) + (1-w) ya.
template <bool BATCH, bool CHECK>
__global__ void __launch_bounds__(kThreads) k_dual(LpView v, int jit) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const bool live = st->status < 0;
    const double sigma = live ? st->eta * st->omega : 1.0;
    const double isig = 1.0 / sigma;
    const double w = pdhg_halpern_weight(st->k0 + jit + 1);
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (live) {
        const double inv_sb = 1.0 / st->sb;
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            double a = 0.0, ax = 0.0;
            const int k1 = v.row_ptr[i + 1];
            const int k0 = v.row_ptr[i];
            const double yv = v.y[e], l = v.rls[e], u = v.rus[e];
            const double yav = CHECK ? 0.0 : v.ya[e];
            if (CHECK) {
                for (int k = k0; k < k1; ++k) {
                    const double av = v.A[(int64_t)k * B + mp.s];
                    const int64_t ce = (int64_t)v.col_idx[k] * B + mp.s;
                    a += av * v.xbar[ce];
                    ax += av * v.x[ce];
                }
            } else {
                a = spmv_row(v.A, v.col_idx, v.xbar, k0, k1, B, mp.s);
            }
            const double ypv = pdhg_dual_step(a, yv, sigma, isig, l, u);
            if (CHECK) {
                v.yp[e] = ypv;
                pdhg_row_terms(ypv, yv, v.ya[e], a, ax, l, u, inv_sb, v.dr[e], acc[0], acc[1], acc[2], acc[3], acc[4]);
            } else {
                v.y[e] = pdhg_halpern(w, pdhg_reflect(ypv, yv), yav);
            }
        }
    }
    if (CHECK) block_reduce_store<BATCH, 5>(acc, 0u, v.partials, Q_DY2, B);
}

// ---- two scenarios per lane (B % 64 == 0): the plain half iterations are bound by the bytes a warp keeps in
// flight along its dependent chain (pointer -> index -> gather), so every lane loads 16 bytes (scenarios 2t, 2t+1
// are adjacent in the element-major layout) and a warp moves 512 B per load.  Loads are never gated on the
// scenario's status; only the stores are.  grid (rows / 8, B / 64), block 256.
struct Lane2 {
    int s0;  // first scenario of the lane
    int64_t first, stride;
    __device__ __forceinline__ Lane2() {
        s0 = (blockIdx.y * 32 + (threadIdx.x & 31)) * 2;
        first = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
        stride = (int64_t)gridDim.x * kWarps;
    }
};
__device__ __forceinline__ double2 ld2(const double *p, int64_t row, int B, int s0) {
    return *reinterpret_cast<const double2 *>(p + row * B + s0);
}
__device__ __forceinline__ void st2(double *p, int64_t row, int B, int s0, double a, double b, bool la, bool lb) {
    if (la && lb)
        *reinterpret_cast<double2 *>(p + row * B + s0) = make_double2(a, b);
    else if (la)
        p[row * B + s0] = a;
    else if (lb)
        p[row * B + s0 + 1] = b;
}
__device__ __forceinline__ double2 spmv_row2(const double *__restrict__ val, const int *__restrict__ idx,
                                             const double *__restrict__ vec, int k0, int k1, int B, int s0) {
    double ax = 0.0, ay = 0.0;
    int k = k0;
    for (; k + 4 <= k1; k += 4) {
        const int i0 = idx[k], i1 = idx[k + 1], i2 = idx[k + 2], i3 = idx[k + 3];
        const double2 a0 = ld2(val, k, B, s0), a1 = ld2(val, k + 1, B, s0), a2 = ld2(val, k + 2, B, s0),
                      a3 = ld2(val, k + 3, B, s0);
        const double2 x0 = ld2(vec, i0, B, s0), x1 = ld2(vec, i1, B, s0), x2 = ld2(vec, i2, B, s0),
                      x3 = ld2(vec, i3, B, s0);
        ax += a0.x * x0.x; ay += a0.y * x0.y;
        ax += a1.x * x1.x; ay += a1.y * x1.y;
        ax += a2.x * x2.x; ay += a2.y * x2.y;
        ax += a3.x * x3.x; ay += a3.y * x3.y;
    }
    for (; k < k1; ++k) {
        const double2 a0 = ld2(val, k, B, s0), x0 = ld2(vec, idx[k], B, s0);
        ax += a0.x * x0.x;
        ay += a0.y * x0.y;
    }
    return make_double2(ax, ay);
}
__global__ void __launch_bounds__(kThreads) k_primal2(LpView v, int jit) {
    Lane2 mp;
    const int B = v.B, s0 = mp.s0;
    const ScenState *sa = v.state + s0, *sb = sa + 1;
    const bool la = sa->status < 0, lb = sb->status < 0;
    const double ta = sa->eta / sa->omega, tb = sb->eta / sb->omega;
    const double wa = pdhg_halpern_weight(sa->k0 + jit + 1), wb = pdhg_halpern_weight(sb->k0 + jit + 1);
    if (!__any_sync(0xffffffffu, la || lb)) return;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int k0 = v.col_ptr[j], k1 = v.col_ptr[j + 1];
        const double2 c = ld2(v.cs, j, B, s0), x = ld2(v.x, j, B, s0), lo = ld2(v.lbs, j, B, s0),
                      up = ld2(v.ubs, j, B, s0), xa = ld2(v.xa, j, B, s0);
        const double2 a = spmv_row2(v.AT, v.row_idx, v.y, k0, k1, B, s0);
        const double pa = pdhg_primal_step(x.x, c.x - a.x, ta, lo.x, up.x);
        const double pb = pdhg_primal_step(x.y, c.y - a.y, tb, lo.y, up.y);
        const double ba = pdhg_reflect(pa, x.x), bb = pdhg_reflect(pb, x.y);
        st2(v.xbar, j, B, s0, ba, bb, la, lb);
        st2(v.x, j, B, s0, pdhg_halpern(wa, ba, xa.x), pdhg_halpern(wb, bb, xa.y), la, lb);
    }
}
__global__ void __launch_bounds__(kThreads) k_dual2(LpView v, int jit) {
    Lane2 mp;
    const int B = v.B, s0 = mp.s0;
    const ScenState *sa = v.state + s0, *sb = sa + 1;
    const bool la = sa->status < 0, lb = sb->status < 0;
    const double ga = la ? sa->eta * sa->omega : 1.0, gb = lb ? sb->eta * sb->omega : 1.0;
    const double ia = 1.0 / ga, ib = 1.0 / gb;
    const double wa = pdhg_halpern_weight(sa->k0 + jit + 1), wb = pdhg_halpern_weight(sb->k0 + jit + 1);
    if (!__any_sync(0xffffffffu, la || lb)) return;
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int k0 = v.row_ptr[i], k1 = v.row_ptr[i + 1];
        const double2 y = ld2(v.y, i, B, s0), l = ld2(v.rls, i, B, s0), u = ld2(v.rus, i, B, s0),
                      ya = ld2(v.ya, i, B, s0);
        const double2 a = spmv_row2(v.A, v.col_idx, v.xbar, k0, k1, B, s0);
        const double pa = pdhg_dual_step(a.x, y.x, ga, ia, l.x, u.x);
        const double pb = pdhg_dual_step(a.y, y.y, gb, ib, l.y, u.y);
        st2(v.y, i, B, s0, pdhg_halpern(wa, pdhg_reflect(pa, y.x), ya.x), pdhg_halpern(wb, pdhg_reflect(pb, y.y), ya.y),
            la, lb);
    }
}

// Reduced costs of (xp, yp):  rc = cs - A'yp ; dual residual and column part of the dual objective.
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_dual_resid(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const bool live = st->status < 0;
    double acc[2] = {0.0, 0.0};
    if (live) {
        const double inv_sc = 1.0 / st->sc;
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            double a = 0.0;
            const int k1 = v.col_ptr[j + 1];
            for (int k = v.col_ptr[j]; k < k1; ++k)
                a += v.AT[(int64_t)k * B + mp.s] * v.yp[(int64_t)v.row_idx[k] * B + mp.s];
            const double rc = v.cs[e] - a;
            v.gyp[e] = rc;
            pdhg_rc_terms(rc, v.xp[e], v.lbs[e], v.ubs[e], inv_sc, v.dc[e], acc[0], acc[1]);
        }
    }
    block_reduce_store<BATCH, 2>(acc, 0u, v.partials, Q_DRES2, B);
}

// Farkas ray from the iterate difference dy = yp - y, projected on the sign cone of the infinite sides.
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ray_rows(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};
    if (live) {
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            const double l = v.rls[e], u = v.rus[e];
            const double d = pdhg_ray(v.yp[e] - v.y[e], l, u);
            v.ray[e] = d;
            pdhg_ray_row_terms(d, l, u, v.dr[e], acc[0], acc[1]);
        }
    }
    block_reduce_store<BATCH, 2>(acc, 2u, v.partials, Q_RAY_ROW, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ray_cols(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};
    if (live) {
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            double a = 0.0;
            const int k1 = v.col_ptr[j + 1];
            for (int k = v.col_ptr[j]; k < k1; ++k)
                a += v.AT[(int64_t)k * B + mp.s] * v.ray[(int64_t)v.row_idx[k] * B + mp.s];
            pdhg_ray_col_terms(a, v.lbs[e], v.ubs[e], v.dc[e], acc[0], acc[1]);
        }
    }
    block_reduce_store<BATCH, 2>(acc, 2u, v.partials, Q_RAY_COL, B);
}

// One block per LP: finish the reductions and take every scalar decision of the check.
__global__ void __launch_bounds__(kFinalThreads) k_decide(LpView v, int jit, int steps_in_graph) {
    const int s = blockIdx.x, B = v.B;
    ScenState *sp = v.state + s;
    if (sp->status >= 0) return;  // uniform per block
    double q[Q_COUNT];
    for (int i = 0; i < Q_COUNT; ++i)
        q[i] = final_reduce(v.partials, i, ((kQRows >> i) & 1u) ? v.nbx_rows : v.nbx_cols, B, s, (kQMax >> i) & 1u);
    if (threadIdx.x != 0) return;
    ScenState st = *sp;
    const DevParams P = *v.prm;
    pdhg_decide(st, P, q, jit, steps_in_graph, s == 0 ? "pdhg" : nullptr);
    if (st.status >= 0) atomicSub(v.n_active, 1);
    *sp = st;
}

// After a check: restart or freeze (x = xa = xp, y = ya = yp), else complete the Halpern step with the w of
// that step (kstep[s] = k of the step, stored before k_decide advanced k0).
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_apply(LpView v, const int *__restrict__ kstep) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const int flag = st->restart_flag;
    if (st->status >= 0 && flag != 2) return;
    const double w = pdhg_halpern_weight(kstep[mp.s]);
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        if (flag) {
            const double t = v.xp[e];
            v.x[e] = t;
            v.xa[e] = t;
        } else {
            v.x[e] = pdhg_halpern(w, v.xbar[e], v.xa[e]);
        }
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        if (flag) {
            const double t = v.yp[e];
            v.y[e] = t;
            v.ya[e] = t;
        } else {
            v.y[e] = pdhg_halpern(w, pdhg_reflect(v.yp[e], v.y[e]), v.ya[e]);
        }
    }
}
// scenarios that finished at this check are frozen exactly once
__global__ void k_after_apply(ScenState *st, int B) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < B && st[s].status >= 0 && st[s].restart_flag == 2) st[s].restart_flag = 3;
}
__global__ void k_store_kstep(const ScenState *st, int *kstep, int jit, int B) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < B) kstep[s] = st[s].k0 + jit + 1;
}
__global__ void k_mark_padding(ScenState *st, int Buser, int B) {
    int s = Buser + blockIdx.x * blockDim.x + threadIdx.x;
    if (s < B) st[s].status = ASM_LP_OPTIMAL;
}

// scenarios masked out of this solve (asm_slp_set_active): never live
__global__ void k_apply_mask(ScenState *st, const int *active, int Buser) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < Buser && !active[s]) {
        st[s].status = ASM_LP_SKIPPED;
        st[s].total = 0;
        st[s].pobj = st[s].dobj = st[s].pres = st[s].dres = st[s].gap = 0.0;
    }
}

// unscale the final iterate; bound duals from the reduced costs of the last check
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_finalize(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const double inv_sb = 1.0 / st->sb, inv_sc = 1.0 / st->sc;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double xs = v.xp[e], l = v.lbs[e], u = v.ubs[e];
        const bool at_l = isfinite(l) && xs <= l, at_u = isfinite(u) && xs >= u;
        // on a bound return the caller's bound itself so that exact comparisons (subproblem.jl:522-529) hold
        v.xo[e] = at_l ? v.lb[e] : (at_u ? v.ub[e] : xs * v.dc[e] * inv_sb);
        const double rc = v.gyp[e] * inv_sc / v.dc[e];
        v.dlo[e] = at_l ? fmax(rc, 0.0) : 0.0;
        v.dup[e] = at_u ? fmin(rc, 0.0) : 0.0;
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        v.yo[e] = v.yp[e] * v.dr[e] * inv_sc;
    }
}

}  // namespace asmb
#include "pdhg_group.cuh"
#include "ipm.cuh"
namespace asmb {

// ---- live-set compaction of a streaming batch ------------------------------------------------------------------
// dst[i * Bd + t] = src[i * Bs + map[t]] (t < cnt; padding lanes copy map[0]) and the reverse scatter
__global__ void k_gather_cols(const double *__restrict__ src, double *__restrict__ dst, int64_t rows, int Bs, int Bd,
                              const int *__restrict__ map, int cnt) {
    const int64_t total = rows * Bd;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / Bd;
        const int t = (int)(e - i * Bd);
        dst[e] = src[i * Bs + map[t < cnt ? t : 0]];
    }
}
__global__ void k_scatter_cols(const double *__restrict__ src, double *__restrict__ dst, int64_t rows, int Bs, int Bd,
                               const int *__restrict__ map, int cnt) {
    const int64_t total = rows * cnt;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / cnt;
        const int t = (int)(e - i * cnt);
        dst[i * Bd + map[t]] = src[i * Bs + t];
    }
}
__global__ void k_gather_state(const ScenState *src, ScenState *dst, const int *map, int cnt, int Bd) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= Bd) return;
    ScenState st = src[map[t < cnt ? t : 0]];
    if (t >= cnt) st.status = ASM_LP_OPTIMAL;  // padding lane: never live
    dst[t] = st;
}
__global__ void k_scatter_state(const ScenState *src, ScenState *dst, const int *map, int cnt) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < cnt) dst[map[t]] = src[t];
}

// ================================================================================================================
#define ASM_KL(...)      \
    do {                 \
        __VA_ARGS__;     \
        ++launches;      \
    } while (0)
// launch the <BATCH> instantiation that matches this handle
#define ASM_KB(kern, geo, ...)                                                    \
    do {                                                                          \
        if (B > 1)                                                                \
            kern<true><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__);      \
        else                                                                      \
            kern<false><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__);     \
        ++launches;                                                               \
    } while (0)
#define ASM_KB2(kern, flag, geo, ...)                                                   \
    do {                                                                                \
        if (B > 1)                                                                      \
            kern<true, flag><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__);      \
        else                                                                            \
            kern<false, flag><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__);     \
        ++launches;                                                                     \
    } while (0)

class LpSolver {
   public:
    int n = 0, m = 0, B = 1, Buser = 1;
    int64_t nnz = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int device = 0;   // the device this handle lives on (current at init)
    // pattern
    DBuf<int> row_ptr, col_idx, col_ptr, row_idx, csc_src;
    std::vector<int> h_row_ptr, h_col_idx, h_col_ptr, h_row_idx, h_csc_src;
    std::map<int, std::unique_ptr<GroupPlan>> plans;  // persistent group engine (pdhg_group.cuh), by group size
    std::map<int, std::pair<size_t, int>> feas;       // group size -> (shared memory bytes, matrix resident)
    GroupPlan *plan = nullptr;
    // live-set compaction (streaming engine): when half of the batch has converged the running LPs are copied
    // into a narrower working set so that no bandwidth is spent on finished ones
    struct WorkSet {
        DBuf<double> A, AT, cs, lbs, ubs, rls, rus, x, xa, xp, xbar, gy, gyp, y, ya, yp, ray, dr, dc, lb, ub, xo, yo, dlo, dup;
        DBuf<ScenState> state;
        DBuf<int> orig;
        std::vector<int> h_orig;  // position in the home batch
        int cap = 0, B = 0, live = 0;
    };
    WorkSet wsets[2];
    WorkSet *cur = nullptr;  // active compact set (nullptr: the home arrays)
    int homeB = 0, homeBuser = 0;
    int compactions = 0;
    int last_engine = 0, last_G = 0, last_groups = 0;
    // per scenario: xo / yo hold a start the next warm PDHG solve may use -- set by asm_lp_set_start and by an OPTIMAL
    // solve, cleared by any other outcome (a Farkas direction or an unconverged point) and by forget_warm_start
    std::vector<int> start_ok;
    DBuf<int> d_prev_ok;              // start_ok on the device (gates k_prepare_finish)
    DBuf<int> d_active;               // asm_slp_set_active: mask of the scenarios the next solves work on
    int n_masked = -1;                // number of active scenarios of the mask; -1 = no mask
    std::unique_ptr<IpmEngine> ipm;   // barrier engine (ipm.cuh), built at the first solve that uses it
    int ipm_failed = 0;               // symbolic analysis refused this pattern: engine 0 stays on PDHG
    // data (unscaled, element-major)
    DBuf<double> vals, c, lb, ub, rl, ru, c0;
    DBuf<double> A, AT, dr, dc, sr, scf, cs, lbs, ubs, rls, rus;
    DBuf<double> x, xa, xp, xbar, gy, gyp, y, ya, yp, ray;
    DBuf<double> xo, yo, dlo, dup, partials, gmax;
    DBuf<ScenState> state;
    DBuf<DevParams> prm;
    DBuf<int> n_active, kstep;
    Pinned pin_flag;
    std::vector<ScenState> host_state;
    cudaGraphExec_t graph_exec = nullptr;
    int graph_steps = 0;
    int64_t launches_per_graph = 0;
    bool has_solution = false;
    int64_t launches = 0;
    double last_loop_ms = 0.0;
    int64_t last_iters = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    ~LpSolver() {
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (own_stream && stream) cudaStreamDestroy(stream);
    }

    // pattern: 0-based CSR with int64 row_ptr on the host
    int init(int n_, int m_, int64_t nnz_, const int64_t *rp64, const int32_t *h_ci, int batch, cudaStream_t st) {
        n = n_;
        m = m_;
        nnz = nnz_;
        Buser = batch;
        B = pad_batch(batch);
        if (n <= 0 || m < 0 || nnz < 0 || batch < 1) return fail(ASM_E_INVALID, "bad LP dimensions");
        ASM_CK(cudaGetDevice(&device));
        if (nnz > 0x7fffffffLL) return fail(ASM_E_INVALID, "nnz exceeds 2^31-1");
        if (rp64[0] != 0 || rp64[m] != nnz) return fail(ASM_E_INVALID, "row_ptr does not match nnz");
        if (st) {
            stream = st;
        } else {
            ASM_CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
            own_stream = true;
        }
        ASM_CK(cudaEventCreate(&ev0));
        ASM_CK(cudaEventCreate(&ev1));
        // host CSC + map CSC position -> CSR position
        h_row_ptr.resize(m + 1);
        h_col_idx.resize(nnz);
        h_col_ptr.assign(n + 1, 0);
        h_row_idx.resize(nnz);
        h_csc_src.resize(nnz);
        std::vector<int> &cp = h_col_ptr, &ri = h_row_idx, &src = h_csc_src;
        for (int i = 0; i <= m; ++i) {
            h_row_ptr[i] = (int)rp64[i];
            if (i && rp64[i] < rp64[i - 1]) return fail(ASM_E_INVALID, "row_ptr not monotone");
        }
        for (int64_t k = 0; k < nnz; ++k) {
            if (h_ci[k] < 0 || h_ci[k] >= n) return fail(ASM_E_INVALID, "column index out of range");
            h_col_idx[k] = h_ci[k];
            cp[h_ci[k] + 1]++;
        }
        for (int j = 0; j < n; ++j) cp[j + 1] += cp[j];
        {
            std::vector<int> cur(cp.begin(), cp.end() - 1);
            for (int i = 0; i < m; ++i)
                for (int k = h_row_ptr[i]; k < h_row_ptr[i + 1]; ++k) {
                    int pos = cur[h_col_idx[k]]++;
                    ri[pos] = i;
                    src[pos] = k;
                }
        }
        ASM_TRY(row_ptr.alloc(m + 1));
        ASM_TRY(col_idx.alloc(nnz));
        ASM_TRY(col_ptr.alloc(n + 1));
        ASM_TRY(row_idx.alloc(nnz));
        ASM_TRY(csc_src.alloc(nnz));
        ASM_CK(cudaMemcpy(row_ptr.p, h_row_ptr.data(), (m + 1) * sizeof(int), cudaMemcpyHostToDevice));
        if (nnz) {
            ASM_CK(cudaMemcpy(col_idx.p, h_col_idx.data(), nnz * sizeof(int), cudaMemcpyHostToDevice));
            ASM_CK(cudaMemcpy(row_idx.p, ri.data(), nnz * sizeof(int), cudaMemcpyHostToDevice));
            ASM_CK(cudaMemcpy(csc_src.p, src.data(), nnz * sizeof(int), cudaMemcpyHostToDevice));
        }
        ASM_CK(cudaMemcpy(col_ptr.p, cp.data(), (n + 1) * sizeof(int), cudaMemcpyHostToDevice));
        const size_t nB = (size_t)n * B, mB = (size_t)m * B, zB = (size_t)nnz * B;
        DBuf<double> *colv[] = {&c, &lb, &ub, &dc, &scf, &cs, &lbs, &ubs, &x, &xa, &xp, &xbar, &gy, &gyp, &xo, &dlo, &dup};
        for (auto *b : colv) ASM_TRY(b->alloc(nB));
        DBuf<double> *rowv[] = {&rl, &ru, &dr, &sr, &rls, &rus, &y, &ya, &yp, &ray, &yo};
        for (auto *b : rowv) ASM_TRY(b->alloc(mB));
        ASM_TRY(vals.alloc(zB));
        ASM_TRY(A.alloc(zB));
        ASM_TRY(AT.alloc(zB));
        ASM_TRY(c0.alloc(B));
        ASM_TRY(partials.alloc((size_t)kPartialSlots * kMaxBlocksX * B));
        ASM_TRY(gmax.alloc(B));
        ASM_TRY(state.alloc(B));
        ASM_TRY(prm.alloc(1));
        ASM_TRY(n_active.alloc(2));   // [0] running LPs, [1] barrier engine: inexact Newton steps seen
        ASM_TRY(kstep.alloc(B));
        ASM_TRY(pin_flag.reserve(64));
        host_state.resize(B);
        start_ok.assign(B, 0);
        ASM_TRY(c0.zero(stream));
        ASM_TRY(xo.zero(stream));
        ASM_TRY(yo.zero(stream));
        ASM_TRY(vals.zero(stream));
        ASM_TRY(partials.zero(stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    LpView view() {
        LpView v;
        v.n = n;
        v.m = m;
        v.B = B;
        v.nbx_rows = geo_for(m, B).grid.x;
        v.nbx_cols = geo_for(n, B).grid.x;
        v.row_ptr = row_ptr.p;
        v.col_idx = col_idx.p;
        v.col_ptr = col_ptr.p;
        v.row_idx = row_idx.p;
        v.csc_src = csc_src.p;
        v.vals = vals.p;
        v.c = c.p;
        v.lb = lb.p;
        v.ub = ub.p;
        v.rl = rl.p;
        v.ru = ru.p;
        v.A = A.p;
        v.AT = AT.p;
        v.dr = dr.p;
        v.dc = dc.p;
        v.sr = sr.p;
        v.scf = scf.p;
        v.cs = cs.p;
        v.lbs = lbs.p;
        v.ubs = ubs.p;
        v.rls = rls.p;
        v.rus = rus.p;
        v.x = x.p;
        v.xa = xa.p;
        v.xp = xp.p;
        v.xbar = xbar.p;
        v.gy = gy.p;
        v.gyp = gyp.p;
        v.y = y.p;
        v.ya = ya.p;
        v.yp = yp.p;
        v.ray = ray.p;
        v.xo = xo.p;
        v.yo = yo.p;
        v.dlo = dlo.p;
        v.dup = dup.p;
        v.partials = partials.p;
        v.gmax = gmax.p;
        v.state = state.p;
        v.prm = prm.p;
        v.n_active = n_active.p;
        if (cur) {
            WorkSet &w = *cur;
            v.A = w.A.p; v.AT = w.AT.p; v.cs = w.cs.p; v.lbs = w.lbs.p; v.ubs = w.ubs.p; v.rls = w.rls.p; v.rus = w.rus.p;
            v.x = w.x.p; v.xa = w.xa.p; v.xp = w.xp.p; v.xbar = w.xbar.p; v.gy = w.gy.p; v.gyp = w.gyp.p;
            v.y = w.y.p; v.ya = w.ya.p; v.yp = w.yp.p; v.ray = w.ray.p; v.dr = w.dr.p; v.dc = w.dc.p;
            v.lb = w.lb.p; v.ub = w.ub.p; v.xo = w.xo.p; v.yo = w.yo.p; v.dlo = w.dlo.p; v.dup = w.dup.p;
            v.state = w.state.p;
        }
        return v;
    }

    int alloc_workset(WorkSet &w, int capB) {
        if (w.cap >= capB) return ASM_OK;
        const size_t nB = (size_t)n * capB, mB = (size_t)std::max(m, 1) * capB, zB = (size_t)std::max<int64_t>(nnz, 1) * capB;
        DBuf<double> *zz[] = {&w.A, &w.AT};
        for (auto *b : zz) ASM_TRY(b->alloc(zB));
        DBuf<double> *nn[] = {&w.cs, &w.lbs, &w.ubs, &w.x, &w.xa, &w.xp, &w.xbar, &w.gy, &w.gyp, &w.dc, &w.lb, &w.ub, &w.xo, &w.dlo, &w.dup};
        for (auto *b : nn) ASM_TRY(b->alloc(nB));
        DBuf<double> *mm[] = {&w.rls, &w.rus, &w.y, &w.ya, &w.yp, &w.ray, &w.dr, &w.yo};
        for (auto *b : mm) ASM_TRY(b->alloc(mB));
        ASM_TRY(w.state.alloc(capB));
        ASM_TRY(w.orig.alloc(capB));
        w.cap = capB;
        return ASM_OK;
    }

    // outputs and states of the active compact set back to their home positions
    int scatter_home() {
        if (!cur) return ASM_OK;
        WorkSet &w = *cur;
        const int cnt = w.live;
        auto sc = [&](const DBuf<double> &src, DBuf<double> &dst, int64_t rows) {
            if (rows == 0 || cnt == 0) return;
            k_scatter_cols<<<ew_grid(rows * cnt), 1024, 0, stream>>>(src.p, dst.p, rows, w.B, homeB, w.orig.p, cnt);
            ++launches;
        };
        sc(w.xo, xo, n);
        sc(w.dlo, dlo, n);
        sc(w.dup, dup, n);
        sc(w.yo, yo, m);
        if (cnt) {
            k_scatter_state<<<(cnt + 127) / 128, 128, 0, stream>>>(w.state.p, state.p, w.orig.p, cnt);
            ++launches;
        }
        ASM_CK(cudaGetLastError());
        return ASM_OK;
    }

    // copy the running LPs of the current set into a narrower one; host_state must hold the current states
    int compact() {
        LpView v = view();
        const Geo gm = geo_for(std::max(n, m), B);
        ASM_KB(k_finalize, gm, v);   // finished LPs get their final outputs now
        ASM_TRY(scatter_home());
        std::vector<int> src, orig;
        for (int s2 = 0; s2 < Buser; ++s2)
            if (host_state[s2].status < 0) {
                src.push_back(s2);
                orig.push_back(cur ? cur->h_orig[s2] : s2);
            }
        const int cnt = (int)src.size();
        if (cnt == 0) return ASM_OK;
        const int Bn = pad_batch(cnt);
        WorkSet &w = (cur == &wsets[0]) ? wsets[1] : wsets[0];
        ASM_TRY(alloc_workset(w, Bn));
        DBuf<int> dsrc;
        ASM_TRY(dsrc.alloc(cnt));
        ASM_CK(cudaMemcpyAsync(dsrc.p, src.data(), sizeof(int) * cnt, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaMemcpyAsync(w.orig.p, orig.data(), sizeof(int) * cnt, cudaMemcpyHostToDevice, stream));
        auto ga = [&](const double *from, DBuf<double> &to, int64_t rows) {
            if (rows == 0) return;
            k_gather_cols<<<ew_grid(rows * Bn), 1024, 0, stream>>>(from, to.p, rows, B, Bn, dsrc.p, cnt);
            ++launches;
        };
        ga(v.A, w.A, nnz); ga(v.AT, w.AT, nnz);
        ga(v.cs, w.cs, n); ga(v.lbs, w.lbs, n); ga(v.ubs, w.ubs, n); ga(v.x, w.x, n); ga(v.xa, w.xa, n); ga(v.dc, w.dc, n);
        ga(v.lb, w.lb, n); ga(v.ub, w.ub, n);
        ga(v.rls, w.rls, m); ga(v.rus, w.rus, m); ga(v.y, w.y, m); ga(v.ya, w.ya, m); ga(v.dr, w.dr, m);
        // the last checked point travels too: an LP that hits the iteration limit reports it
        ga(v.xp, w.xp, n); ga(v.gyp, w.gyp, n); ga(v.yp, w.yp, m);
        k_gather_state<<<(Bn + 127) / 128, 128, 0, stream>>>(v.state, w.state.p, dsrc.p, cnt, Bn);
        ++launches;
        ASM_CK(cudaGetLastError());
        ASM_CK(cudaMemcpyAsync(n_active.p, &cnt, sizeof(int), cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));   // dsrc / src / cnt go out of scope
        w.h_orig = orig;
        w.B = Bn;
        w.live = cnt;
        cur = &w;
        B = Bn;
        Buser = cnt;
        if (graph_exec) {
            cudaGraphExecDestroy(graph_exec);
            graph_exec = nullptr;
        }
        ++compactions;
        return ASM_OK;
    }

    static unsigned ew_grid(int64_t cnt) {
        return (unsigned)std::max<int64_t>(1, std::min<int64_t>((cnt + 1023) / 1024, kSMs * 16));
    }

    double tiny_rel = kTinyRel;  // asm_lp_params.tiny_rel of the current solve
    int precondition(int ruiz_iters, int warm) {
        LpView v = view();
        const Geo gr = geo_for(m, B), gc = geo_for(n, B), gm = geo_for(std::max(n, m), B);
        const int64_t nB = (int64_t)n * B, mB = (int64_t)m * B;
        ASM_KL(k_fill<<<ew_grid(mB), 1024, 0, stream>>>(dr.p, 1.0, mB));
        ASM_KL(k_fill<<<ew_grid(nB), 1024, 0, stream>>>(dc.p, 1.0, nB));
        {
            const Geo gz = geo_for(std::max<int64_t>(nnz, 1), B);
            ASM_KB(k_absmax, gz, v, nnz);
            ASM_KL(k_final_max<<<B, kFinalThreads, 0, stream>>>(partials.p, (int)gz.grid.x, B, gmax.p, tiny_rel / kTinyRel));
        }
        for (int it = 0; it <= ruiz_iters; ++it) {
            if (it == ruiz_iters) {  // last pass: Pock-Chambolle (alpha = 1): 1-norms
                ASM_KB2(k_ruiz_rows, true, gr, v);
                ASM_KB2(k_ruiz_cols, true, gc, v);
            } else {
                ASM_KB2(k_ruiz_rows, false, gr, v);
                ASM_KB2(k_ruiz_cols, false, gc, v);
            }
            ASM_KL(k_mul_inplace<<<ew_grid(mB), 1024, 0, stream>>>(dr.p, sr.p, mB));
            ASM_KL(k_mul_inplace<<<ew_grid(nB), 1024, 0, stream>>>(dc.p, scf.p, nB));
        }
        ASM_KB(k_build_scaled_csr, gr, v);
        ASM_KB(k_build_scaled_csc, gc, v);
        ASM_KB(k_prepare_cols, gc, v);
        ASM_KB(k_prepare_rows, gr, v);
        ASM_KL(k_init_state<<<B, kFinalThreads, 0, stream>>>(v));
        ASM_KB(k_prepare_finish, gm, v, warm, (const int *)(warm ? d_prev_ok.p : nullptr));
        if (B > Buser) ASM_KL(k_mark_padding<<<(B - Buser + 127) / 128, 128, 0, stream>>>(state.p, Buser, B));
        ASM_CK(cudaGetLastError());
        return ASM_OK;
    }

    // enqueue `steps` iterations; the first and the last are check steps
    void enqueue_block(int steps) {
        LpView v = view();
        const Geo gr = geo_for(m, B), gc = geo_for(n, B), gm = geo_for(std::max(n, m), B);
        for (int j = 0; j < steps; ++j) {
            if (j == 0 || j == steps - 1) {
                ASM_KB2(k_primal, true, gc, v, j);
                ASM_KB2(k_dual, true, gr, v, j);
                ASM_KB(k_dual_resid, gc, v);
                ASM_KB(k_ray_rows, gr, v);
                ASM_KB(k_ray_cols, gc, v);
                // v.state: after a compaction the running LPs' states live in the working set, not in `state`
                ASM_KL(k_store_kstep<<<(B + 127) / 128, 128, 0, stream>>>(v.state, kstep.p, j, B));
                ASM_KL(k_decide<<<B, kFinalThreads, 0, stream>>>(v, j, steps));
                ASM_KB(k_apply, gm, v, kstep.p);
                ASM_KL(k_after_apply<<<(B + 127) / 128, 128, 0, stream>>>(v.state, B));
            } else if (B % 64 == 0) {
                Geo g2c = gc, g2r = gr;
                g2c.grid.y = g2r.grid.y = B / 64;
                ASM_KL(k_primal2<<<g2c.grid, g2c.block, 0, stream>>>(v, j));
                ASM_KL(k_dual2<<<g2r.grid, g2r.block, 0, stream>>>(v, j));
            } else {
                ASM_KB2(k_primal, false, gc, v, j);
                ASM_KB2(k_dual, false, gr, v, j);
            }
        }
    }

    int build_graph(int steps) {
        if (graph_exec && graph_steps == steps) return ASM_OK;
        if (graph_exec) {
            cudaGraphExecDestroy(graph_exec);
            graph_exec = nullptr;
        }
        cudaGraph_t g = nullptr;
        const int64_t keep = launches;
        ASM_CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        enqueue_block(steps);
        cudaError_t e = cudaStreamEndCapture(stream, &g);
        launches_per_graph = launches - keep;
        launches = keep;
        ASM_CK(e);
        ASM_CK(cudaGraphInstantiate(&graph_exec, g, 0));
        cudaGraphDestroy(g);
        graph_steps = steps;
        return ASM_OK;
    }


    // ---- persistent group engine -------------------------------------------------------------------------------
    static constexpr size_t kSmemLimit = 227 * 1024 - 4096;  // dynamic shared memory available to one block

    // sliced-ELL layout of the pattern for groups of G blocks; returns the dynamic shared memory a block needs
    // (matrix values kept in shared memory when they fit, else streamed from L2), or 0 when G is infeasible
    static size_t plan_layout(const LpSolver &L, int G, SellSide &R, SellSide &C, GroupSmem &sm) {
        build_sell_side(L.m, L.n, L.h_row_ptr.data(), L.h_col_idx.data(), nullptr, G, R);
        build_sell_side(L.n, L.m, L.h_col_ptr.data(), L.h_row_idx.data(), nullptr, G, C);
        sm = GroupSmem();
        for (int c = 0; c < G; ++c) {
            sm.maxSellR = std::max(sm.maxSellR, R.ecnt[c]);
            sm.maxSellC = std::max(sm.maxSellC, C.ecnt[c]);
            sm.maxRpad = std::max(sm.maxRpad, R.nslice[c] * 32);
            sm.maxCpad = std::max(sm.maxCpad, C.nslice[c] * 32);
            sm.maxNSR = std::max(sm.maxNSR, R.nslice[c]);
            sm.maxNSC = std::max(sm.maxNSC, C.nslice[c]);
            sm.maxHaloR = std::max(sm.maxHaloR, R.halo_cnt[c]);
            sm.maxHaloC = std::max(sm.maxHaloC, C.halo_cnt[c]);
        }
        if (sm.maxHaloR > 65535 || sm.maxHaloC > 65535) return 0;  // halo positions are 16-bit
        // keep every carved array 8-byte aligned
        sm.maxSellR = (sm.maxSellR + 3) & ~3;
        sm.maxSellC = (sm.maxSellC + 3) & ~3;
        sm.maxHaloR = (sm.maxHaloR + 1) & ~1;
        sm.maxHaloC = (sm.maxHaloC + 1) & ~1;
        sm.maxNSR |= 1;   // (maxNSR + 1) + (maxNSC + 1) ints: keep the 16-bit arrays 8-byte aligned
        sm.maxNSC |= 1;
        sm.mats = 1;
        sm.push = 0;
        sm.maxPushR = sm.maxPushC = 0;
        if (sm.bytes() > kSmemLimit) sm.mats = 0;
        if (sm.mats && G <= kMaxClusterG) {   // exchange through (distributed) shared memory when it fits too
            std::vector<int> ptr, dst, base, cnt;
            build_push(R, C, G, ptr, dst, base, cnt);
            for (int c = 0; c < G; ++c) sm.maxPushR = std::max(sm.maxPushR, cnt[c]);
            build_push(C, R, G, ptr, dst, base, cnt);
            for (int c = 0; c < G; ++c) sm.maxPushC = std::max(sm.maxPushC, cnt[c]);
            sm.push = 1;
            if (sm.bytes() > kSmemLimit) {
                sm.push = 0;
                sm.maxPushR = sm.maxPushC = 0;
            }
        }
        return sm.bytes();
    }
    static bool plan_fits(size_t bytes) { return bytes > 0 && bytes <= kSmemLimit; }

    // Push lists for the distributed-shared-memory exchange: `prod` is the side that produces the vector (rows
    // produce y, columns produce xbar), `cons` the side whose halo lists name the entries it gathers.  For every
    // slot of every producing block: the (consumer rank << 16 | halo position) pairs, CSR by slot; ptr arrays are
    // concatenated per block with one extra entry each.
    static void build_push(const SellSide &prod, const SellSide &cons, int G, std::vector<int> &ptr, std::vector<int> &dst,
                           std::vector<int> &dst_base, std::vector<int> &dst_cnt) {
        ptr.clear();
        dst.clear();
        dst_base.assign(G, 0);
        dst_cnt.assign(G, 0);
        int total = 0;
        for (int c = 0; c < G; ++c) total = std::max(total, prod.first[c] + prod.cnt[c]);
        std::vector<std::vector<int>> who(total);
        for (int c = 0; c < G; ++c)
            for (int t = 0; t < cons.halo_cnt[c]; ++t) who[cons.halo[cons.halo_base[c] + t]].push_back((c << 16) | t);
        for (int o = 0; o < G; ++o) {
            dst_base[o] = (int)dst.size();
            const int nslot = prod.nslice[o] * 32;
            int local = 0;
            for (int sl = 0; sl < nslot; ++sl) {
                ptr.push_back(local);
                const int id = prod.slot[prod.slot_base[o] + sl];
                if (id >= 0)
                    for (int w : who[id]) {
                        dst.push_back(w);
                        ++local;
                    }
            }
            ptr.push_back(local);
            dst_cnt[o] = local;
        }
    }

    const std::pair<size_t, int> &feasible(int G) {
        auto it = feas.find(G);
        if (it != feas.end()) return it->second;
        SellSide R, C;
        GroupSmem sm;
        const size_t b = plan_layout(*this, G, R, C, sm);
        return feas[G] = std::make_pair(plan_fits(b) ? b : (size_t)0, sm.mats);
    }

    // Blocks per LP for `live` LPs that want to run at once.  Cost model from measurements on B200 (profiles/):
    // one iteration takes ~2.8 us of synchronisation in a cluster (4.4 us across clusters) plus ~1.5 ns per
    // matrix entry divided by the blocks.  Many LPs: the smallest group that keeps the matrix in shared memory
    // (throughput); few LPs: widen until the machine is used (latency).
    int choose_group(int want, int live, int n_sms) {
        static const int cand[] = {1, 2, 4, 8, 16, 24, 32, 48, 64, 74, 96, 128, 148};
        if (want > 0) return feasible(want).first ? want : -1;
        int base = -1;
        for (int g : cand) {
            if (g > n_sms) break;
            const auto &f = feasible(g);
            if (!f.first) continue;
            if (base < 0) base = g;
            if (f.second) {                       // matrix resident: take it unless it needs the slow barrier
                if (g <= kMaxClusterG || base > kMaxClusterG) base = g;
                break;
            }
            if (g >= kMaxClusterG && base <= kMaxClusterG) break;
        }
        if (base < 0) return -1;
        const double work = 1.5e-3 * (double)nnz;
        auto cost = [&](int g) { return (g <= kMaxClusterG ? 2.8 : 4.4) + work / g; };
        int G = base;
        for (int g : cand) {
            if (g <= base || g > n_sms) continue;
            if ((long long)live * g > n_sms) break;
            if (!feasible(g).first) continue;
            if (cost(g) < 0.92 * cost(G)) G = g;
        }
        return G;
    }

    static const void *group_kernel(bool cluster, bool mats, bool push = false) {
        if (cluster && mats && push) return (const void *)k_pdhg_group<true, true, true>;
        if (cluster) return mats ? (const void *)k_pdhg_group<true, true> : (const void *)k_pdhg_group<true, false>;
        return mats ? (const void *)k_pdhg_group<false, true> : (const void *)k_pdhg_group<false, false>;
    }

    int ensure_plan(int want_G, int live) {
        int dev = 0, n_sms = kSMs;
        ASM_CK(cudaGetDevice(&dev));
        ASM_CK(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        const int G = choose_group(want_G, std::max(1, live), n_sms);
        if (G < 0) return fail(ASM_E_INVALID, "LP does not fit the shared memory of the machine (group engine)");
        auto found = plans.find(G);
        if (found != plans.end()) {
            plan = found->second.get();
            return ASM_OK;
        }
        std::unique_ptr<GroupPlan> pl(new GroupPlan());
        pl->G = G;
        pl->cluster = G <= kMaxClusterG;
        SellSide R, C;
        plan_layout(*this, G, R, C, pl->sm);
        // the value source of the column side is the CSC position itself (AT is stored in CSC order)
        pl->cta.resize(G);
        for (int c = 0; c < G; ++c) {
            GroupCta &d = pl->cta[c];
            d.r0 = R.first[c];
            d.nR = R.cnt[c];
            d.nSR = R.nslice[c];
            d.sellR_base = R.base[c];
            d.sellR_cnt = R.ecnt[c];
            d.ptrR_base = R.ptr_base[c];
            d.slotR_base = R.slot_base[c];
            d.haloR_base = R.halo_base[c];
            d.haloR_cnt = R.halo_cnt[c];
            d.c0 = C.first[c];
            d.nC = C.cnt[c];
            d.nSC = C.nslice[c];
            d.sellC_base = C.base[c];
            d.sellC_cnt = C.ecnt[c];
            d.ptrC_base = C.ptr_base[c];
            d.slotC_base = C.slot_base[c];
            d.haloC_base = C.halo_base[c];
            d.haloC_cnt = C.halo_cnt[c];
        }
        pl->totSellR = (int)R.src.size();
        pl->totSellC = (int)C.src.size();
        if (pl->sm.push && getenv("ASM_NO_PUSH")) {   // debugging switch: exchange through L2 instead
            pl->sm.push = 0;
            pl->sm.maxPushR = pl->sm.maxPushC = 0;
        }
        {
            std::vector<int> ptr, dst, base, cnt;
            auto upl = [&](DBuf<int> &b, const std::vector<int> &h) -> int {
                ASM_TRY(b.alloc(std::max<size_t>(h.size(), 1)));
                if (!h.empty()) ASM_CK(cudaMemcpy(b.p, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice));
                return ASM_OK;
            };
            if (pl->sm.push) {
                build_push(R, C, G, ptr, dst, base, cnt);
                for (int c = 0; c < G; ++c) {
                    pl->cta[c].pushR_base = base[c];
                    pl->cta[c].pushR_cnt = cnt[c];
                }
                ASM_TRY(upl(pl->pushR_ptr, ptr));
                ASM_TRY(upl(pl->pushR_dst, dst));
                build_push(C, R, G, ptr, dst, base, cnt);
                for (int c = 0; c < G; ++c) {
                    pl->cta[c].pushC_base = base[c];
                    pl->cta[c].pushC_cnt = cnt[c];
                }
                ASM_TRY(upl(pl->pushC_ptr, ptr));
                ASM_TRY(upl(pl->pushC_dst, dst));
            } else {
                for (int c = 0; c < G; ++c) pl->cta[c].pushR_base = pl->cta[c].pushR_cnt = pl->cta[c].pushC_base = pl->cta[c].pushC_cnt = 0;
            }
        }
        auto up = [&](DBuf<int> &b, const std::vector<int> &h) -> int {
            ASM_TRY(b.alloc(std::max<size_t>(h.size(), 1)));
            if (!h.empty()) ASM_CK(cudaMemcpy(b.p, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice));
            return ASM_OK;
        };
        ASM_TRY(up(pl->sellR_src, R.src));
        ASM_TRY(up(pl->sellR_idx, R.idx));
        ASM_TRY(up(pl->ptrR, R.ptr));
        ASM_TRY(up(pl->slotR, R.slot));
        ASM_TRY(up(pl->haloR, R.halo));
        ASM_TRY(up(pl->haloC, C.halo));
        ASM_TRY(pl->tailR.alloc(std::max<size_t>(R.tail.size(), 1)));
        ASM_TRY(pl->tailC.alloc(std::max<size_t>(C.tail.size(), 1)));
        if (!R.tail.empty()) ASM_CK(cudaMemcpy(pl->tailR.p, R.tail.data(), R.tail.size(), cudaMemcpyHostToDevice));
        if (!C.tail.empty()) ASM_CK(cudaMemcpy(pl->tailC.p, C.tail.data(), C.tail.size(), cudaMemcpyHostToDevice));
        ASM_TRY(up(pl->sellC_src, C.src));
        ASM_TRY(up(pl->sellC_idx, C.idx));
        ASM_TRY(up(pl->ptrC, C.ptr));
        ASM_TRY(up(pl->slotC, C.slot));
        ASM_TRY(pl->d_cta.alloc(G));
        ASM_CK(cudaMemcpy(pl->d_cta.p, pl->cta.data(), sizeof(GroupCta) * G, cudaMemcpyHostToDevice));
        // how many groups can be resident at once
        const size_t smem = pl->sm.bytes();
        int groups = 1;
        const void *fn = group_kernel(pl->cluster, pl->sm.mats != 0, pl->sm.push != 0);
        ASM_CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (pl->cluster) {
            if (G > 8) ASM_CK(cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(G);
            cfg.blockDim = dim3(kGThreads);
            cfg.dynamicSmemBytes = smem;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = G;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            int nc = 0;
            ASM_CK(cudaOccupancyMaxActiveClusters(&nc, fn, &cfg));
            if (nc < 1) return fail(ASM_E_CUDA, "a cluster of this size cannot be scheduled");
            groups = nc;
        } else {
            int per_sm = 0;
            ASM_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kGThreads, smem));
            if (per_sm < 1) return fail(ASM_E_CUDA, "group kernel does not fit on an SM");
            groups = (n_sms * per_sm) / G;
            if (groups < 1) return fail(ASM_E_CUDA, "group larger than the machine");
        }
        groups = std::min(groups, Buser);
        pl->n_groups = groups;
        pl->max_groups = groups;
        const size_t gn = (size_t)groups * n, gm = (size_t)groups * std::max(m, 1);
        DBuf<double> *cn[] = {&pl->gx, &pl->gx2, &pl->gxp, &pl->grc};
        for (auto *b : cn) {
            ASM_TRY(b->alloc(gn));
            ASM_TRY(b->zero(stream));
        }
        DBuf<double> *rm[] = {&pl->gy, &pl->gyp, &pl->gray};
        for (auto *b : rm) {
            ASM_TRY(b->alloc(gm));
            ASM_TRY(b->zero(stream));
        }
        if (!pl->sm.mats) {
            ASM_TRY(pl->gA.alloc((size_t)groups * pl->totSellR));
            ASM_TRY(pl->gAT.alloc((size_t)groups * pl->totSellC));
            ASM_TRY(pl->gconst.alloc((size_t)groups * G * (2 * (size_t)pl->sm.maxRpad + 3 * (size_t)pl->sm.maxCpad)));
        }
        ASM_TRY(pl->part.alloc((size_t)groups * G * Q_COUNT));
        ASM_TRY(pl->bar.alloc(groups));
        ASM_TRY(pl->queue.alloc(1));
        ASM_TRY(pl->slot.alloc(groups));
        plan = pl.get();
        plans[G] = std::move(pl);
        return ASM_OK;
    }

    int run_group(const asm_lp_params &P, int steps, int live, long long budget) {
        GroupPlan &pl = *plan;
        pl.n_groups = std::max(1, std::min(pl.max_groups, live));
        GroupArgs a;
        a.v = view();
        a.cta = pl.d_cta.p;
        a.sellR_src = pl.sellR_src.p;
        a.sellR_idx = pl.sellR_idx.p;
        a.ptrR = pl.ptrR.p;
        a.slotR = pl.slotR.p;
        a.haloR = pl.haloR.p;
        a.haloC = pl.haloC.p;
        a.tailR = pl.tailR.p;
        a.tailC = pl.tailC.p;
        a.pushR_ptr = pl.pushR_ptr.p;
        a.pushR_dst = pl.pushR_dst.p;
        a.pushC_ptr = pl.pushC_ptr.p;
        a.pushC_dst = pl.pushC_dst.p;
        a.gA = pl.gA.p;
        a.gAT = pl.gAT.p;
        a.gconst = pl.gconst.p;
        a.totSellR = pl.totSellR;
        a.totSellC = pl.totSellC;
        a.sellC_src = pl.sellC_src.p;
        a.sellC_idx = pl.sellC_idx.p;
        a.ptrC = pl.ptrC.p;
        a.slotC = pl.slotC.p;
        a.gx = pl.gx.p;
        a.gx2 = pl.gx2.p;
        a.gxp = pl.gxp.p;
        a.grc = pl.grc.p;
        a.gy = pl.gy.p;
        a.gyp = pl.gyp.p;
        a.gray = pl.gray.p;
        a.part = pl.part.p;
        a.bar = pl.bar.p;
        a.queue = pl.queue.p;
        a.slot = pl.slot.p;
        a.G = pl.G;
        a.Buser = Buser;
        a.max_iter = P.max_iter;
        a.budget = budget;
        a.steps = std::min(steps, kMaxSteps);
        a.sm = pl.sm;
        ASM_TRY(pl.bar.zero(stream));
        ASM_TRY(pl.queue.zero(stream));
        const size_t smem = pl.sm.bytes();
        const unsigned grid = (unsigned)(pl.n_groups * pl.G);
        const void *fn = group_kernel(pl.cluster, pl.sm.mats != 0, pl.sm.push != 0);
        void *args[] = {(void *)&a};
        // plans of different group sizes share the kernel: the attribute must match this launch
        ASM_CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (pl.cluster) {
            ASM_CK(cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, pl.G > 8 ? 1 : 0));
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid);
            cfg.blockDim = dim3(kGThreads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = pl.G;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            ASM_CK(cudaLaunchKernelExC(&cfg, fn, args));
        } else {
            ASM_CK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kGThreads), args, smem, stream));
        }
        ++launches;
        last_G = pl.G;
        last_groups = pl.n_groups;
        return ASM_OK;
    }

    int set_active(const int32_t *active) {
        if (!active) {
            n_masked = -1;
            return ASM_OK;
        }
        if (d_active.n < (size_t)Buser) ASM_TRY(d_active.alloc(Buser));
        std::vector<int> h(active, active + Buser);
        n_masked = 0;
        for (int v : h) n_masked += v != 0;
        ASM_CK(cudaMemcpyAsync(d_active.p, h.data(), sizeof(int) * Buser, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    // the scenarios in `lanes` were replaced: their next PDHG solve starts cold.  The barrier engine keeps nothing
    // across solves.
    void forget_warm_start(const int32_t *lanes, int k) {
        for (int j = 0; j < k; ++j)
            if (lanes[j] >= 0 && lanes[j] < (int)start_ok.size()) start_ok[lanes[j]] = 0;
    }

    // the caller's start (asm_lp_set_start) is used by the next warm solve of every scenario, whatever ended the last
    void accept_start() {
        std::fill(start_ok.begin(), start_ok.end(), 1);
        has_solution = true;
    }

    // start_ok -> d_prev_ok for the warm solve about to be preconditioned
    int upload_start_ok() {
        if (d_prev_ok.n < (size_t)B) ASM_TRY(d_prev_ok.alloc(B));
        std::vector<int> ok(B, 0);
        for (int s = 0; s < Buser; ++s) ok[s] = start_ok[s];
        ASM_CK(cudaMemcpyAsync(d_prev_ok.p, ok.data(), sizeof(int) * B, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    // ---- barrier engine: Mehrotra predictor-corrector on the fixed-pattern L D L' (ipm.cuh) ----------------------
    int ensure_ipm() {
        if (ipm) return ASM_OK;
        std::unique_ptr<IpmEngine> e(new IpmEngine);
        const int rc = e->init(n, m, h_row_ptr, h_col_idx, B);
        if (rc != ASM_OK) {
            ipm_failed = 1;
            return rc;
        }
        ipm = std::move(e);
        return ASM_OK;
    }
    int solve_ipm(const asm_lp_params &P, int *flag) {
        ASM_TRY(ensure_ipm());
        IpmEngine &E = *ipm;
        LpView v = view();
        IpmView g = E.iview(P);
        g.c0 = c0.p;
        KktDev d = E.dev();
        const Geo gr = geo_for(m, B), gc = geo_for(n, B), gm = geo_for(std::max(n, m), B), gN = geo_for((int64_t)n + m, B);
        // refinement passes per linear solve: ipm_refine to start with (default 1), one more (at most two more) each time
        // k_ipm_decide reports LPs stuck between the acceptable and the target tolerance
        int refine = P.ipm_refine >= 0 ? P.ipm_refine : 0;
        const int base_refine = refine, refine_max = refine + 2;
        g.need_refine = n_active.p + 1;
        flag[1] = 0;
        ASM_CK(cudaMemcpyAsync(n_active.p + 1, flag + 1, sizeof(int), cudaMemcpyHostToDevice, stream));
        const int max_it = P.ipm_max_iter > 0 ? P.ipm_max_iter : 200;
        const bool trace = getenv("ASM_TRACE") != nullptr;
        ASM_TRY(E.capture(stream, &E.g_factor, E.launches_factor, [&](int64_t &c) { E.enqueue_factor(v, stream, c); }));
        ASM_TRY(E.capture(stream, &E.g_solve_sol, E.launches_solve, [&](int64_t &c) { E.enqueue_solve(v, g.sol, stream, c); }));
        ASM_TRY(E.capture(stream, &E.g_solve_work, E.launches_solve, [&](int64_t &c) { E.enqueue_solve(v, g.work, stream, c); }));
        E.last_pairs = 0;
        E.last_factorisations = 0;
        auto solve_refined = [&](int passes) -> int {
            E.last_pairs += 1 + passes;
            ASM_CK(cudaGraphLaunch(E.g_solve_sol, stream));
            launches += E.launches_solve;
            for (int r = 0; r < passes; ++r) {
                ASM_KB(k_kkt_res_cols, gc, v, g);
                ASM_KB(k_kkt_res_rows, gr, v, g);
                ASM_CK(cudaGraphLaunch(E.g_solve_work, stream));
                launches += E.launches_solve;
                ASM_KB(k_kkt_add, gN, v, g, (int64_t)n + m);
            }
            return ASM_OK;
        };
        ASM_KB(k_ipm_init_cols, gc, v, g);
        ASM_KB(k_ipm_init_rows, gr, v, g);
        ASM_KL(k_ipm_init_state<<<B, kFinalThreads, 0, stream>>>(v, g));
        int it = 0, refine_seen = 0;
        for (;; ++it) {
            ASM_KB(k_ipm_res_cols, gc, v, g);
            ASM_KB(k_ipm_res_rows, gr, v, g);
            ASM_KL(k_ipm_decide<<<B, kFinalThreads, 0, stream>>>(v, g, it, it >= max_it ? 1 : 0));
            ASM_KB(k_ipm_save, gm, v, g);
            ASM_CK(cudaMemcpyAsync(flag, n_active.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
            ASM_CK(cudaStreamSynchronize(stream));
            if (*flag <= 0 || it >= max_it) break;
            if (flag[1] > refine_seen && refine < refine_max) {
                ++refine;
                if (trace) fprintf(stderr, "[asm] barrier engine: step %d, %d LPs stuck at the acceptable level -> %d refinement passes\n", it, flag[1], refine);
            }
            refine_seen = flag[1];
            ASM_KB(k_ipm_diag, gm, v, g, d);
            const bool timed = trace && it == 1;
            cudaEvent_t te[3] = {nullptr, nullptr, nullptr};
            if (timed) {
                for (auto &e : te) cudaEventCreate(&e);
                cudaEventRecord(te[0], stream);
            }
            ASM_CK(cudaGraphLaunch(E.g_factor, stream));
            launches += E.launches_factor;
            E.last_factorisations += 1;
            if (timed) cudaEventRecord(te[1], stream);
            ASM_KB2(k_ipm_rhs, false, gm, v, g);
            // the affine direction only sets the centring parameter and the second-order term: it is not refined
            // unless the LPs are already stuck on solve accuracy
            ASM_TRY(solve_refined(refine > base_refine ? refine : 0));
            if (timed) {
                cudaEventRecord(te[2], stream);
                cudaEventSynchronize(te[2]);
                cudaEventElapsedTime(&E.last_factor_ms, te[0], te[1]);
                cudaEventElapsedTime(&E.last_solve_ms, te[1], te[2]);
                fprintf(stderr, "[asm] barrier engine: N %d nnz(L) %lld terms %lld levels %d | factor %.3f ms (%lld launches) | "
                        "solve + %d refinements %.3f ms (%lld launches per substitution pair) | symbolic %.0f ms\n",
                        E.sym.N, (long long)E.sym.nnzL, (long long)E.sym.nterms, E.sym.n_levels, E.last_factor_ms,
                        (long long)E.launches_factor, refine, E.last_solve_ms, (long long)E.launches_solve, E.symbolic_ms);
                for (auto &e : te) cudaEventDestroy(e);
            }
            ASM_KB2(k_ipm_dirs_cols, false, gc, v, g);
            ASM_KB2(k_ipm_dirs_rows, false, gr, v, g);
            ASM_KL(k_ipm_scalars<<<B, kFinalThreads, 0, stream>>>(v, g, 0, (int)gm.grid.x));
            ASM_KB(k_ipm_muaff, gm, v, g);
            ASM_KL(k_ipm_scalars<<<B, kFinalThreads, 0, stream>>>(v, g, 1, (int)gm.grid.x));
            ASM_KB2(k_ipm_rhs, true, gm, v, g);
            ASM_TRY(solve_refined(refine));
            ASM_KB2(k_ipm_dirs_cols, true, gc, v, g);
            ASM_KB2(k_ipm_dirs_rows, true, gr, v, g);
            ASM_KB(k_ipm_ray, gr, v, g);
            ASM_KB(k_ipm_ray_cols, gc, v, g);
            ASM_KL(k_ipm_scalars<<<B, kFinalThreads, 0, stream>>>(v, g, 2, (int)gm.grid.x));
            ASM_KB(k_ipm_update, gm, v, g);
            ASM_CK(cudaGetLastError());
        }
        ASM_KB(k_ipm_final_obj, gc, v);
        ASM_KL(k_ipm_final_state<<<B, kFinalThreads, 0, stream>>>(v, Buser));
        E.last_newton = it;
        last_engine = 4;
        return ASM_OK;
    }

    // average device time of one numeric factorisation and of one substitution pair of the barrier engine (CUDA events
    // on this handle's stream); scenarios are re-activated for the measurement, the result buffers are not touched
    int time_ipm_kernels(int reps, double *factor_ms, double *solve_ms) {
        if (!ipm || !ipm->g_factor || !ipm->g_solve_work) return fail(ASM_E_STATE, "the barrier engine has not run on this handle");
        IpmEngine &E = *ipm;
        std::vector<ScenState> keep(B), live(B);
        ASM_CK(cudaMemcpyAsync(keep.data(), state.p, sizeof(ScenState) * B, cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        live = keep;
        for (int s = 0; s < Buser; ++s) live[s].status = -1;
        ASM_CK(cudaMemcpyAsync(state.p, live.data(), sizeof(ScenState) * B, cudaMemcpyHostToDevice, stream));
        float t = 0.f;
        for (int w = 0; w < 2; ++w) {
            ASM_CK(cudaGraphLaunch(E.g_factor, stream));
            ASM_CK(cudaGraphLaunch(E.g_solve_work, stream));
        }
        ASM_CK(cudaEventRecord(ev0, stream));
        for (int r = 0; r < reps; ++r) ASM_CK(cudaGraphLaunch(E.g_factor, stream));
        ASM_CK(cudaEventRecord(ev1, stream));
        ASM_CK(cudaEventSynchronize(ev1));
        ASM_CK(cudaEventElapsedTime(&t, ev0, ev1));
        if (factor_ms) *factor_ms = t / reps;
        ASM_CK(cudaEventRecord(ev0, stream));
        for (int r = 0; r < reps; ++r) ASM_CK(cudaGraphLaunch(E.g_solve_work, stream));
        ASM_CK(cudaEventRecord(ev1, stream));
        ASM_CK(cudaEventSynchronize(ev1));
        ASM_CK(cudaEventElapsedTime(&t, ev0, ev1));
        if (solve_ms) *solve_ms = t / reps;
        launches += (int64_t)(reps + 2) * (E.launches_factor + E.launches_solve);
        ASM_CK(cudaMemcpyAsync(state.p, keep.data(), sizeof(ScenState) * B, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    // average device time of one launch of each streaming kernel; scenarios are re-activated for the measurement
    int time_streaming_kernels(int reps, double *primal_ms, double *dual_ms) {
        LpView v = view();
        const Geo gr = geo_for(m, B), gc = geo_for(n, B);
        std::vector<ScenState> keep(B), live(B);
        ASM_CK(cudaMemcpyAsync(keep.data(), state.p, sizeof(ScenState) * B, cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        live = keep;
        for (auto &s : live) s.status = -1;
        ASM_CK(cudaMemcpyAsync(state.p, live.data(), sizeof(ScenState) * B, cudaMemcpyHostToDevice, stream));
        float t = 0.f;
        const bool wide = B % 64 == 0;
        Geo g2c = gc, g2r = gr;
        if (wide) g2c.grid.y = g2r.grid.y = B / 64;
        auto primal = [&]() {
            if (wide)
                k_primal2<<<g2c.grid, g2c.block, 0, stream>>>(v, 1);
            else if (B > 1)
                k_primal<true, false><<<gc.grid, gc.block, 0, stream>>>(v, 1);
            else
                k_primal<false, false><<<gc.grid, gc.block, 0, stream>>>(v, 1);
            ++launches;
        };
        auto dual = [&]() {
            if (wide)
                k_dual2<<<g2r.grid, g2r.block, 0, stream>>>(v, 1);
            else if (B > 1)
                k_dual<true, false><<<gr.grid, gr.block, 0, stream>>>(v, 1);
            else
                k_dual<false, false><<<gr.grid, gr.block, 0, stream>>>(v, 1);
            ++launches;
        };
        for (int w = 0; w < 3; ++w) {
            primal();
            dual();
        }
        ASM_CK(cudaEventRecord(ev0, stream));
        for (int r = 0; r < reps; ++r) primal();
        ASM_CK(cudaEventRecord(ev1, stream));
        ASM_CK(cudaEventSynchronize(ev1));
        ASM_CK(cudaEventElapsedTime(&t, ev0, ev1));
        if (primal_ms) *primal_ms = t / reps;
        ASM_CK(cudaEventRecord(ev0, stream));
        for (int r = 0; r < reps; ++r) dual();
        ASM_CK(cudaEventRecord(ev1, stream));
        ASM_CK(cudaEventSynchronize(ev1));
        ASM_CK(cudaEventElapsedTime(&t, ev0, ev1));
        if (dual_ms) *dual_ms = t / reps;
        ASM_CK(cudaMemcpyAsync(state.p, keep.data(), sizeof(ScenState) * B, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    int solve(const asm_lp_params &P, asm_lp_info *info) {
        if (cur) {   // a previous solve failed half way through a compacted batch: back to the home batch
            cur = nullptr;
            B = homeB;
            Buser = homeBuser;
            if (graph_exec) {
                cudaGraphExecDestroy(graph_exec);
                graph_exec = nullptr;
            }
        }
        const DevParams dp = dev_params(P);
        int *flag = (int *)pin_flag.p;
        DevParams *pdp = (DevParams *)((char *)pin_flag.p + 16);
        static_assert(sizeof(DevParams) + 16 <= 128, "pinned flag area too small");  // 9 doubles + int
        ASM_TRY(pin_flag.reserve(128));
        flag = (int *)pin_flag.p;
        pdp = (DevParams *)((char *)pin_flag.p + 16);
        *pdp = dp;
        *flag = Buser;
        ASM_CK(cudaMemcpyAsync(prm.p, pdp, sizeof dp, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaMemcpyAsync(n_active.p, flag, sizeof(int), cudaMemcpyHostToDevice, stream));
        tiny_rel = P.tiny_rel > 0.0 ? P.tiny_rel : kTinyRel;
        // engine 0 (auto) and 4: barrier method on the fixed-pattern L D L'; 1 / 2 / 5: the PDHG engines
        bool use_ipm = P.engine == 4 || (P.engine == 0 && !ipm_failed);
        if (use_ipm && ensure_ipm() != ASM_OK) {
            if (P.engine == 4) return ASM_E_INVALID;
            use_ipm = false;
        }
        const int warm = (!use_ipm && P.warm_start && has_solution) ? (int)P.warm_start : 0;
        if (warm) ASM_TRY(upload_start_ok());
        ASM_TRY(precondition(P.ruiz_iters, warm));
        if (n_masked >= 0) {
            ASM_KL(k_apply_mask<<<(Buser + 127) / 128, 128, 0, stream>>>(state.p, d_active.p, Buser));
            *flag = n_masked;
            ASM_CK(cudaMemcpyAsync(n_active.p, flag, sizeof(int), cudaMemcpyHostToDevice, stream));
            ASM_CK(cudaStreamSynchronize(stream));
        }
        const int steps = std::max(2, (int)P.check_every);
        // engine 1: streaming kernels only (one launch per half iteration, CUDA graph per check period);
        // engine 2: persistent group kernel only;
        // engine 0: a single LP runs on the group kernel; a batch streams, compacting the running LPs into a narrower
        //           working set as they converge, and hands the stragglers to the group kernel when the cost model
        //           says so -- every LP stops at its own convergence
        homeB = B;
        homeBuser = Buser;
        compactions = 0;
        const int hand_over = Buser == 1 ? 0 : std::max(1, std::min(Buser, (int)(P.hand_over * Buser)));
        const bool plan_ok = !use_ipm && P.engine != 1 &&
                             ensure_plan(P.group_size, P.engine == 2 ? Buser : std::max(1, hand_over)) == ASM_OK;
        if (P.engine == 2 && !plan_ok) return ensure_plan(P.group_size, Buser);
        const bool group_only = plan_ok && (P.engine == 2 || Buser == 1);
        ASM_CK(cudaEventRecord(ev0, stream));
        last_engine = 0;
        last_G = 0;
        last_groups = 0;
        int live = n_masked >= 0 ? n_masked : Buser;
        bool limit = false;
        const bool trace = getenv("ASM_TRACE") != nullptr;
        auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        double t_phase = now();
        if (use_ipm) {
            ASM_TRY(solve_ipm(P, flag));
            live = 0;
        } else if (!group_only) {
            // cost model (seconds per iteration of one running LP), calibrated on B200 (profiles/): the streaming
            // kernels move the whole working set at ~4.4 TB/s plus two launches; the group kernel costs
            // (sync + work / G) on G of the machine's SMs
            int n_sms = kSMs;
            cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device);
            const double bytes_it = 16.0 * (double)nnz + 64.0 * n + 48.0 * m;
            auto stream_cost = [&](int Bc, int lv) { return ((double)Bc * bytes_it / 4.4e12 + 8e-6) / std::max(1, lv); };
            auto group_cost = [&](int lv) {
                const int G = choose_group(P.group_size, lv, n_sms);
                if (G < 0) return 1e30;
                const double t = ((G <= kMaxClusterG ? 2.8 : 4.4) + 1.5e-3 * (double)nnz / G) * 1e-6;
                const int resident = std::max(1, (int)(0.8 * n_sms) / G);
                return t / std::min(lv, resident);
            };
            int64_t it = 0;
            while (it < P.max_iter) {
                ASM_TRY(build_graph(steps));
                ASM_CK(cudaGraphLaunch(graph_exec, stream));
                launches += launches_per_graph;
                it += steps;
                ASM_CK(cudaMemcpyAsync(flag, n_active.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
                ASM_CK(cudaStreamSynchronize(stream));
                live = *flag;
                if (live <= 0) break;
                const bool shrink = (P.engine == 0 || P.engine == 5) && B >= 128 && pad_batch(live) * 2 <= B;
                if (plan_ok && live <= hand_over && group_cost(live) < stream_cost(shrink ? pad_batch(live) : B, live)) break;
                if (shrink) {
                    LpView vv = view();
                    ASM_CK(cudaMemcpyAsync(host_state.data(), vv.state, sizeof(ScenState) * B, cudaMemcpyDeviceToHost, stream));
                    ASM_CK(cudaStreamSynchronize(stream));
                    const int before = B;
                    ASM_TRY(compact());
                    if (trace)
                        fprintf(stderr, "[asm] it %lld: %d LPs running, batch %d -> %d (%.3f s since last event)\n",
                                (long long)it, live, before, B, now() - t_phase);
                    t_phase = now();
                }
            }
            limit = it >= P.max_iter;
            last_engine |= 1;
        }
        // group phase: re-planned as the live set thins out (wider groups for the last stragglers)
        if (trace && !group_only && !use_ipm)
            fprintf(stderr, "[asm] streaming phase done: %d LPs still running (%.3f s since last event)\n", live, now() - t_phase);
        t_phase = now();
        while (plan_ok && live > 0 && !limit) {
            ASM_TRY(ensure_plan(P.group_size, live));
            const long long budget = live > 1 ? (1LL << 16) : P.max_iter;
            ASM_TRY(run_group(P, steps, live, budget));
            last_engine |= 2;
            LpView vv = view();
            ASM_CK(cudaMemcpyAsync(host_state.data(), vv.state, sizeof(ScenState) * B, cudaMemcpyDeviceToHost, stream));
            ASM_CK(cudaStreamSynchronize(stream));
            if (trace) {
                fprintf(stderr, "[asm] group launch: %d LPs, G = %d (%s, matrix %s), %d groups resident, %.3f s\n", live,
                        plan->G, plan->cluster ? (plan->sm.push ? "cluster, DSMEM exchange" : "cluster") : "grid",
                        plan->sm.mats ? "resident" : "streamed", plan->n_groups,
                        now() - t_phase);
                t_phase = now();
            }
            live = 0;
            for (int s = 0; s < Buser; ++s)
                if (host_state[s].status < 0 && host_state[s].total < P.max_iter) ++live;
        }
        ASM_CK(cudaEventRecord(ev1, stream));
        {
            LpView v = view();
            const Geo gm = geo_for(std::max(n, m), B);
            ASM_KB(k_finalize, gm, v);
        }
        if (cur) {   // back to the home batch
            ASM_TRY(scatter_home());
            cur = nullptr;
            B = homeB;
            Buser = homeBuser;
            if (graph_exec) {
                cudaGraphExecDestroy(graph_exec);
                graph_exec = nullptr;
            }
        }
        ASM_CK(cudaMemcpyAsync(host_state.data(), state.p, sizeof(ScenState) * B, cudaMemcpyDeviceToHost, stream));
        std::vector<double> hc0(B, 0.0);
        ASM_CK(cudaMemcpyAsync(hc0.data(), c0.p, sizeof(double) * B, cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        float ms = 0.f;
        ASM_CK(cudaEventElapsedTime(&ms, ev0, ev1));
        last_loop_ms = ms;
        last_iters = 0;
        for (int s = 0; s < Buser; ++s) {
            ScenState &st = host_state[s];
            if (st.status < 0) st.status = ASM_LP_ITERATION_LIMIT;
            start_ok[s] = st.status == ASM_LP_OPTIMAL;
            last_iters = std::max<int64_t>(last_iters, st.total);
            if (info) lp_info(st, hc0[s], info[s]);
        }
        has_solution = true;
        return ASM_OK;
    }
};

}  // namespace asmb
