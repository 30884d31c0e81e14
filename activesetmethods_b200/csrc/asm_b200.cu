// C ABI of the B200 sub-LP engine (include/asm_b200.h) and the SLP layer above the PDHG LP solver:
// Jacobian pattern analysis, ordered COO->CSR assembly, sub-LP bound construction (normal phase and
// feasibility restoration), read-back with the reference's masking, merit / KKT reductions.
//
// Reference functions restated here (paths relative to /root/reference):
//   compute_jacobian_matrix   src/algorithms/common.jl:12-20      -> Pattern + k_assemble
//   create_model!             src/algorithms/subproblem.jl:51-215 -> Pattern::build_fr (column / row layout)
//   sub_optimize! (update)    src/algorithms/subproblem.jl:248-484 -> k_slp_cols / k_slp_rows / k_fr_*
//   sub_optimize! (read-back) src/algorithms/subproblem.jl:491-541 -> k_extract
//   norm_violations / KT_residuals / norm_complementarity   src/algorithms/common.jl:35-98
//   compute_phi / compute_derivative                         src/algorithms/slp.jl:79-147
#include <math.h>
#include <string.h>

#include <algorithm>
#include <limits>
#include <memory>
#include <numeric>

#include "lp_dist.cuh"

namespace asmb {

// row classes of create_model! (subproblem.jl:143-197)
enum : uint8_t { ROW_EQ = 0, ROW_RANGE = 1, ROW_LOWER = 2, ROW_UPPER = 3 };

// =================================== SLP kernels ================================================================
// compute_jacobian_matrix (common.jl:12-20): every CSR slot is ((0.0 + v1) + v2) + ... with the duplicates
// of the slot taken in j_str order -> bit-identical to the reference's J[r, c] += v loop.
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_assemble(const int *__restrict__ dup_ptr, const int *__restrict__ dup_idx,
                                                        const double *__restrict__ dE, double *__restrict__ vals,
                                                        int64_t nslots, int B) {
    Map<BATCH> mp;
    for (int64_t k = mp.first; k < nslots; k += mp.stride) {
        double a = 0.0;
        const int d1 = dup_ptr[k + 1];
        for (int d = dup_ptr[k]; d < d1; ++d) a += dE[(int64_t)dup_idx[d] * B + mp.s];
        vals[k * B + mp.s] = a;
    }
}

struct SlpView {
    int n, m, B, Bb;  // Bb: batch stride of the NLP bounds (1 = shared, B = per scenario)
    int n_adj;
    const double *xL, *xU, *gL, *gU;         // NLP bounds
    const double *xk, *df, *E, *delta;       // current point (element-major), delta[B]
    const uint8_t *cls;                      // row class
    const int *s1, *s2, *adj, *adj_of_row;   // slack columns (FR LP), range rows
};

__device__ __forceinline__ double pos_zero(double v) { return v == 0.0 ? 0.0 : v; }  // tol_error = 0 snap (App. C-9)

// column bounds of the step (subproblem.jl:427-434) and objective (:384-408 normal, :252-272 restoration)
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_slp_cols(SlpView sv, double *__restrict__ lb, double *__restrict__ ub,
                                                        double *__restrict__ c, int fr) {
    Map<BATCH> mp;
    const int B = sv.B;
    const double delta = sv.delta[mp.s];
    for (int64_t j = mp.first; j < sv.n; j += mp.stride) {
        const int64_t e = j * B + mp.s, eb = j * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double xk = sv.xk[e];
        lb[e] = pos_zero(fmax(-delta, sv.xL[eb] - xk));
        ub[e] = pos_zero(fmin(delta, sv.xU[eb] - xk));
        c[e] = fr ? 0.0 : sv.df[e];
    }
}
// row bounds g_L - b, g_U - b by row class (subproblem.jl:461-484); range rows stay two-sided
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_slp_rows(SlpView sv, double *__restrict__ rl, double *__restrict__ ru) {
    Map<BATCH> mp;
    const int B = sv.B;
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s, eb = i * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double b = sv.E[e];
        const double lo = sv.gL[eb] - b, up = sv.gU[eb] - b;
        const uint8_t cl = sv.cls[i];
        rl[e] = (cl == ROW_UPPER) ? -INFINITY : lo;
        ru[e] = (cl == ROW_EQ) ? lo : ((cl == ROW_LOWER) ? INFINITY : up);
    }
}
// feasibility restoration (subproblem.jl:277-382, :461-484): shifted right-hand sides and slack bounds.
// LP columns: p[0,n), then the slacks; LP rows: [0,m) and one extra <= row per range row.
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_fr_rows(SlpView sv, double *__restrict__ rl, double *__restrict__ ru,
                                                       double *__restrict__ lb, double *__restrict__ ub,
                                                       double *__restrict__ c) {
    Map<BATCH> mp;
    const int B = sv.B;
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s, eb = i * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double b = sv.E[e], gl = sv.gL[eb], gu = sv.gU[eb];
        double viol = 0.0;                       // :289-294
        if (b > gu)
            viol = gu - b;
        else if (b < gl)
            viol = gl - b;
        const double bs = b - fabs(viol);        // :295
        const uint8_t cl = sv.cls[i];
        const double lo = gl - bs, up = gu - bs;
        rl[e] = (cl == ROW_UPPER) ? -INFINITY : lo;
        ru[e] = (cl == ROW_EQ) ? lo : ((cl == ROW_UPPER) ? up : INFINITY);
        const int64_t c1 = (int64_t)sv.s1[i] * B + mp.s;
        const int s2 = sv.s2[i];
        if (s2 >= 0) {                           // two slacks (:298-361)
            const int64_t c2 = (int64_t)s2 * B + mp.s;
            if (viol < 0.0) {
                lb[c1] = 0.0;
                lb[c2] = viol;
            } else {
                lb[c1] = pos_zero(-viol);
                lb[c2] = 0.0;
            }
            ub[c2] = INFINITY;
            c[c2] = 1.0;
            const int a = sv.adj_of_row[i];
            if (a >= 0) {                        // extra <= row of a range row (:480-484)
                const int64_t er = (int64_t)(sv.m + a) * B + mp.s;
                rl[er] = -INFINITY;
                ru[er] = up;
            }
        } else {                                 // one slack (:362-378)
            lb[c1] = pos_zero(-fabs(viol));
        }
        ub[c1] = INFINITY;
        c[c1] = 1.0;
    }
}
// FR matrix values: Jacobian slots are gathered, slack coefficients are the constants +-1
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_fr_vals(const int *__restrict__ src, const double *__restrict__ jvals,
                                                       double *__restrict__ vals, int64_t nnz_fr, int B) {
    Map<BATCH> mp;
    for (int64_t k = mp.first; k < nnz_fr; k += mp.stride) {
        const int sidx = src[k];
        vals[k * B + mp.s] = sidx >= 0 ? jvals[(int64_t)sidx * B + mp.s] : (sidx == -1 ? 1.0 : -1.0);
    }
}

struct ExtractView {
    const double *xo, *yo, *dlo, *dup;  // LP solution (element-major)
    const ScenState *state;
    double *p, *lam, *muU, *muL, *pslack;  // outputs (element-major; pslack [2m][B])
    int *status;
};
// read-back of subproblem.jl:500-536
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_extract(SlpView sv, ExtractView ev, int fr) {
    Map<BATCH> mp;
    const int B = sv.B;
    const int status = ev.state[mp.s].status;
    const bool ok = status == ASM_LP_OPTIMAL;
    if (mp.first == 0) ev.status[mp.s] = status < 0 ? ASM_LP_ITERATION_LIMIT : status;
    for (int64_t j = mp.first; j < sv.n; j += mp.stride) {
        const int64_t e = j * B + mp.s, eb = j * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double pj = ok ? ev.xo[e] : 0.0;
        const double xk = sv.xk[e];
        double mu_u = ok ? ev.dup[e] : 0.0, mu_l = ok ? ev.dlo[e] : 0.0;
        if (pj < sv.xU[eb] - xk) mu_u = 0.0;  // :522-529: keep only multipliers of the original bounds
        if (pj > sv.xL[eb] - xk) mu_l = 0.0;
        ev.p[e] = pj;
        ev.muU[e] = mu_u;
        ev.muL[e] = mu_l;
    }
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        double l = ok ? ev.yo[e] : 0.0;
        double sl1 = 0.0, sl2 = 0.0;
        if (fr && ok) {
            const int a = sv.adj_of_row[i];
            if (a >= 0) l += ev.yo[(int64_t)(sv.m + a) * B + mp.s];  // :513-515
            sl1 = ev.xo[(int64_t)sv.s1[i] * B + mp.s];
            if (sv.s2[i] >= 0) sl2 = ev.xo[(int64_t)sv.s2[i] * B + mp.s];
        }
        ev.lam[e] = l;
        ev.pslack[(2 * i) * B + mp.s] = sl1;
        ev.pslack[(2 * i + 1) * B + mp.s] = sl2;
    }
}

// ---- merit / KKT reductions ------------------------------------------------------------------------------------
enum { R_A = 0, R_B, R_C, R_D, R_COUNT };

// norm_violations (common.jl:75-98): rows then columns; mode 0 = inf-norm, 1 = 1-norm, 2 = sum of squares
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_viol(SlpView sv, const double *__restrict__ E, const double *__restrict__ x,
                                                    int mode, double *partials) {
    Map<BATCH> mp;
    const int B = sv.B;
    double acc[1] = {0.0};
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s, eb = i * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double v = E[e], gu = sv.gU[eb], gl = sv.gL[eb];
        const double t = v > gu ? v - gu : (v < gl ? gl - v : 0.0);
        acc[0] = mode == 0 ? fmax(acc[0], fabs(t)) : (mode == 1 ? acc[0] + fabs(t) : acc[0] + t * t);
    }
    for (int64_t j = mp.first; j < sv.n; j += mp.stride) {
        const int64_t e = j * B + mp.s, eb = j * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double v = x[e], xu = sv.xU[eb], xl = sv.xL[eb];
        const double t = v > xu ? v - xu : (v < xl ? xl - v : 0.0);
        acc[0] = mode == 0 ? fmax(acc[0], fabs(t)) : (mode == 1 ? acc[0] + fabs(t) : acc[0] + t * t);
    }
    block_reduce_store<BATCH, 1>(acc, mode == 0 ? 1u : 0u, partials, R_A, B);
}
// row 2-norms of the assembled Jacobian, and max_i |lambda_i| * ||J_i|| (common.jl:40-42) when lam != null
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_row_norms(const int *__restrict__ row_ptr, const double *__restrict__ vals,
                                                         const double *__restrict__ lam, double *__restrict__ out, int m,
                                                         int B, double *partials) {
    Map<BATCH> mp;
    double acc[1] = {0.0};
    for (int64_t i = mp.first; i < m; i += mp.stride) {
        double a = 0.0;
        for (int k = row_ptr[i]; k < row_ptr[i + 1]; ++k) {
            const double t = vals[(int64_t)k * B + mp.s];
            a += t * t;
        }
        a = sqrt(a);
        if (out) out[i * B + mp.s] = a;
        if (lam) acc[0] = fmax(acc[0], fabs(lam[i * B + mp.s]) * a);
    }
    block_reduce_store<BATCH, 1>(acc, 1u, partials, R_B, B);
}
// KT residual vector df - J'lam - mu_U - mu_L (common.jl:38): sums of squares of the residual and of df
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_kt(const int *__restrict__ col_ptr, const int *__restrict__ row_idx,
                                                  const int *__restrict__ csc_src, const double *__restrict__ vals,
                                                  const double *__restrict__ df, const double *__restrict__ lam,
                                                  const double *__restrict__ muU, const double *__restrict__ muL, int n,
                                                  int B, double *partials) {
    Map<BATCH> mp;
    double acc[2] = {0.0, 0.0};
    for (int64_t j = mp.first; j < n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        double a = 0.0;
        for (int k = col_ptr[j]; k < col_ptr[j + 1]; ++k)
            a += vals[(int64_t)csc_src[k] * B + mp.s] * lam[(int64_t)row_idx[k] * B + mp.s];
        const double d = df[e];
        const double r = d - a - muU[e] - muL[e];
        acc[0] += r * r;
        acc[1] += d * d;
    }
    block_reduce_store<BATCH, 2>(acc, 0u, partials, R_C, B);
}
// norm_complementarity (common.jl:51-68), inf-norm: max |min(E-gL, gU-E) lam| over inequality rows, sum lam^2
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_compl(SlpView sv, const double *__restrict__ E,
                                                     const double *__restrict__ lam, double *partials) {
    Map<BATCH> mp;
    const int B = sv.B;
    double acc[2] = {0.0, 0.0};
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s, eb = i * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double gl = sv.gL[eb], gu = sv.gU[eb];
        if (gl != gu) {
            const double l = lam[e], v = E[e];
            acc[0] = fmax(acc[0], fabs(fmin(v - gl, gu - v) * l));
            acc[1] += l * l;
        }
    }
    block_reduce_store<BATCH, 2>(acc, 1u, partials, R_A, B);
}
// constraint part of compute_phi (slp.jl:79-115) and compute_derivative (slp.jl:122-147):
//   normal:      sum_i nu_i max(0, Et_i - gU_i, gL_i - Et_i)
//   restoration: sum_i nu_i max(0, lhs_i - gU_i, gL_i - lhs_i),  lhs = Et - viol(E) + alpha * (signed slacks),
//                plus sum of slacks (second slot)
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_merit(SlpView sv, const double *__restrict__ Et, const double *__restrict__ nu,
                                                     const double *__restrict__ pslack, const double *__restrict__ alpha,
                                                     int fr, double *partials) {
    Map<BATCH> mp;
    const int B = sv.B;
    const double al = alpha ? alpha[mp.s] : 0.0;
    double acc[2] = {0.0, 0.0};
    for (int64_t i = mp.first; i < sv.m; i += mp.stride) {
        const int64_t e = i * B + mp.s, eb = i * sv.Bb + (sv.Bb > 1 ? mp.s : 0);
        const double gl = sv.gL[eb], gu = sv.gU[eb];
        double lhs = Et[e];
        if (fr) {
            const double b = sv.E[e];
            const double viol = fmax(0.0, fmax(b - gu, gl - b));  // slp.jl:90-91
            lhs -= viol;
            const double s1 = pslack[(2 * i) * B + mp.s], s2 = pslack[(2 * i + 1) * B + mp.s];
            const uint8_t cl = sv.cls[i];
            if (cl == ROW_EQ || cl == ROW_RANGE)
                lhs += al * (s1 - s2);
            else if (cl == ROW_LOWER)
                lhs += al * s1;
            else
                lhs -= al * s1;
            acc[1] += s1 + s2;
        }
        acc[0] += nu[e] * fmax(0.0, fmax(lhs - gu, gl - lhs));
    }
    block_reduce_store<BATCH, 2>(acc, 0u, partials, R_A, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_dot(const double *__restrict__ a, const double *__restrict__ b, int64_t n,
                                                   int B, double *partials) {
    Map<BATCH> mp;
    double acc[1] = {0.0};
    for (int64_t j = mp.first; j < n; j += mp.stride) acc[0] += a[j * B + mp.s] * b[j * B + mp.s];
    block_reduce_store<BATCH, 1>(acc, 0u, partials, R_C, B);
}
// second stage of the small reductions: out[s * R_COUNT + q]
__global__ void __launch_bounds__(kFinalThreads) k_final(const double *partials, int nbx, int B, unsigned maxmask,
                                                          double *out) {
    const int s = blockIdx.x;
    for (int q = 0; q < R_COUNT; ++q) {
        double v = final_reduce(partials, q, nbx, B, s, (maxmask >> q) & 1u);
        if (threadIdx.x == 0) out[s * R_COUNT + q] = v;
    }
}

// =================================== device-side ACOPF evaluator ================================================
// SURVEY.md 8(f)-1: f, grad f, g and the Jacobian values of the ACP-polar OPF written straight into the SLP handle's
// device buffers (the role of the JuMP NLPEvaluator callbacks at /root/reference/src/MOI_wrapper.jl:1047-1069 and
// eval_functions!, src/algorithms/slp.jl:186-191), and compute_phi's trial evaluations g(x + alpha p), f(x + alpha p)
// (slp.jl:79-115, slp_line_search.jl:228-241) without a host round trip.  Variable / row / Jacobian layout is the one
// of activesetmethods_b200/examples/acopf.py (PowerModels' row classes in the order of MOI_wrapper.jl:683-689).
struct AcopfDev {
    int nb = 0, ng = 0, nl = 0, nd = 0, ref_bus = 0, nnz_bal = 0;
    // variable offsets, row offsets, Jacobian block offsets
    int o_va, o_vm, o_pg, o_qg, o_p, o_q, o_pdc, o_qdc;
    int r_angmax, r_angmin, r_ref, r_dc, r_thermal, r_bal, r_ohm;
    int k_angmax, k_angmin, k_ref, k_dc, k_thermal, k_bal, k_ohm;
    const int *f_bus, *t_bus, *bal_ptr, *bal_col;
    const double *coef, *gs, *bs, *cost2, *cost1, *cost0, *dc_loss1, *bal_coef;
};
struct AcopfIo {
    const double *xk, *p, *alpha;   // evaluation point x = xk (+ alpha p when TRIAL)
    double *f, *df, *E, *dE;        // outputs (df, dE unused when TRIAL)
    int B;
};
template <bool TRIAL>
__device__ __forceinline__ double acopf_x(const AcopfIo &io, int j, int s) {
    const double v = io.xk[(int64_t)j * io.B + s];
    return TRIAL ? v + io.alpha[s] * io.p[(int64_t)j * io.B + s] : v;
}
// one branch per item: angle-difference rows, thermal limits, Ohm's law rows and their derivatives
template <bool BATCH, bool TRIAL>
__global__ void __launch_bounds__(kThreads) k_acopf_branch(AcopfDev a, AcopfIo io) {
    Map<BATCH> mp;
    const int B = io.B, s = mp.s, nl = a.nl;
    for (int64_t l = mp.first; l < nl; l += mp.stride) {
        const int fb = a.f_bus[l], tb = a.t_bus[l];
        const double vaf = acopf_x<TRIAL>(io, a.o_va + fb, s), vat = acopf_x<TRIAL>(io, a.o_va + tb, s);
        const double vf = acopf_x<TRIAL>(io, a.o_vm + fb, s), vt = acopf_x<TRIAL>(io, a.o_vm + tb, s);
        const double pf = acopf_x<TRIAL>(io, a.o_p + (int)l, s), qf = acopf_x<TRIAL>(io, a.o_q + (int)l, s);
        const double pt = acopf_x<TRIAL>(io, a.o_p + nl + (int)l, s), qt = acopf_x<TRIAL>(io, a.o_q + nl + (int)l, s);
        const double d = vaf - vat;
        double sn, cs;
        sincos(d, &sn, &cs);
        const double vv = vf * vt;
        double c[12];
#pragma unroll
        for (int t = 0; t < 12; ++t) c[t] = a.coef[(int64_t)t * nl + l];
        auto E = [&](int row) -> double & { return io.E[(int64_t)row * B + s]; };
        E(a.r_angmax + (int)l) = d;
        E(a.r_angmin + (int)l) = d;
        E(a.r_thermal + 2 * (int)l) = pf * pf + qf * qf;
        E(a.r_thermal + 2 * (int)l + 1) = pt * pt + qt * qt;
        const double e_pf = c[0] * vf * vf + c[1] * vv * cs + c[2] * vv * sn;
        const double e_qf = c[3] * vf * vf + c[4] * vv * cs + c[5] * vv * sn;
        const double e_pt = c[6] * vt * vt + c[7] * vv * cs - c[8] * vv * sn;
        const double e_qt = c[9] * vt * vt + c[10] * vv * cs - c[11] * vv * sn;
        E(a.r_ohm + 4 * (int)l) = pf - e_pf;
        E(a.r_ohm + 4 * (int)l + 1) = qf - e_qf;
        E(a.r_ohm + 4 * (int)l + 2) = pt - e_pt;
        E(a.r_ohm + 4 * (int)l + 3) = qt - e_qt;
        if (!TRIAL) {
            auto J = [&](int k) -> double & { return io.dE[(int64_t)k * B + s]; };
            J(a.k_angmax + 2 * (int)l) = 1.0;
            J(a.k_angmax + 2 * (int)l + 1) = -1.0;
            J(a.k_angmin + 2 * (int)l) = 1.0;
            J(a.k_angmin + 2 * (int)l + 1) = -1.0;
            J(a.k_thermal + 4 * (int)l) = 2.0 * pf;
            J(a.k_thermal + 4 * (int)l + 1) = 2.0 * qf;
            J(a.k_thermal + 4 * (int)l + 2) = 2.0 * pt;
            J(a.k_thermal + 4 * (int)l + 3) = 2.0 * qt;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const double aa = c[3 * r], bb = c[3 * r + 1], cc = c[3 * r + 2];
                const bool own_from = r < 2;
                const double sgn = own_from ? 1.0 : -1.0;
                const double cross = bb * cs + sgn * cc * sn;
                const int k0 = a.k_ohm + 20 * (int)l + 5 * r;
                J(k0) = 1.0;
                if (own_from) {
                    J(k0 + 1) = -(2.0 * aa * vf + cross * vt);
                    J(k0 + 2) = -(cross * vf);
                } else {
                    J(k0 + 1) = -(cross * vt);
                    J(k0 + 2) = -(2.0 * aa * vt + cross * vf);
                }
                const double dd = vv * (-bb * sn + sgn * cc * cs);
                J(k0 + 3) = -dd;
                J(k0 + 4) = dd;
            }
        }
    }
}
// one balance row per item (2 per bus: P, Q): affine entries in j_str order, shunt term, and their derivatives
template <bool BATCH, bool TRIAL>
__global__ void __launch_bounds__(kThreads) k_acopf_bus(AcopfDev a, AcopfIo io) {
    Map<BATCH> mp;
    const int B = io.B, s = mp.s;
    for (int64_t r = mp.first; r < 2 * a.nb; r += mp.stride) {
        const int bus = (int)(r >> 1), is_q = (int)(r & 1);
        const double vm = acopf_x<TRIAL>(io, a.o_vm + bus, s);
        double acc = 0.0;
        for (int k = a.bal_ptr[r]; k < a.bal_ptr[r + 1]; ++k) {
            const double cf = a.bal_coef[k];
            const bool shunt = cf != cf;   // NaN marks the vm^2 slot
            acc += (shunt ? 0.0 : cf) * acopf_x<TRIAL>(io, a.bal_col[k], s);
            if (!TRIAL)
                io.dE[(int64_t)(a.k_bal + k) * B + s] = shunt ? (is_q ? -2.0 * a.bs[bus] : 2.0 * a.gs[bus]) * vm : cf;
        }
        acc += is_q ? -(a.bs[bus] * vm * vm) : a.gs[bus] * vm * vm;
        io.E[(int64_t)(a.r_bal + r) * B + s] = acc;
    }
}
// objective, its gradient, reference-angle row and dc-line loss rows: one thread per scenario
template <bool TRIAL>
__global__ void k_acopf_misc(AcopfDev a, AcopfIo io, int n) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= io.B) return;
    const int B = io.B;
    double f = 0.0;
    for (int k = 0; k < a.ng; ++k) {
        const double pg = acopf_x<TRIAL>(io, a.o_pg + k, s);
        f += a.cost2[k] * pg * pg + a.cost1[k] * pg + a.cost0[k];
        if (!TRIAL) io.df[(int64_t)(a.o_pg + k) * B + s] = 2.0 * a.cost2[k] * pg + a.cost1[k];
    }
    io.f[s] = f;
    io.E[(int64_t)a.r_ref * B + s] = acopf_x<TRIAL>(io, a.o_va + a.ref_bus, s);
    if (!TRIAL) io.dE[(int64_t)a.k_ref * B + s] = 1.0;
    for (int d = 0; d < a.nd; ++d) {
        const double pf = acopf_x<TRIAL>(io, a.o_pdc + d, s), pt = acopf_x<TRIAL>(io, a.o_pdc + a.nd + d, s);
        io.E[(int64_t)(a.r_dc + d) * B + s] = (1.0 - a.dc_loss1[d]) * pf + pt;
        if (!TRIAL) {
            io.dE[(int64_t)(a.k_dc + 2 * d) * B + s] = 1.0 - a.dc_loss1[d];
            io.dE[(int64_t)(a.k_dc + 2 * d + 1) * B + s] = 1.0;
        }
    }
}

// =================================== host side: pattern analysis ================================================
struct Pattern {
    int n = 0, m = 0;
    int64_t nnz_coo = 0, nnz = 0;
    std::vector<int64_t> row_ptr;  // CSR of the deduplicated Jacobian
    std::vector<int32_t> col_idx;
    std::vector<int> dup_ptr, dup_idx;  // per slot: COO entries in j_str order
    std::vector<int> slot_of_coo;

    int analyse(int n_, int m_, int64_t nz, const int64_t *jr, const int64_t *jc) {
        n = n_;
        m = m_;
        nnz_coo = nz;
        if (nz > 0x7fffffffLL) return fail(ASM_E_INVALID, "too many Jacobian entries");
        std::vector<int> order(nz);
        std::iota(order.begin(), order.end(), 0);
        for (int64_t k = 0; k < nz; ++k)
            if (jr[k] < 1 || jr[k] > m || jc[k] < 1 || jc[k] > n)
                return fail(ASM_E_INVALID, "j_str entry out of range (expected 1-based row <= m, col <= n)");
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
            if (jr[a] != jr[b]) return jr[a] < jr[b];
            return jc[a] < jc[b];
        });
        row_ptr.assign(m + 1, 0);
        col_idx.clear();
        dup_ptr.clear();
        dup_idx.resize(nz);
        slot_of_coo.resize(nz);
        int64_t slot = -1;
        for (int64_t t = 0; t < nz; ++t) {
            const int k = order[t];
            if (t == 0 || jr[k] != jr[order[t - 1]] || jc[k] != jc[order[t - 1]]) {
                ++slot;
                dup_ptr.push_back((int)t);
                col_idx.push_back((int32_t)(jc[k] - 1));
                row_ptr[jr[k]]++;
            }
            dup_idx[t] = k;
            slot_of_coo[k] = (int)slot;
        }
        dup_ptr.push_back((int)nz);
        nnz = slot + 1;
        for (int i = 0; i < m; ++i) row_ptr[i + 1] += row_ptr[i];
        return ASM_OK;
    }
};

struct SlpHandle {
    int n = 0, m = 0, B = 1, Buser = 1, Bb = 1, device = 0;
    Pattern pat;
    cudaStream_t stream = nullptr;
    // row structure (host)
    std::vector<uint8_t> cls;
    std::vector<int> s1, s2, adj, adj_of_row;
    int ncol_fr = 0, nrow_fr = 0;
    int64_t nnz_fr = 0;
    // device
    DBuf<int> dup_ptr, dup_idx, d_s1, d_s2, d_adj, d_adj_of_row, fr_src;
    DBuf<uint8_t> d_cls;
    DBuf<double> xL, xU, gL, gU, xk, df, E, dE, fval, delta, d_alpha;
    DBuf<double> p, lam, muU, muL, pslack, tmp_m, tmp_m2, tmp_n, tmp_n2, tmp_n3, small_out, partials;
    DBuf<int> d_status;
    DBuf<double> stage;
    // device staging for layout changes
    PinnedRing ring;   // host -> device copies of pageable caller arrays (see util.cuh)
    std::unique_ptr<LpSolver> normal, fr;
    std::vector<int32_t> mask;   // asm_slp_set_active (kept for the restoration solver, which is built lazily)
    int phase = -1;  // phase of the last update
    bool solved = false, extracted = false;
    Pinned pin_small;
    int64_t own_launches = 0;
    cudaEvent_t tev0 = nullptr, tev1 = nullptr;
    // device-side ACOPF evaluator (optional)
    bool has_acopf = false;
    AcopfDev acopf;
    DBuf<int> ac_f, ac_t, ac_bal_ptr, ac_bal_col;
    DBuf<double> ac_coef, ac_gs, ac_bs, ac_c2, ac_c1, ac_c0, ac_loss1, ac_bal_coef, ac_ftrial;

    ~SlpHandle() {
        normal.reset();
        fr.reset();
        if (tev0) cudaEventDestroy(tev0);
        if (tev1) cudaEventDestroy(tev1);
        if (stream) cudaStreamDestroy(stream);
    }
    LpSolver *cur() { return phase == 1 ? fr.get() : normal.get(); }

    SlpView view() {
        SlpView v;
        v.n = n;
        v.m = m;
        v.B = B;
        v.Bb = Bb;
        v.n_adj = (int)adj.size();
        v.xL = xL.p;
        v.xU = xU.p;
        v.gL = gL.p;
        v.gU = gU.p;
        v.xk = xk.p;
        v.df = df.p;
        v.E = E.p;
        v.delta = delta.p;
        v.cls = d_cls.p;
        v.s1 = d_s1.p;
        v.s2 = d_s2.p;
        v.adj = d_adj.p;
        v.adj_of_row = d_adj_of_row.p;
        return v;
    }

    // host [S][len] -> device [len][B]
    int put(const double *host, int64_t len, int S, double *dst) {
        if (len == 0) return ASM_OK;
        if (B == 1) return ring.h2d(dst, host, len * sizeof(double), stream);
        if (stage.n < (size_t)len * S) {
            ASM_CK(cudaStreamSynchronize(stream));   // earlier layout kernels may still read the old buffer
            ASM_TRY(stage.alloc((size_t)len * S));
        }
        ASM_TRY(ring.h2d(stage.p, host, (size_t)len * S * sizeof(double), stream));
        dim3 grid((unsigned)((len + 31) / 32), B / 32), block(32, 8);
        k_layout_in<<<grid, block, 0, stream>>>(stage.p, dst, len, S, B);
        ++own_launches;
        return ASM_OK;
    }
    // device [len][B] -> host [Buser][len]
    int get(const double *src, int64_t len, double *host) {
        if (len == 0 || !host) return ASM_OK;
        if (B == 1) {
            ASM_CK(cudaMemcpyAsync(host, src, len * sizeof(double), cudaMemcpyDeviceToHost, stream));
            return ASM_OK;
        }
        if (stage.n < (size_t)len * Buser) {
            ASM_CK(cudaStreamSynchronize(stream));   // earlier copies may still read the old buffer
            ASM_TRY(stage.alloc((size_t)len * Buser));
        }
        dim3 grid((unsigned)((len + 31) / 32), B / 32), block(32, 8);
        k_layout_out<<<grid, block, 0, stream>>>(src, stage.p, len, Buser, B);
        ++own_launches;
        // stream order protects the staging buffer (the next get()'s kernel runs after this copy); the caller of get()
        // synchronises ONCE, after its last array
        ASM_CK(cudaMemcpyAsync(host, stage.p, (size_t)len * Buser * sizeof(double), cudaMemcpyDeviceToHost, stream));
        return ASM_OK;
    }

    int create(int n_, int m_, int64_t nz, const int64_t *jr, const int64_t *jc, const double *hxL, const double *hxU,
               const double *hgL, const double *hgU, int batch, int per_scen, int dev) {
        n = n_;
        m = m_;
        Buser = batch;
        B = pad_batch(batch);
        Bb = (per_scen && B > 1) ? B : 1;
        device = dev;
        if (n <= 0 || m < 0 || nz < 0 || batch < 1) return fail(ASM_E_INVALID, "bad dimensions");
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
            return fail(ASM_E_CUDA, "no CUDA device: this library has no CPU fallback");
        if (dev < 0 || dev >= ndev) return fail(ASM_E_INVALID, "device index out of range");
        ASM_CK(cudaSetDevice(dev));
        ASM_TRY(pat.analyse(n, m, nz, jr, jc));
        // row classes from the bounds of scenario 0; every scenario must agree (one LP skeleton per handle)
        cls.resize(m);
        s1.assign(m, 0);
        s2.assign(m, -1);
        adj_of_row.assign(m, -1);
        const int S = per_scen ? batch : 1;
        int col = n;
        for (int i = 0; i < m; ++i) {
            auto classify = [&](double l, double u, uint8_t &out) -> int {
                const bool lf = l > -INFINITY, uf = u < INFINITY;
                if (!lf && !uf) return ASM_E_FREE_ROW;
                if (l == u)
                    out = ROW_EQ;
                else if (lf && uf)
                    out = ROW_RANGE;
                else if (lf)
                    out = ROW_LOWER;
                else
                    out = ROW_UPPER;
                return ASM_OK;
            };
            uint8_t c0 = 0;
            if (classify(hgL[i], hgU[i], c0) != ASM_OK)
                return fail(ASM_E_FREE_ROW, "row with two infinite bounds (unsupported by the reference builder)");
            for (int s = 1; s < S; ++s) {
                uint8_t cs = 0;
                if (classify(hgL[(size_t)s * m + i], hgU[(size_t)s * m + i], cs) != ASM_OK || cs != c0)
                    return fail(ASM_E_INVALID, "row classes differ between scenarios");
            }
            cls[i] = c0;
            s1[i] = col++;
            if (c0 == ROW_EQ || c0 == ROW_RANGE) s2[i] = col++;  // subproblem.jl:87: two slacks iff both bounds finite
            if (c0 == ROW_RANGE) {
                adj_of_row[i] = (int)adj.size();
                adj.push_back(i);
            }
        }
        ncol_fr = col;
        nrow_fr = m + (int)adj.size();
        ASM_CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        normal.reset(new LpSolver());
        ASM_TRY(normal->init(n, m, pat.nnz, pat.row_ptr.data(), pat.col_idx.data(), batch, stream));
        ASM_TRY(dup_ptr.alloc(pat.dup_ptr.size()));
        ASM_TRY(dup_idx.alloc(pat.dup_idx.size()));
        ASM_CK(cudaMemcpy(dup_ptr.p, pat.dup_ptr.data(), pat.dup_ptr.size() * sizeof(int), cudaMemcpyHostToDevice));
        if (nz) ASM_CK(cudaMemcpy(dup_idx.p, pat.dup_idx.data(), nz * sizeof(int), cudaMemcpyHostToDevice));
        ASM_TRY(d_cls.alloc(m));
        ASM_TRY(d_s1.alloc(m));
        ASM_TRY(d_s2.alloc(m));
        ASM_TRY(d_adj_of_row.alloc(m));
        ASM_TRY(d_adj.alloc(adj.size()));
        if (m) {
            ASM_CK(cudaMemcpy(d_cls.p, cls.data(), m, cudaMemcpyHostToDevice));
            ASM_CK(cudaMemcpy(d_s1.p, s1.data(), m * sizeof(int), cudaMemcpyHostToDevice));
            ASM_CK(cudaMemcpy(d_s2.p, s2.data(), m * sizeof(int), cudaMemcpyHostToDevice));
            ASM_CK(cudaMemcpy(d_adj_of_row.p, adj_of_row.data(), m * sizeof(int), cudaMemcpyHostToDevice));
        }
        if (!adj.empty()) ASM_CK(cudaMemcpy(d_adj.p, adj.data(), adj.size() * sizeof(int), cudaMemcpyHostToDevice));
        const size_t nB = (size_t)n * B, mB = (size_t)m * B;
        ASM_TRY(xL.alloc((size_t)n * Bb));
        ASM_TRY(xU.alloc((size_t)n * Bb));
        ASM_TRY(gL.alloc((size_t)m * Bb));
        ASM_TRY(gU.alloc((size_t)m * Bb));
        DBuf<double> *nb[] = {&xk, &df, &p, &muU, &muL, &tmp_n, &tmp_n2, &tmp_n3};
        for (auto *b : nb) ASM_TRY(b->alloc(nB));
        DBuf<double> *mb[] = {&E, &lam, &tmp_m, &tmp_m2};
        for (auto *b : mb) ASM_TRY(b->alloc(mB));
        ASM_TRY(pslack.alloc(2 * mB));
        ASM_TRY(dE.alloc((size_t)nz * B));
        ASM_TRY(fval.alloc(B));
        ASM_TRY(delta.alloc(B));
        ASM_TRY(d_alpha.alloc(B));
        ASM_TRY(d_status.alloc(B));
        ASM_TRY(small_out.alloc((size_t)B * R_COUNT));
        ASM_TRY(partials.alloc((size_t)R_COUNT * kMaxBlocksX * B));
        ASM_TRY(pin_small.reserve(sizeof(double) * (size_t)B * (R_COUNT + 4)));
        ASM_TRY(pslack.zero(stream));
        ASM_TRY(lam.zero(stream));
        ASM_TRY(p.zero(stream));
        if (Bb == 1) {
            ASM_CK(cudaMemcpyAsync(xL.p, hxL, n * sizeof(double), cudaMemcpyHostToDevice, stream));
            ASM_CK(cudaMemcpyAsync(xU.p, hxU, n * sizeof(double), cudaMemcpyHostToDevice, stream));
            ASM_CK(cudaMemcpyAsync(gL.p, hgL, m * sizeof(double), cudaMemcpyHostToDevice, stream));
            ASM_CK(cudaMemcpyAsync(gU.p, hgU, m * sizeof(double), cudaMemcpyHostToDevice, stream));
        } else {
            ASM_TRY(put(hxL, n, batch, xL.p));
            ASM_TRY(put(hxU, n, batch, xU.p));
            ASM_TRY(put(hgL, m, batch, gL.p));
            ASM_TRY(put(hgU, m, batch, gU.p));
        }
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    // LP of the restoration phase in the reference's column / row layout (subproblem.jl:75-214)
    int build_fr() {
        if (fr) return ASM_OK;
        std::vector<int64_t> rp(nrow_fr + 1, 0);
        std::vector<int32_t> ci;
        std::vector<int> src;
        ci.reserve(pat.nnz + 2 * (size_t)m);
        src.reserve(pat.nnz + 2 * (size_t)m);
        auto push_row = [&](int i, bool extra) {
            for (int64_t k = pat.row_ptr[i]; k < pat.row_ptr[i + 1]; ++k) {
                ci.push_back(pat.col_idx[k]);
                src.push_back((int)k);
            }
            if (!extra) {
                // row i: +s1 (>= rows and equalities), -s1 (<= rows); equalities also -s2
                ci.push_back(s1[i]);
                src.push_back(cls[i] == ROW_UPPER ? -2 : -1);
                if (cls[i] == ROW_EQ) {
                    ci.push_back(s2[i]);
                    src.push_back(-2);
                }
            } else {
                ci.push_back(s2[i]);  // extra <= row of a range row carries -s2 (subproblem.jl:200-214)
                src.push_back(-2);
            }
        };
        for (int i = 0; i < m; ++i) {
            push_row(i, false);
            rp[i + 1] = (int64_t)ci.size();
        }
        for (size_t a = 0; a < adj.size(); ++a) {
            push_row(adj[a], true);
            rp[m + a + 1] = (int64_t)ci.size();
        }
        nnz_fr = (int64_t)ci.size();
        fr.reset(new LpSolver());
        ASM_TRY(fr->init(ncol_fr, nrow_fr, nnz_fr, rp.data(), ci.data(), Buser, stream));
        if (!mask.empty()) ASM_TRY(fr->set_active(mask.data()));
        ASM_TRY(fr_src.alloc(src.size()));
        ASM_CK(cudaMemcpy(fr_src.p, src.data(), src.size() * sizeof(int), cudaMemcpyHostToDevice));
        return ASM_OK;
    }

    int update(const double *hx, const double *hf, const double *hdf, const double *hE, const double *hdE,
               const double *hdelta, int feas) {
        if (!hx || !hdf || !hE || !hdE || !hdelta) return fail(ASM_E_INVALID, "null input to asm_slp_update");
        ASM_CK(cudaSetDevice(device));
        ASM_TRY(put(hx, n, Buser, xk.p));
        ASM_TRY(put(hdf, n, Buser, df.p));
        ASM_TRY(put(hE, m, Buser, E.p));
        ASM_TRY(put(hdE, pat.nnz_coo, Buser, dE.p));
        // per-scenario scalars (padding replicates scenario 0)
        double *ps = (double *)pin_small.p;
        for (int s = 0; s < B; ++s) {
            ps[s] = hdelta[s < Buser ? s : 0];
            ps[B + s] = hf ? hf[s < Buser ? s : 0] : 0.0;
        }
        ASM_CK(cudaMemcpyAsync(delta.p, ps, B * sizeof(double), cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaMemcpyAsync(fval.p, ps + B, B * sizeof(double), cudaMemcpyHostToDevice, stream));
        return update_device(feas);
    }

    // everything after the copies: assemble + bounds on the device
    int update_device(int feas) {
        SlpView sv = view();
        const Geo gz = geo_for(pat.nnz, B), gc = geo_for(n, B), gr = geo_for(m, B);
#define SLP_KB(kern, geo, ...)                                                \
    do {                                                                      \
        if (B > 1)                                                            \
            kern<true><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__);  \
        else                                                                  \
            kern<false><<<(geo).grid, (geo).block, 0, stream>>>(__VA_ARGS__); \
        ++own_launches;                                                       \
    } while (0)
        SLP_KB(k_assemble, gz, dup_ptr.p, dup_idx.p, dE.p, normal->vals.p, pat.nnz, B);
        if (!feas) {
            SLP_KB(k_slp_cols, gc, sv, normal->lb.p, normal->ub.p, normal->c.p, 0);
            SLP_KB(k_slp_rows, gr, sv, normal->rl.p, normal->ru.p);
            ASM_CK(cudaMemcpyAsync(normal->c0.p, fval.p, B * sizeof(double), cudaMemcpyDeviceToDevice, stream));
            phase = 0;
        } else {
            ASM_TRY(build_fr());
            const Geo gf = geo_for(nnz_fr, B);
            SLP_KB(k_fr_vals, gf, fr_src.p, normal->vals.p, fr->vals.p, nnz_fr, B);
            SLP_KB(k_slp_cols, gc, sv, fr->lb.p, fr->ub.p, fr->c.p, 1);
            SLP_KB(k_fr_rows, gr, sv, fr->rl.p, fr->ru.p, fr->lb.p, fr->ub.p, fr->c.p);
            ASM_TRY(fr->c0.zero(stream));
            phase = 1;
        }
        ASM_CK(cudaGetLastError());
        solved = false;
        extracted = false;
        return ASM_OK;
    }

    int solve(const asm_lp_params *P, asm_lp_info *info) {
        if (phase < 0) return fail(ASM_E_STATE, "asm_slp_solve before asm_slp_update");
        ASM_CK(cudaSetDevice(device));
        asm_lp_params dflt;
        if (!P) {
            asm_lp_default_params(&dflt);
            P = &dflt;
        }
        ASM_TRY(cur()->solve(*P, info));
        solved = true;
        extracted = false;
        return ASM_OK;
    }

    int extract_device() {
        if (!solved) return fail(ASM_E_STATE, "extract before solve");
        if (extracted) return ASM_OK;
        LpSolver *lp = cur();
        SlpView sv = view();
        ExtractView ev;
        ev.xo = lp->xo.p;
        ev.yo = lp->yo.p;
        ev.dlo = lp->dlo.p;
        ev.dup = lp->dup.p;
        ev.state = lp->state.p;
        ev.p = p.p;
        ev.lam = lam.p;
        ev.muU = muU.p;
        ev.muL = muL.p;
        ev.pslack = pslack.p;
        ev.status = d_status.p;
        const Geo g = geo_for(std::max(n, m), B);
        SLP_KB(k_extract, g, sv, ev, phase);
        ASM_CK(cudaGetLastError());
        extracted = true;
        return ASM_OK;
    }

    int extract(double *hp, double *hlam, double *hmuU, double *hmuL, double *hslack, int32_t *hstatus) {
        ASM_CK(cudaSetDevice(device));
        ASM_TRY(extract_device());
        ASM_TRY(get(p.p, n, hp));
        ASM_TRY(get(lam.p, m, hlam));
        ASM_TRY(get(muU.p, n, hmuU));
        ASM_TRY(get(muL.p, n, hmuL));
        if (hslack) {
            // device [2m][B] -> host [Buser][m][2]
            ASM_TRY(get(pslack.p, 2 * (int64_t)m, hslack));
        }
        if (hstatus) ASM_CK(cudaMemcpyAsync(hstatus, d_status.p, Buser * sizeof(int), cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        return ASM_OK;
    }

    // small reductions: run the second stage and bring R_COUNT doubles per scenario to the host
    int finish_reduce(int nbx, unsigned maxmask, std::vector<double> &out) {
        k_final<<<B, kFinalThreads, 0, stream>>>(partials.p, nbx, B, maxmask, small_out.p);
        ++own_launches;
        ASM_CK(cudaGetLastError());
        double *ps = (double *)pin_small.p;
        ASM_CK(cudaMemcpyAsync(ps, small_out.p, sizeof(double) * B * R_COUNT, cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        out.assign(ps, ps + (size_t)B * R_COUNT);
        return ASM_OK;
    }
};

}  // namespace asmb

using namespace asmb;

// ================================================= C ABI =======================================================
struct asm_slp {
    SlpHandle h;
};
struct asm_lp {
    LpSolver own;
    std::unique_ptr<DistLp> dist;  // row-partitioned instance (lp_dist.cuh); `s` is then its local block
    LpSolver &s;
    int device = 0;
    explicit asm_lp(bool partitioned) : dist(partitioned ? new DistLp() : nullptr), s(partitioned ? dist->lp : own) {}
    DBuf<double> stage;
    PinnedRing ring;
    int put(const double *host, int64_t len, int S, double *dst) {
        if (len == 0) return ASM_OK;
        if (s.B == 1) return ring.h2d(dst, host, len * sizeof(double), s.stream);
        if (stage.n < (size_t)len * S) ASM_TRY(stage.alloc((size_t)len * S));
        ASM_TRY(ring.h2d(stage.p, host, (size_t)len * S * sizeof(double), s.stream));
        dim3 grid((unsigned)((len + 31) / 32), s.B / 32), block(32, 8);
        k_layout_in<<<grid, block, 0, s.stream>>>(stage.p, dst, len, S, s.B);
        ASM_CK(cudaStreamSynchronize(s.stream));
        return ASM_OK;
    }
    int get(const double *src, int64_t len, double *host) {
        if (len == 0 || !host) return ASM_OK;
        if (s.B == 1) {
            ASM_CK(cudaMemcpyAsync(host, src, len * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
            ASM_CK(cudaStreamSynchronize(s.stream));
            return ASM_OK;
        }
        if (stage.n < (size_t)len * s.Buser) ASM_TRY(stage.alloc((size_t)len * s.Buser));
        dim3 grid((unsigned)((len + 31) / 32), s.B / 32), block(32, 8);
        k_layout_out<<<grid, block, 0, s.stream>>>(src, stage.p, len, s.Buser, s.B);
        ASM_CK(cudaMemcpyAsync(host, stage.p, (size_t)len * s.Buser * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
        ASM_CK(cudaStreamSynchronize(s.stream));
        return ASM_OK;
    }
};

extern "C" {

const char *asm_last_error(void) { return err_slot().c_str(); }
const char *asm_version(void) { return "asm_b200 0.1 (sm_100a)"; }
int asm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void asm_lp_default_params(asm_lp_params *p) {
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->eps_rel = 1e-8;
    p->eps_infeas = 1e-9;
    p->max_iter = 2000000;
    p->check_every = 64;
    p->ruiz_iters = 10;
    p->warm_start = 0;
    p->verbose = 0;
    p->restart_sufficient = 0.2;
    p->restart_necessary = 0.8;
    p->restart_artificial = 0.36;
    p->pid_kp = 0.5;
    p->pid_ki = 0.0;
    p->pid_kd = 0.0;
    p->engine = 0;
    p->group_size = 0;
    p->hand_over = 0.5;
    p->ipm_max_iter = 200;
    p->ipm_refine = 0;
    p->ipm_reg = 1e-8;
    p->ipm_prox = 1e-7;
}

// ---- generic LP -------------------------------------------------------------------------------------------------
int asm_lp_create(int32_t n_cols, int32_t n_rows, int64_t nnz, const int64_t *row_ptr, const int32_t *col_idx,
                  int32_t batch, int32_t device, asm_lp **out) {
    if (!out || !row_ptr || (nnz > 0 && !col_idx)) return fail(ASM_E_INVALID, "null argument");
    *out = nullptr;
    int ndev = asm_device_count();
    if (ndev == 0) return fail(ASM_E_CUDA, "no CUDA device: this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(ASM_E_INVALID, "device index out of range");
    ASM_CK(cudaSetDevice(device));
    asm_lp *h = new (std::nothrow) asm_lp(false);
    if (!h) return fail(ASM_E_INVALID, "out of host memory");
    h->device = device;
    int rc = h->s.init(n_cols, n_rows, nnz, row_ptr, col_idx, batch, nullptr);
    if (rc != ASM_OK) {
        delete h;
        return rc;
    }
    // defaults: free columns, free rows are not allowed to stay (caller sets bounds)
    *out = h;
    return ASM_OK;
}
void asm_lp_destroy(asm_lp *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h;
}
int asm_lp_set_matrix_values(asm_lp *h, const double *vals) {
    if (!h || !vals) return fail(ASM_E_INVALID, "null argument");
    ASM_CK(cudaSetDevice(h->device));
    return h->put(vals, h->s.nnz, h->s.Buser, h->s.vals.p);
}
int asm_lp_set_objective(asm_lp *h, const double *c, const double *c0) {
    if (!h || !c) return fail(ASM_E_INVALID, "null argument");
    ASM_CK(cudaSetDevice(h->device));
    ASM_TRY(h->put(c, h->s.n, h->s.Buser, h->s.c.p));
    std::vector<double> t(h->s.B, 0.0);
    if (c0)
        for (int s = 0; s < h->s.B; ++s) t[s] = c0[s < h->s.Buser ? s : 0];
    ASM_CK(cudaMemcpy(h->s.c0.p, t.data(), sizeof(double) * h->s.B, cudaMemcpyHostToDevice));
    return ASM_OK;
}
int asm_lp_set_col_bounds(asm_lp *h, const double *lb, const double *ub) {
    if (!h || !lb || !ub) return fail(ASM_E_INVALID, "null argument");
    ASM_CK(cudaSetDevice(h->device));
    ASM_TRY(h->put(lb, h->s.n, h->s.Buser, h->s.lb.p));
    return h->put(ub, h->s.n, h->s.Buser, h->s.ub.p);
}
int asm_lp_set_row_bounds(asm_lp *h, const double *rl, const double *ru) {
    if (!h || !rl || !ru) return fail(ASM_E_INVALID, "null argument");
    ASM_CK(cudaSetDevice(h->device));
    ASM_TRY(h->put(rl, h->s.m, h->s.Buser, h->s.rl.p));
    return h->put(ru, h->s.m, h->s.Buser, h->s.ru.p);
}
int asm_lp_solve(asm_lp *h, const asm_lp_params *params, asm_lp_info *info) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    ASM_CK(cudaSetDevice(h->device));
    asm_lp_params d;
    if (!params) {
        asm_lp_default_params(&d);
        params = &d;
    }
    if (h->dist) return h->dist->solve(*params, info);
    return h->s.solve(*params, info);
}
int asm_lp_get_primal(asm_lp *h, double *x) {
    if (!h || !x) return fail(ASM_E_INVALID, "null argument");
    if (!h->s.has_solution) return fail(ASM_E_STATE, "no solution yet");
    ASM_CK(cudaSetDevice(h->device));
    return h->get(h->s.xo.p, h->s.n, x);
}
int asm_lp_get_row_dual(asm_lp *h, double *y) {
    if (!h || !y) return fail(ASM_E_INVALID, "null argument");
    if (!h->s.has_solution) return fail(ASM_E_STATE, "no solution yet");
    ASM_CK(cudaSetDevice(h->device));
    return h->get(h->s.yo.p, h->s.m, y);
}
int asm_lp_get_col_dual(asm_lp *h, double *dual_lb, double *dual_ub) {
    if (!h) return fail(ASM_E_INVALID, "null argument");
    if (!h->s.has_solution) return fail(ASM_E_STATE, "no solution yet");
    ASM_CK(cudaSetDevice(h->device));
    ASM_TRY(h->get(h->s.dlo.p, h->s.n, dual_lb));
    return h->get(h->s.dup.p, h->s.n, dual_ub);
}
int asm_lp_set_start(asm_lp *h, const double *x, const double *y) {
    if (!h) return fail(ASM_E_INVALID, "null argument");
    ASM_CK(cudaSetDevice(h->device));
    if (x) ASM_TRY(h->put(x, h->s.n, h->s.Buser, h->s.xo.p));
    if (y) ASM_TRY(h->put(y, h->s.m, h->s.Buser, h->s.yo.p));
    ASM_CK(cudaStreamSynchronize(h->s.stream));
    h->s.has_solution = true;
    return ASM_OK;
}

// ---- row-partitioned single LP over NCCL ------------------------------------------------------------------------
int asm_dist_unique_id(char *id128) {
    if (!id128) return fail(ASM_E_INVALID, "null argument");
    ASM_TRY(nccl().load());
    NcclApi::UniqueId id;
    ASM_NCCL(nccl().GetUniqueId(&id));
    memcpy(id128, id.internal, sizeof id.internal);
    return ASM_OK;
}
int asm_lp_dist_create(int32_t n_cols, int32_t n_rows_local, int64_t nnz_local, const int64_t *row_ptr,
                       const int32_t *col_idx, int32_t rank, int32_t world, const char *id128, int32_t device,
                       asm_lp **out) {
    if (!out || !row_ptr || (nnz_local > 0 && !col_idx) || !id128) return fail(ASM_E_INVALID, "null argument");
    *out = nullptr;
    int ndev = asm_device_count();
    if (ndev == 0) return fail(ASM_E_CUDA, "no CUDA device: this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(ASM_E_INVALID, "device index out of range");
    asm_lp *h = new (std::nothrow) asm_lp(true);
    if (!h) return fail(ASM_E_INVALID, "out of host memory");
    h->device = device;
    int rc = h->dist->init(n_cols, n_rows_local, nnz_local, row_ptr, col_idx, rank, world, id128, device);
    if (rc != ASM_OK) {
        delete h;
        return rc;
    }
    *out = h;
    return ASM_OK;
}

// ---- SLP fast path --------------------------------------------------------------------------------------------
int asm_slp_create(int32_t n, int32_t m, int64_t nnz_coo, const int64_t *j_row, const int64_t *j_col,
                   const double *x_L, const double *x_U, const double *g_L, const double *g_U, int32_t batch,
                   int32_t per_scenario_bounds, int32_t device, asm_slp **out) {
    if (!out) return fail(ASM_E_INVALID, "null out pointer");
    *out = nullptr;
    if ((nnz_coo > 0 && (!j_row || !j_col)) || !x_L || !x_U || (m > 0 && (!g_L || !g_U)))
        return fail(ASM_E_INVALID, "null argument");
    asm_slp *h = new (std::nothrow) asm_slp();
    if (!h) return fail(ASM_E_INVALID, "out of host memory");
    int rc = h->h.create(n, m, nnz_coo, j_row, j_col, x_L, x_U, g_L, g_U, batch, per_scenario_bounds, device);
    if (rc != ASM_OK) {
        delete h;
        return rc;
    }
    *out = h;
    return ASM_OK;
}
void asm_slp_destroy(asm_slp *h) {
    if (!h) return;
    cudaSetDevice(h->h.device);
    delete h;
}
int asm_slp_sizes(asm_slp *h, int64_t *nnz_csr, int32_t *lp_cols, int32_t *lp_rows) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    if (nnz_csr) *nnz_csr = h->h.pat.nnz;
    if (lp_cols) *lp_cols = h->h.ncol_fr;
    if (lp_rows) *lp_rows = h->h.nrow_fr;
    return ASM_OK;
}
int asm_slp_get_csr(asm_slp *hh, int32_t s, int64_t *row_ptr, int32_t *col_idx, double *vals) {
    if (!hh) return fail(ASM_E_INVALID, "null handle");
    SlpHandle &h = hh->h;
    if (s < 0 || s >= h.Buser) return fail(ASM_E_INVALID, "scenario out of range");
    if (row_ptr) memcpy(row_ptr, h.pat.row_ptr.data(), sizeof(int64_t) * (h.m + 1));
    if (col_idx && h.pat.nnz) memcpy(col_idx, h.pat.col_idx.data(), sizeof(int32_t) * h.pat.nnz);
    if (vals && h.pat.nnz) {
        if (h.phase < 0) return fail(ASM_E_STATE, "no update yet");
        ASM_CK(cudaSetDevice(h.device));
        ASM_CK(cudaMemcpy2DAsync(vals, sizeof(double), h.normal->vals.p + s, sizeof(double) * h.B, sizeof(double),
                                 h.pat.nnz, cudaMemcpyDeviceToHost, h.stream));
        ASM_CK(cudaStreamSynchronize(h.stream));
    }
    return ASM_OK;
}
int asm_slp_get_lp(asm_slp *hh, int32_t s, int32_t *cols, int32_t *rows, int64_t *nnz, int64_t *row_ptr,
                   int32_t *col_idx, double *vals, double *c, double *c0, double *lb, double *ub, double *rl,
                   double *ru, double *x, double *y, double *dual_lb, double *dual_ub, int32_t *status) {
    if (!hh) return fail(ASM_E_INVALID, "null handle");
    SlpHandle &h = hh->h;
    if (s < 0 || s >= h.Buser) return fail(ASM_E_INVALID, "scenario out of range");
    if (h.phase < 0) return fail(ASM_E_STATE, "no update yet");
    if ((x || y || dual_lb || dual_ub || status) && !h.solved) return fail(ASM_E_STATE, "no solve since the last update");
    LpSolver &lp = *h.cur();
    if (cols) *cols = lp.n;
    if (rows) *rows = lp.m;
    if (nnz) *nnz = lp.nnz;
    if (row_ptr)
        for (int i = 0; i <= lp.m; ++i) row_ptr[i] = lp.h_row_ptr[i];
    if (col_idx) std::copy(lp.h_col_idx.begin(), lp.h_col_idx.begin() + lp.nnz, col_idx);
    ASM_CK(cudaSetDevice(h.device));
    // one lane of an element-major [len][B] array
    auto lane = [&](double *dst, const DBuf<double> &src, int64_t len) -> int {
        if (dst && len)
            ASM_CK(cudaMemcpy2DAsync(dst, sizeof(double), src.p + s, sizeof(double) * h.B, sizeof(double), len,
                                     cudaMemcpyDeviceToHost, h.stream));
        return ASM_OK;
    };
    ASM_TRY(lane(vals, lp.vals, lp.nnz));
    ASM_TRY(lane(c, lp.c, lp.n));
    ASM_TRY(lane(c0, lp.c0, 1));
    ASM_TRY(lane(lb, lp.lb, lp.n));
    ASM_TRY(lane(ub, lp.ub, lp.n));
    ASM_TRY(lane(rl, lp.rl, lp.m));
    ASM_TRY(lane(ru, lp.ru, lp.m));
    ASM_TRY(lane(x, lp.xo, lp.n));
    ASM_TRY(lane(y, lp.yo, lp.m));
    ASM_TRY(lane(dual_lb, lp.dlo, lp.n));
    ASM_TRY(lane(dual_ub, lp.dup, lp.n));
    ScenState st;
    if (status) ASM_CK(cudaMemcpyAsync(&st, lp.state.p + s, sizeof st, cudaMemcpyDeviceToHost, h.stream));
    ASM_CK(cudaStreamSynchronize(h.stream));
    if (status) *status = st.status;
    return ASM_OK;
}
int asm_slp_update(asm_slp *h, const double *x_k, const double *f, const double *df, const double *E,
                   const double *dE, const double *delta, int32_t feasibility) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    return h->h.update(x_k, f, df, E, dE, delta, feasibility);
}
int asm_slp_solve(asm_slp *h, const asm_lp_params *params, asm_lp_info *info) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    return h->h.solve(params, info);
}
int asm_slp_set_active(asm_slp *h, const int32_t *active) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    ASM_CK(cudaSetDevice(h->h.device));
    ASM_TRY(h->h.normal->set_active(active));
    if (h->h.fr) ASM_TRY(h->h.fr->set_active(active));
    if (active)
        h->h.mask.assign(active, active + h->h.Buser);
    else
        h->h.mask.clear();
    return ASM_OK;
}
int asm_slp_extract(asm_slp *h, double *p, double *lambda, double *mult_x_U, double *mult_x_L, double *p_slack,
                    int32_t *status) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    return h->h.extract(p, lambda, mult_x_U, mult_x_L, p_slack, status);
}
int asm_slp_sub_optimize(asm_slp *h, const double *x_k, const double *f, const double *df, const double *E,
                         const double *dE, const double *delta, int32_t feasibility, const asm_lp_params *params,
                         double *p, double *lambda, double *mult_x_U, double *mult_x_L, double *p_slack,
                         int32_t *status, asm_lp_info *info) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    ASM_TRY(h->h.update(x_k, f, df, E, dE, delta, feasibility));
    ASM_TRY(h->h.solve(params, info));
    return h->h.extract(p, lambda, mult_x_U, mult_x_L, p_slack, status);
}

// ---- merit / KKT reductions -----------------------------------------------------------------------------------
#define SLP_GUARD()                                          \
    if (!hh) return fail(ASM_E_INVALID, "null handle");      \
    SlpHandle &h = hh->h;                                    \
    const int B = h.B;                                       \
    cudaStream_t stream = h.stream;                          \
    int64_t &own_launches = h.own_launches;                  \
    (void)own_launches;                                      \
    ASM_CK(cudaSetDevice(h.device))

int asm_slp_norm_violations(asm_slp *hh, const double *E, const double *x, int32_t p_norm, double *out) {
    SLP_GUARD();
    if (!out || p_norm < 0 || p_norm > 2) return fail(ASM_E_INVALID, "bad argument");
    const double *dEv = h.E.p, *dx = h.xk.p;
    if (E) {
        ASM_TRY(h.put(E, h.m, h.Buser, h.tmp_m.p));
        dEv = h.tmp_m.p;
    }
    if (x) {
        ASM_TRY(h.put(x, h.n, h.Buser, h.tmp_n.p));
        dx = h.tmp_n.p;
    }
    SlpView sv = h.view();
    const Geo g = geo_for(std::max(h.n, h.m), B);
    SLP_KB(k_viol, g, sv, dEv, dx, (int)p_norm, h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(g.grid.x, p_norm == 0 ? 1u : 0u, r));
    for (int s = 0; s < h.Buser; ++s) out[s] = p_norm == 2 ? sqrt(r[s * R_COUNT + R_A]) : r[s * R_COUNT + R_A];
    return ASM_OK;
}

int asm_slp_row_norms(asm_slp *hh, double *out) {
    SLP_GUARD();
    if (h.phase < 0) return fail(ASM_E_STATE, "no update yet");
    const Geo g = geo_for(h.m, B);
    SLP_KB(k_row_norms, g, h.normal->row_ptr.p, h.normal->vals.p, (const double *)nullptr, h.tmp_m.p, h.m, B,
           h.partials.p);
    ASM_CK(cudaGetLastError());
    ASM_TRY(h.get(h.tmp_m.p, h.m, out));
    ASM_CK(cudaStreamSynchronize(stream));
    return ASM_OK;
}

int asm_slp_kt_residuals(asm_slp *hh, const double *df, const double *lambda, const double *mult_x_U,
                         const double *mult_x_L, double *out) {
    SLP_GUARD();
    if (!out || !lambda || !mult_x_U || !mult_x_L) return fail(ASM_E_INVALID, "null argument");
    if (h.phase < 0) return fail(ASM_E_STATE, "no update yet");
    const double *ddf = h.df.p;
    if (df) {
        ASM_TRY(h.put(df, h.n, h.Buser, h.tmp_n.p));
        ddf = h.tmp_n.p;
    }
    ASM_TRY(h.put(lambda, h.m, h.Buser, h.tmp_m.p));
    ASM_TRY(h.put(mult_x_U, h.n, h.Buser, h.tmp_n2.p));
    ASM_TRY(h.put(mult_x_L, h.n, h.Buser, h.tmp_n3.p));
    LpSolver *lp = h.normal.get();
    const Geo gr = geo_for(h.m, B), gc = geo_for(h.n, B);
    // zero the slots a smaller grid leaves untouched
    ASM_TRY(h.partials.zero(stream));
    SLP_KB(k_row_norms, gr, lp->row_ptr.p, lp->vals.p, (const double *)h.tmp_m.p, (double *)nullptr, h.m, B,
           h.partials.p);
    SLP_KB(k_kt, gc, lp->col_ptr.p, lp->row_idx.p, lp->csc_src.p, lp->vals.p, ddf, h.tmp_m.p, h.tmp_n2.p, h.tmp_n3.p,
           h.n, B, h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(std::max(gr.grid.x, gc.grid.x), 1u << R_B, r));
    for (int s = 0; s < h.Buser; ++s) {
        const double kt = sqrt(r[s * R_COUNT + R_C]);
        double scalar = std::max(1.0, sqrt(r[s * R_COUNT + R_D]));
        if (h.m > 0) scalar = std::max(scalar, r[s * R_COUNT + R_B]);
        out[s] = kt / scalar;
    }
    return ASM_OK;
}

int asm_slp_norm_complementarity(asm_slp *hh, const double *E, const double *lambda, double *out) {
    SLP_GUARD();
    if (!out || !lambda) return fail(ASM_E_INVALID, "null argument");
    const double *dEv = h.E.p;
    if (E) {
        ASM_TRY(h.put(E, h.m, h.Buser, h.tmp_m.p));
        dEv = h.tmp_m.p;
    }
    ASM_TRY(h.put(lambda, h.m, h.Buser, h.tmp_m2.p));
    SlpView sv = h.view();
    const Geo g = geo_for(h.m, B);
    SLP_KB(k_compl, g, sv, dEv, h.tmp_m2.p, h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(g.grid.x, 1u << R_A, r));
    for (int s = 0; s < h.Buser; ++s) out[s] = r[s * R_COUNT + R_A] / (1.0 + sqrt(r[s * R_COUNT + R_B]));
    return ASM_OK;
}

int asm_slp_merit_phi(asm_slp *hh, const double *base, const double *E_trial, const double *nu, const double *alpha,
                      int32_t feasibility, double *out) {
    SLP_GUARD();
    if (!out || !base || !nu) return fail(ASM_E_INVALID, "null argument");
    if (h.phase < 0) return fail(ASM_E_STATE, "no update yet");
    const double *dEt = h.E.p;
    if (E_trial) {
        ASM_TRY(h.put(E_trial, h.m, h.Buser, h.tmp_m.p));
        dEt = h.tmp_m.p;
    }
    ASM_TRY(h.put(nu, h.m, h.Buser, h.tmp_m2.p));
    double *ps = (double *)h.pin_small.p + (size_t)B * R_COUNT;
    for (int s = 0; s < B; ++s) ps[s] = alpha ? alpha[s < h.Buser ? s : 0] : 0.0;
    ASM_CK(cudaMemcpyAsync(h.d_alpha.p, ps, sizeof(double) * B, cudaMemcpyHostToDevice, stream));
    SlpView sv = h.view();
    const Geo g = geo_for(h.m, B);
    SLP_KB(k_merit, g, sv, dEt, h.tmp_m2.p, h.pslack.p, (const double *)h.d_alpha.p, (int)feasibility, h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(g.grid.x, 0u, r));
    for (int s = 0; s < h.Buser; ++s) {
        const double al = alpha ? alpha[s] : 0.0;
        out[s] = base[s] + (feasibility ? al * r[s * R_COUNT + R_B] : 0.0) + r[s * R_COUNT + R_A];
    }
    return ASM_OK;
}

int asm_slp_merit_derivative(asm_slp *hh, const double *nu, int32_t feasibility, double *out) {
    SLP_GUARD();
    if (!out || !nu) return fail(ASM_E_INVALID, "null argument");
    if (h.phase < 0 || !h.solved) return fail(ASM_E_STATE, "no solved sub-LP yet");
    ASM_TRY(h.extract_device());
    ASM_TRY(h.put(nu, h.m, h.Buser, h.tmp_m2.p));
    SlpView sv = h.view();
    const Geo g = geo_for(h.m, B), gc = geo_for(h.n, B);
    ASM_TRY(h.partials.zero(stream));
    SLP_KB(k_merit, g, sv, (const double *)h.E.p, h.tmp_m2.p, h.pslack.p, (const double *)nullptr, (int)feasibility,
           h.partials.p);
    if (!feasibility) SLP_KB(k_dot, gc, h.df.p, h.p.p, (int64_t)h.n, B, h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(std::max(g.grid.x, gc.grid.x), 0u, r));
    for (int s = 0; s < h.Buser; ++s)
        out[s] = (feasibility ? r[s * R_COUNT + R_B] : r[s * R_COUNT + R_C]) - r[s * R_COUNT + R_A];
    return ASM_OK;
}

// ---- device-side ACOPF evaluator ------------------------------------------------------------------------------
int asm_slp_attach_acopf(asm_slp *hh, const asm_acopf_desc *d) {
    SLP_GUARD();
    (void)B;
    if (!d || d->nb <= 0 || d->ng < 0 || d->nl < 0 || d->nd < 0) return fail(ASM_E_INVALID, "bad ACOPF description");
    if (!d->f_bus || !d->t_bus || !d->coef || !d->gs || !d->bs || !d->cost2 || !d->cost1 || !d->cost0 || !d->bal_ptr ||
        (d->nd > 0 && !d->dc_loss1))
        return fail(ASM_E_INVALID, "null array in the ACOPF description");
    if (d->bal_ptr[0] != 0) return fail(ASM_E_INVALID, "bal_ptr must start at 0");
    for (int i = 0; i < 2 * d->nb; ++i)
        if (d->bal_ptr[i + 1] < d->bal_ptr[i]) return fail(ASM_E_INVALID, "bal_ptr is not monotone");
    if (d->bal_ptr[2 * d->nb] > 0 && (!d->bal_col || !d->bal_coef))
        return fail(ASM_E_INVALID, "null balance-row lists in the ACOPF description");
    AcopfDev a;
    a.nb = d->nb; a.ng = d->ng; a.nl = d->nl; a.nd = d->nd; a.ref_bus = d->ref_bus;
    a.nnz_bal = d->bal_ptr[2 * d->nb];
    int o = 0;
    a.o_va = o; o += a.nb;
    a.o_vm = o; o += a.nb;
    a.o_pg = o; o += a.ng;
    a.o_qg = o; o += a.ng;
    a.o_p = o; o += 2 * a.nl;
    a.o_q = o; o += 2 * a.nl;
    a.o_pdc = o; o += 2 * a.nd;
    a.o_qdc = o; o += 2 * a.nd;
    const int n = o;
    int r = 0;
    a.r_angmax = r; r += a.nl;
    a.r_angmin = r; r += a.nl;
    a.r_ref = r; r += 1;
    a.r_dc = r; r += a.nd;
    a.r_thermal = r; r += 2 * a.nl;
    a.r_bal = r; r += 2 * a.nb;
    a.r_ohm = r; r += 4 * a.nl;
    const int m = r;
    int k = 0;
    a.k_angmax = k; k += 2 * a.nl;
    a.k_angmin = k; k += 2 * a.nl;
    a.k_ref = k; k += 1;
    a.k_dc = k; k += 2 * a.nd;
    a.k_thermal = k; k += 4 * a.nl;
    a.k_bal = k; k += a.nnz_bal;
    a.k_ohm = k; k += 20 * a.nl;
    if (n != h.n || m != h.m || (int64_t)k != h.pat.nnz_coo)
        return fail(ASM_E_INVALID, "ACOPF description does not match the handle's n, m, nnz (layout of examples/acopf.py)");
    if (a.ref_bus < 0 || a.ref_bus >= a.nb) return fail(ASM_E_INVALID, "reference bus out of range");
    for (int l = 0; l < a.nl; ++l)
        if (d->f_bus[l] < 0 || d->f_bus[l] >= a.nb || d->t_bus[l] < 0 || d->t_bus[l] >= a.nb)
            return fail(ASM_E_INVALID, "branch terminal out of range");
    for (int t = 0; t < a.nnz_bal; ++t)
        if (d->bal_col[t] < 0 || d->bal_col[t] >= n) return fail(ASM_E_INVALID, "balance column out of range");
    auto upi = [&](DBuf<int> &b, const int32_t *src, size_t cnt) -> int {
        ASM_TRY(b.alloc(std::max<size_t>(cnt, 1)));
        if (cnt) ASM_CK(cudaMemcpy(b.p, src, cnt * sizeof(int), cudaMemcpyHostToDevice));
        return ASM_OK;
    };
    auto upd = [&](DBuf<double> &b, const double *src, size_t cnt) -> int {
        ASM_TRY(b.alloc(std::max<size_t>(cnt, 1)));
        if (cnt) ASM_CK(cudaMemcpy(b.p, src, cnt * sizeof(double), cudaMemcpyHostToDevice));
        return ASM_OK;
    };
    ASM_TRY(upi(h.ac_f, d->f_bus, a.nl));
    ASM_TRY(upi(h.ac_t, d->t_bus, a.nl));
    ASM_TRY(upi(h.ac_bal_ptr, d->bal_ptr, 2 * (size_t)a.nb + 1));
    ASM_TRY(upi(h.ac_bal_col, d->bal_col, a.nnz_bal));
    ASM_TRY(upd(h.ac_coef, d->coef, 12 * (size_t)a.nl));
    ASM_TRY(upd(h.ac_gs, d->gs, a.nb));
    ASM_TRY(upd(h.ac_bs, d->bs, a.nb));
    ASM_TRY(upd(h.ac_c2, d->cost2, a.ng));
    ASM_TRY(upd(h.ac_c1, d->cost1, a.ng));
    ASM_TRY(upd(h.ac_c0, d->cost0, a.ng));
    ASM_TRY(upd(h.ac_loss1, d->dc_loss1, a.nd));
    ASM_TRY(upd(h.ac_bal_coef, d->bal_coef, a.nnz_bal));
    ASM_TRY(h.ac_ftrial.alloc(h.B));
    a.f_bus = h.ac_f.p; a.t_bus = h.ac_t.p; a.bal_ptr = h.ac_bal_ptr.p; a.bal_col = h.ac_bal_col.p;
    a.coef = h.ac_coef.p; a.gs = h.ac_gs.p; a.bs = h.ac_bs.p; a.cost2 = h.ac_c2.p; a.cost1 = h.ac_c1.p;
    a.cost0 = h.ac_c0.p; a.dc_loss1 = h.ac_loss1.p; a.bal_coef = h.ac_bal_coef.p;
    h.acopf = a;
    h.has_acopf = true;
    return ASM_OK;
}

// eval_functions! on the device followed by the data push of sub_optimize!: x[batch][n], delta[batch]
int asm_slp_eval_acopf(asm_slp *hh, const double *x, const double *delta, int32_t feasibility) {
    SLP_GUARD();
    if (!h.has_acopf) return fail(ASM_E_STATE, "asm_slp_attach_acopf first");
    if (!x || !delta) return fail(ASM_E_INVALID, "null argument");
    ASM_TRY(h.put(x, h.n, h.Buser, h.xk.p));
    double *ps = (double *)h.pin_small.p;
    for (int s = 0; s < B; ++s) ps[s] = delta[s < h.Buser ? s : 0];
    ASM_CK(cudaMemcpyAsync(h.delta.p, ps, B * sizeof(double), cudaMemcpyHostToDevice, stream));
    ASM_TRY(h.df.zero(stream));
    AcopfIo io;
    io.xk = h.xk.p; io.p = nullptr; io.alpha = nullptr;
    io.f = h.fval.p; io.df = h.df.p; io.E = h.E.p; io.dE = h.dE.p; io.B = B;
    const Geo gl = geo_for(std::max(h.acopf.nl, 1), B), gb = geo_for(2 * h.acopf.nb, B);
    if (B > 1) {
        k_acopf_branch<true, false><<<gl.grid, gl.block, 0, stream>>>(h.acopf, io);
        k_acopf_bus<true, false><<<gb.grid, gb.block, 0, stream>>>(h.acopf, io);
    } else {
        k_acopf_branch<false, false><<<gl.grid, gl.block, 0, stream>>>(h.acopf, io);
        k_acopf_bus<false, false><<<gb.grid, gb.block, 0, stream>>>(h.acopf, io);
    }
    k_acopf_misc<false><<<(B + 127) / 128, 128, 0, stream>>>(h.acopf, io, h.n);
    own_launches += 3;
    ASM_CK(cudaGetLastError());
    return h.update_device(feasibility);
}

// the evaluation of the last asm_slp_eval_acopf / asm_slp_update, back on the host (tests, drivers): any may be NULL
int asm_slp_get_eval(asm_slp *hh, double *f, double *df, double *E, double *dE) {
    SLP_GUARD();
    (void)B;
    if (h.phase < 0) return fail(ASM_E_STATE, "no evaluation yet");
    if (f) ASM_CK(cudaMemcpyAsync(f, h.fval.p, h.Buser * sizeof(double), cudaMemcpyDeviceToHost, stream));
    ASM_TRY(h.get(h.df.p, h.n, df));
    ASM_TRY(h.get(h.E.p, h.m, E));
    ASM_TRY(h.get(h.dE.p, h.pat.nnz_coo, dE));
    ASM_CK(cudaStreamSynchronize(stream));
    return ASM_OK;
}

// compute_phi(x + alpha p) (slp.jl:79-115) with g and f evaluated on the device at the trial point: x_k of the last
// evaluation, p of the last solve.  base[batch] is only read in feasibility restoration (prim_infeas); otherwise the
// base is f(x + alpha p).  out[batch].
int asm_slp_acopf_trial(asm_slp *hh, const double *alpha, const double *nu, const double *base, int32_t feasibility,
                        double *out) {
    SLP_GUARD();
    if (!h.has_acopf) return fail(ASM_E_STATE, "asm_slp_attach_acopf first");
    if (!alpha || !nu || !out || (feasibility && !base)) return fail(ASM_E_INVALID, "null argument");
    if (h.phase < 0 || !h.solved) return fail(ASM_E_STATE, "no solved sub-LP yet");
    ASM_TRY(h.extract_device());
    ASM_TRY(h.put(nu, h.m, h.Buser, h.tmp_m2.p));
    double *ps = (double *)h.pin_small.p + (size_t)B * R_COUNT;
    for (int s = 0; s < B; ++s) ps[s] = alpha[s < h.Buser ? s : 0];
    ASM_CK(cudaMemcpyAsync(h.d_alpha.p, ps, sizeof(double) * B, cudaMemcpyHostToDevice, stream));
    AcopfIo io;
    io.xk = h.xk.p; io.p = h.p.p; io.alpha = h.d_alpha.p;
    io.f = h.ac_ftrial.p; io.df = nullptr; io.E = h.tmp_m.p; io.dE = nullptr; io.B = B;
    const Geo gl = geo_for(std::max(h.acopf.nl, 1), B), gb = geo_for(2 * h.acopf.nb, B);
    if (B > 1) {
        k_acopf_branch<true, true><<<gl.grid, gl.block, 0, stream>>>(h.acopf, io);
        k_acopf_bus<true, true><<<gb.grid, gb.block, 0, stream>>>(h.acopf, io);
    } else {
        k_acopf_branch<false, true><<<gl.grid, gl.block, 0, stream>>>(h.acopf, io);
        k_acopf_bus<false, true><<<gb.grid, gb.block, 0, stream>>>(h.acopf, io);
    }
    k_acopf_misc<true><<<(B + 127) / 128, 128, 0, stream>>>(h.acopf, io, h.n);
    own_launches += 3;
    SlpView sv = h.view();
    const Geo g = geo_for(h.m, B);
    SLP_KB(k_merit, g, sv, (const double *)h.tmp_m.p, h.tmp_m2.p, h.pslack.p, (const double *)h.d_alpha.p, (int)feasibility,
           h.partials.p);
    std::vector<double> r;
    ASM_TRY(h.finish_reduce(g.grid.x, 0u, r));
    std::vector<double> ft(B, 0.0);
    ASM_CK(cudaMemcpyAsync(ft.data(), h.ac_ftrial.p, sizeof(double) * B, cudaMemcpyDeviceToHost, stream));
    ASM_CK(cudaStreamSynchronize(stream));
    for (int s = 0; s < h.Buser; ++s) {
        const double b0 = feasibility ? base[s] + alpha[s] * r[s * R_COUNT + R_B] : ft[s];
        out[s] = b0 + r[s * R_COUNT + R_A];
    }
    return ASM_OK;
}

int64_t asm_slp_launch_count(asm_slp *h) {
    if (!h) return 0;
    int64_t t = h->h.own_launches;
    if (h->h.normal) t += h->h.normal->launches;
    if (h->h.fr) t += h->h.fr->launches;
    return t;
}
int asm_slp_last_solve_timing(asm_slp *h, double *loop_ms, int64_t *iterations) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    if (!h->h.solved) return fail(ASM_E_STATE, "no solve yet");
    if (loop_ms) *loop_ms = h->h.cur()->last_loop_ms;
    if (iterations) *iterations = h->h.cur()->last_iters;
    return ASM_OK;
}

// Host-only self-check of the group engine's layout (no device needed): builds the sliced-ELL / halo layout of a
// CSR pattern for groups of G blocks, rebuilds every row from it and compares with the input.
int asm_plan_check(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx, int32_t G,
                   int64_t *smem_bytes, int32_t *matrix_resident, int64_t *padded_entries) {
    if (!row_ptr || n_cols <= 0 || n_rows < 0 || G < 1) return fail(ASM_E_INVALID, "bad argument");
    const int64_t nnz = row_ptr[n_rows];
    if (nnz > 0 && !col_idx) return fail(ASM_E_INVALID, "null col_idx");
    std::vector<int> rp(n_rows + 1), ci(nnz);
    for (int i = 0; i <= n_rows; ++i) rp[i] = (int)row_ptr[i];
    for (int64_t k = 0; k < nnz; ++k) {
        if (col_idx[k] < 0 || col_idx[k] >= n_cols) return fail(ASM_E_INVALID, "column index out of range");
        ci[k] = col_idx[k];
    }
    SellSide R;
    build_sell_side(n_rows, n_cols, rp.data(), ci.data(), nullptr, G, R);
    if ((int)R.first.size() != G) return fail(ASM_E_STATE, "wrong number of blocks");
    std::vector<char> seen(nnz, 0);
    int64_t rows_seen = 0, padded = 0;
    int next_first = 0;
    for (int c = 0; c < G; ++c) {
        if (R.first[c] != next_first) return fail(ASM_E_STATE, "row ranges are not contiguous");
        next_first += R.cnt[c];
        const int *ptr = R.ptr.data() + R.ptr_base[c];
        const int *halo = R.halo.data() + R.halo_base[c];
        for (int t = 1; t < R.halo_cnt[c]; ++t)
            if (halo[t - 1] >= halo[t]) return fail(ASM_E_STATE, "halo list is not strictly increasing");
        for (int q = 0; q < R.nslice[c]; ++q) {
            const int len = ptr[q + 1] - ptr[q];
            for (int lane = 0; lane < 32; ++lane) {
                const int sl = R.slot_base[c] + q * 32 + lane;
                const int row = R.slot[sl], tail = R.tail[sl];
                if (lane + tail > 31) return fail(ASM_E_STATE, "row group crosses a slice");
                if (row >= 0) {
                    if (row < R.first[c] || row >= R.first[c] + R.cnt[c]) return fail(ASM_E_STATE, "row outside its block");
                    ++rows_seen;
                    // entries of the head lane and of its `tail` followers, in lane order, must be the CSR row
                    int64_t k = rp[row];
                    for (int g = 0; g <= tail; ++g)
                        for (int e = 0; e < len; ++e) {
                            const size_t at = (size_t)R.base[c] + ((size_t)ptr[q] + e) * 32 + lane + g;
                            const int src = R.src[at];
                            if (src < 0) continue;
                            if (src != k || seen[src]) return fail(ASM_E_STATE, "sliced-ELL entry out of order");
                            if (R.idx[at] < 0 || R.idx[at] >= R.halo_cnt[c] || halo[R.idx[at]] != ci[src])
                                return fail(ASM_E_STATE, "halo position does not map back to the column");
                            seen[src] = 1;
                            ++k;
                        }
                    if (k != rp[row + 1]) return fail(ASM_E_STATE, "row incomplete in the sliced-ELL layout");
                }
            }
            padded += (int64_t)len * 32;
        }
    }
    if (next_first != n_rows || rows_seen != n_rows) return fail(ASM_E_STATE, "rows lost by the partition");
    for (int64_t k = 0; k < nnz; ++k)
        if (!seen[k]) return fail(ASM_E_STATE, "matrix entry missing from the layout");
    // shared-memory need of the full (two-sided) plan
    std::vector<int> cp(n_cols + 1, 0), ri(nnz);
    for (int64_t k = 0; k < nnz; ++k) cp[ci[k] + 1]++;
    for (int j = 0; j < n_cols; ++j) cp[j + 1] += cp[j];
    {
        std::vector<int> cur(cp.begin(), cp.end() - 1);
        for (int i = 0; i < n_rows; ++i)
            for (int k = rp[i]; k < rp[i + 1]; ++k) ri[cur[ci[k]]++] = i;
    }
    LpSolver tmp;
    tmp.n = n_cols;
    tmp.m = n_rows;
    tmp.nnz = nnz;
    tmp.h_row_ptr = rp;
    tmp.h_col_idx = ci;
    tmp.h_col_ptr = cp;
    tmp.h_row_idx = ri;
    SellSide R2, C2;
    GroupSmem sm;
    const size_t bytes = LpSolver::plan_layout(tmp, G, R2, C2, sm);
    if (smem_bytes) *smem_bytes = (int64_t)bytes;
    if (matrix_resident) *matrix_resident = sm.mats;
    if (padded_entries) *padded_entries = padded;
    return ASM_OK;
}

int asm_slp_engine_info(asm_slp *h, int32_t *engine, int32_t *group_size, int32_t *groups) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    if (!h->h.solved) return fail(ASM_E_STATE, "no solve yet");
    LpSolver *lp = h->h.cur();
    if (engine) *engine = lp->last_engine;
    if (group_size) *group_size = lp->last_G;
    if (groups) *groups = lp->last_groups;
    return ASM_OK;
}
int asm_slp_reassemble(asm_slp *h, int32_t feasibility) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    if (h->h.phase < 0) return fail(ASM_E_STATE, "asm_slp_reassemble before asm_slp_update");
    ASM_CK(cudaSetDevice(h->h.device));
    return h->h.update_device(feasibility);
}
int asm_slp_extract_device(asm_slp *h) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    ASM_CK(cudaSetDevice(h->h.device));
    return h->h.extract_device();
}
int asm_slp_timer_start(asm_slp *h) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    ASM_CK(cudaSetDevice(h->h.device));
    if (!h->h.tev0) {
        ASM_CK(cudaEventCreate(&h->h.tev0));
        ASM_CK(cudaEventCreate(&h->h.tev1));
    }
    ASM_CK(cudaEventRecord(h->h.tev0, h->h.stream));
    return ASM_OK;
}
int asm_slp_timer_stop(asm_slp *h, double *ms) {
    if (!h || !ms) return fail(ASM_E_INVALID, "null argument");
    if (!h->h.tev0) return fail(ASM_E_STATE, "timer not started");
    ASM_CK(cudaSetDevice(h->h.device));
    ASM_CK(cudaEventRecord(h->h.tev1, h->h.stream));
    ASM_CK(cudaEventSynchronize(h->h.tev1));
    float t = 0.f;
    ASM_CK(cudaEventElapsedTime(&t, h->h.tev0, h->h.tev1));
    *ms = t;
    return ASM_OK;
}
int asm_slp_kernel_timing(asm_slp *h, int32_t reps, double *primal_ms, double *dual_ms) {
    if (!h || reps < 1) return fail(ASM_E_INVALID, "bad argument");
    if (!h->h.solved) return fail(ASM_E_STATE, "no solve yet");
    ASM_CK(cudaSetDevice(h->h.device));
    return h->h.cur()->time_streaming_kernels(reps, primal_ms, dual_ms);
}

// sizes of the barrier engine's factorisation (stats[14]: KKT dimension, nnz(L), update terms, levels, factor chunks,
// forward chunks, launches per factorisation, launches per substitution pair, factorisations and substitution pairs of
// the last solve, distinct operand reads / targets per factorisation, per substitution pair, summed over the levels) and (times[4]) symbolic analysis ms,
// Newton steps of the last solve, factor / solve ms of the traced step (ASM_TRACE)
int asm_slp_ipm_info(asm_slp *h, int64_t *stats, double *times) {
    if (!h) return fail(ASM_E_INVALID, "null handle");
    LpSolver *lp = h->h.cur();
    if (!lp || !lp->ipm) return fail(ASM_E_STATE, "the barrier engine has not run on this handle");
    const IpmEngine &E = *lp->ipm;
    if (stats) {
        stats[0] = E.sym.N;
        stats[1] = E.sym.nnzL;
        stats[2] = E.sym.nterms;
        stats[3] = E.sym.n_levels;
        stats[4] = E.n_fchunks;
        stats[5] = E.sym.n_wchunks;
        stats[6] = E.launches_factor;
        stats[7] = E.launches_solve;
        stats[8] = E.last_factorisations;
        stats[9] = E.last_pairs;
        stats[10] = E.sym.f_distinct_reads;
        stats[11] = E.sym.f_targets;
        stats[12] = E.sym.w_distinct_reads + E.sym.b_distinct_reads;
        stats[13] = E.sym.w_targets + E.sym.b_targets;
    }
    if (times) {
        times[0] = E.symbolic_ms;
        times[1] = E.last_newton;
        times[2] = E.last_factor_ms;
        times[3] = E.last_solve_ms;
    }
    return ASM_OK;
}
int asm_slp_ipm_timing(asm_slp *h, int32_t reps, double *factor_ms, double *solve_ms) {
    if (!h || reps < 1) return fail(ASM_E_INVALID, "bad argument");
    if (!h->h.solved) return fail(ASM_E_STATE, "no solve yet");
    ASM_CK(cudaSetDevice(h->h.device));
    return h->h.cur()->time_ipm_kernels(reps, factor_ms, solve_ms);
}

// Host-only self test of the barrier engine's symbolic analysis (no device needed): orders and analyses the KKT
// pattern of the m x n CSR matrix K, then factorises  [-diag(dx) K'; K diag(ew)]  and solves one right-hand side ON
// THE HOST with exactly the lists and the summation order the device kernels use.  rhs_sol: n + m values, right-hand
// side in (columns then rows), solution out.  stats[8]: nnz(L), terms, levels, steps with fan-out items in the
// factorisation / forward / backward substitution (the step-kernel launches of each), longest chunk, chunks.
int asm_kkt_selftest(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx, const double *vals,
                     const double *dx, const double *ew, double *rhs_sol, int64_t *stats) {
    if (!row_ptr || n_cols <= 0 || n_rows < 0 || !dx || !rhs_sol) return fail(ASM_E_INVALID, "bad argument");
    const int64_t nnz = row_ptr[n_rows];
    if (nnz > 0 && (!col_idx || !vals)) return fail(ASM_E_INVALID, "null matrix");
    std::vector<int> rp(n_rows + 1), ci(nnz);
    for (int i = 0; i <= n_rows; ++i) rp[i] = (int)row_ptr[i];
    for (int64_t k = 0; k < nnz; ++k) ci[k] = col_idx[k];
    KktSymbolic S;
    // supernodes as a handle would use them (ASM_IPM_SUPERNODE=1 turns them off)
    if (S.build(n_cols, n_rows, rp.data(), ci.data(), kkt_supernode_width())) return fail(ASM_E_INVALID, "symbolic analysis failed");
    std::vector<double> W(S.nnzL, 0.0), d0(S.N), invd;
    for (int64_t q = 0; q < nnz; ++q) W[S.kmap[q]] = vals[q];
    for (int j = 0; j < n_cols; ++j) d0[S.inv[j]] = -dx[j];
    for (int i = 0; i < n_rows; ++i) d0[S.inv[n_cols + i]] = ew[i];
    S.factor_host(W, d0, invd);
    std::vector<double> v(rhs_sol, rhs_sol + S.N);
    S.solve_host(W, invd, v);
    std::copy(v.begin(), v.end(), rhs_sol);
    if (stats) {
        const int64_t longest = std::max(1, S.longest_chunk);
        stats[0] = S.nnzL;
        stats[1] = S.nterms;
        stats[2] = S.n_levels;
        auto fanout_steps = [&](const std::vector<int> &sb, const std::vector<int> &se, const std::vector<int> &ms) {
            int64_t c = 0;
            for (int l = 0; l < S.n_levels; ++l) c += se[l] > sb[l] || ms[l + 1] > ms[l];
            return c;
        };
        stats[3] = fanout_steps(S.fs_beg, S.fs_end, S.fmstep);
        stats[4] = fanout_steps(S.ws_beg, S.ws_end, S.wmstep);
        stats[5] = fanout_steps(S.bs_beg, S.bs_end, S.bmstep);
        stats[6] = longest;
        stats[7] = S.n_fchunks;
    }
    return ASM_OK;
}

// Device counterpart of asm_kkt_selftest: the same matrix, factorised and solved for a batch of scenarios by the
// barrier engine's own symbolic analysis (IpmEngine::init), launch sequences and captured graphs, as LpSolver::solve_ipm
// runs them.  Only the inputs differ: the pivots come straight from dx / ew (no regularisation) instead of k_ipm_diag.
int asm_kkt_device_selftest(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx,
                            int32_t batch, const double *vals, const double *dx, const double *ew,
                            const int32_t *active, double *rhs_sol, double *inv_pivots, int32_t device,
                            int64_t *stats) {
    if (!row_ptr || n_cols <= 0 || n_rows < 0 || batch < 1 || !dx || (n_rows > 0 && !ew) || !rhs_sol)
        return fail(ASM_E_INVALID, "bad argument");
    if (row_ptr[0] != 0) return fail(ASM_E_INVALID, "row_ptr[0] != 0");
    for (int i = 0; i < n_rows; ++i)
        if (row_ptr[i + 1] < row_ptr[i]) return fail(ASM_E_INVALID, "row_ptr is not non-decreasing");
    const int64_t nnz = row_ptr[n_rows];
    if (nnz > INT32_MAX) return fail(ASM_E_INVALID, "more than 2^31 - 1 entries");
    if (nnz > 0 && (!col_idx || !vals)) return fail(ASM_E_INVALID, "null matrix");
    for (int64_t q = 0; q < nnz; ++q)
        if (col_idx[q] < 0 || col_idx[q] >= n_cols) return fail(ASM_E_INVALID, "column index out of range");
    const int ndev = asm_device_count();
    if (ndev == 0) return fail(ASM_E_CUDA, "no CUDA device: this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(ASM_E_INVALID, "device index out of range");
    ASM_CK(cudaSetDevice(device));

    struct Stream {   // destroyed after the engine, which is declared below it
        cudaStream_t s = nullptr;
        ~Stream() {
            if (s) cudaStreamDestroy(s);
        }
    } stream;
    ASM_CK(cudaStreamCreateWithFlags(&stream.s, cudaStreamNonBlocking));
    const cudaStream_t st = stream.s;
    const int n = n_cols, m = n_rows, B = pad_batch(batch);
    std::vector<int> rp(m + 1), ci(nnz);
    for (int i = 0; i <= m; ++i) rp[i] = (int)row_ptr[i];
    for (int64_t q = 0; q < nnz; ++q) ci[q] = col_idx[q];
    IpmEngine E;
    ASM_TRY(E.init(n, m, rp, ci, B));
    const int N = E.sym.N;
    const std::vector<int> &inv = E.sym.inv;

    // element-major device layout v[i * B + s].  Padding lanes carry NaN: a kernel that mixes lanes spreads it
    const double nan = std::numeric_limits<double>::quiet_NaN();
    std::vector<double> hA((size_t)std::max<int64_t>(nnz, 1) * B, nan), hd((size_t)N * B, nan), hv((size_t)N * B, nan);
    std::vector<ScenState> hst(B);
    for (int s = 0; s < B; ++s) hst[s].status = s >= batch ? ASM_LP_OPTIMAL : (active && !active[s] ? ASM_LP_SKIPPED : -1);
    for (int s = 0; s < batch; ++s) {
        for (int64_t q = 0; q < nnz; ++q) hA[q * B + s] = vals[(int64_t)s * nnz + q];
        for (int j = 0; j < n; ++j) hd[(size_t)inv[j] * B + s] = -dx[(int64_t)s * n + j];
        for (int i = 0; i < m; ++i) hd[(size_t)inv[n + i] * B + s] = ew[(int64_t)s * m + i];
        for (int k = 0; k < N; ++k) hv[(size_t)k * B + s] = rhs_sol[(int64_t)s * N + k];
    }
    std::vector<double> hi(hd.size());
    for (size_t e = 0; e < hd.size(); ++e) hi[e] = 1.0 / hd[e];
    DBuf<double> A;
    DBuf<ScenState> state;
    ASM_TRY(A.alloc(hA.size()));
    ASM_TRY(state.alloc(B));
    double *vec = E.kktv[1].p;
    ASM_CK(cudaMemcpyAsync(A.p, hA.data(), hA.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    ASM_CK(cudaMemcpyAsync(state.p, hst.data(), hst.size() * sizeof(ScenState), cudaMemcpyHostToDevice, st));
    ASM_CK(cudaMemcpyAsync(E.diag0.p, hd.data(), hd.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    ASM_CK(cudaMemcpyAsync(E.invd.p, hi.data(), hi.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    ASM_CK(cudaMemcpyAsync(vec, hv.data(), hv.size() * sizeof(double), cudaMemcpyHostToDevice, st));

    LpView v = {};   // what k_kkt_scatter and the step kernels read
    v.n = n;
    v.m = m;
    v.B = B;
    v.A = A.p;
    v.state = state.p;
    ASM_TRY(E.capture(st, &E.g_factor, E.launches_factor, [&](int64_t &c) { E.enqueue_factor(v, st, c); }));
    ASM_TRY(E.capture(st, &E.g_solve_sol, E.launches_solve, [&](int64_t &c) { E.enqueue_solve(v, vec, st, c); }));
    ASM_CK(cudaGraphLaunch(E.g_factor, st));
    ASM_CK(cudaGraphLaunch(E.g_solve_sol, st));
    ASM_CK(cudaMemcpyAsync(hv.data(), vec, hv.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    ASM_CK(cudaMemcpyAsync(hi.data(), E.invd.p, hi.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    const int nfm = E.sym.fmstep[E.sym.n_levels];
    std::vector<KktRange> fm(nfm);
    if (nfm) ASM_CK(cudaMemcpyAsync(fm.data(), E.fmchunk.p, nfm * sizeof(KktRange), cudaMemcpyDeviceToHost, st));
    ASM_CK(cudaStreamSynchronize(st));
    ASM_CK(cudaGetLastError());
    for (int s = 0; s < batch; ++s)
        for (int k = 0; k < N; ++k) {
            rhs_sol[(int64_t)s * N + k] = hv[(size_t)k * B + s];
            if (inv_pivots) inv_pivots[(int64_t)s * N + k] = hi[(size_t)inv[k] * B + s];
        }
    if (stats) {
        const KktSymbolic &S = E.sym;
        int64_t narrow = 0, wide = 0, narrow_split = 0, wide_multi = 0, longest = 0, capped = 0;
        for (const KktPanel &P : S.panels) {
            if (P.w > kSnSmall) {
                ++wide;
                wide_multi += P.nr > kPanelRowsWide;
            } else {
                ++narrow;
            }
        }
        for (const KktPanelTask &t : S.ptasks) narrow_split += S.panels[t.panel].w <= kSnSmall && t.r0 > 0;
        for (int l = 0; l < S.n_levels; ++l) longest = std::max<int64_t>(longest, S.fs_end[l] > S.fs_beg[l]);
        for (const KktRange &r : fm) longest = std::max<int64_t>(longest, r.end - r.begin);
        // launches whose grid-stride loops take a second pass: the capped grid has fewer threads (batch: warps) than
        // single-term units (batch: four terms each) or multi-term chunks
        auto count_capped = [&](const std::vector<int> &sb, const std::vector<int> &se, const std::vector<int> &ms) {
            for (int l = 0; l < S.n_levels; ++l) {
                const int multi = ms[l + 1] - ms[l], singles = se[l] - sb[l];
                if (singles + multi == 0) continue;
                const int64_t threads = (int64_t)E.level_grid(singles + multi, multi).x * (B == 1 ? kThreads : kWarps);
                capped += std::max<int64_t>(B == 1 ? singles : (singles + 3) / 4, multi) > threads;
            }
        };
        count_capped(S.fs_beg, S.fs_end, S.fmstep);
        count_capped(S.ws_beg, S.ws_end, S.wmstep);
        count_capped(S.bs_beg, S.bs_end, S.bmstep);
        const int64_t out[10] = {S.nnzL, S.n_levels, narrow, wide, narrow_split, wide_multi, longest, capped,
                                 E.launches_factor, E.launches_solve};
        std::copy(out, out + 10, stats);
    }
    return ASM_OK;
}

}  // extern "C"
