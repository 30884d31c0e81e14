// Batched primal-dual barrier engine for   min c'x  s.t.  rl <= Kx <= ru,  lb <= x <= ub   on sm_100a.
//
// Stands where GLPK's simplex stands in the reference (MOI.optimize!(qp.model),
// /root/reference/src/algorithms/subproblem.jl:490), next to the PDHG engines of lp_solver.cuh: measured on the SLP
// sub-LPs of ACOPF (profiles/), first-order iterations cost 1e5 - 1e6 passes over the matrix per LP because the
// linearised power-flow equations are an ill-conditioned, almost square equality system; a barrier method needs
// 20 - 40 Newton steps, and every Newton step of every LP of a batch and of every SLP iteration factorises a matrix
// with the SAME sparsity pattern (the Jacobian pattern is uploaded once, src/model.jl:10).  So:
//   * symbolic work once per handle on the host (kkt_symbolic.hpp): ordering, pattern of L, supernodes, step schedule,
//     the fan-out lists of update products grouped by the step of their source column;
//   * numeric L D L' of the quasi-definite system  [-(Dx + d) K'; K (Ew + d)]  on the device: per step the dense panels
//     of its supernodes (k_sn_diag, k_sn_rows), then the updates that leave them (k_ldl_factor), every target written
//     by exactly one thread per step, scenarios across the lanes of a warp (element-major v[i * B + s]: index loads are
//     warp-uniform, value loads coalesced); no pivoting, no atomics, bit-reproducible;
//   * step-scheduled substitutions (k_sn_solve, k_ldl_fwd / k_ldl_diag / k_ldl_bwd), iterative refinement against the
//     unregularised matrix on demand (k_kkt_res_*); the step kernels are programmatic dependents of one another
//     and the three launch sequences are captured once as CUDA graphs;
//   * Mehrotra predictor-corrector with every scalar decision taken on the device per scenario (k_ipm_decide,
//     k_ipm_scalars); the host enqueues a fixed kernel sequence per Newton step and reads two 4-byte counters.
// A small proximal term (q/2)|x|^2 selects the least-norm optimal step among the minimisers (restoration LPs,
// min sum of slacks, always have a face of them); q is sized so that the dual residual and the duality gap it leaves
// in the LP stay below ipm_prox relative (for q below a threshold the minimiser is an exact LP solution anyway:
// Mangasarian & Meyer 1979).  Variables that end strictly complementary on a bound are returned exactly on it, as a
// simplex code does: the reference compares them with == (subproblem.jl:522-529).
// Algorithm: textbook (Mehrotra 1992; Vanderbei's quasi-definite systems) -- nothing here comes from the reference.
#pragma once
#include "kkt_symbolic.hpp"

namespace asmb {

enum {
    I_RDX2 = 0,  // |rdx|^2 unscaled (proximal system)
    I_RLP2,      // |c - K'y - z|^2 unscaled (the LP's own dual residual)
    I_POBJ,      // sum cs x
    I_QT,        // 1/2 sum Q x^2
    I_DOBJC,     // l'zl - u'zu (+ fixed columns)
    I_MUC,       // complementarity products of the columns
    I_XN2,       // |x|^2 unscaled
    I_RAYC,      // Farkas: box support of -(K'y)
    I_KTY,       // max |(K'y)_j / dc_j|
    I_RP2,       // |Kx - w|^2 unscaled
    I_RDW2,      // |y - zl + zu|^2 unscaled
    I_DOBJR,     // row part of the dual objective
    I_MUR,       // complementarity products of the rows
    I_RAYR,      // Farkas: rl'y+ + ru'y-
    I_YMAX,      // max |y_i dr_i|
    I_COUNT
};
// slots reused inside a Newton step (the residual slots are consumed by k_ipm_decide before)
enum { J_AP = 0, J_AD, J_MUC, J_MUR, J_AP_R, J_AD_R, J_RAY /* 4 slots */ };

struct IpmState {
    double mu, smu, ap, ad, qs, q_un;
    double ray_obj, ray_kty;  // Farkas test of the last step direction dy (normalised)
    double kept[5];           // pobj, dobj, pres, dres, gap of the point kept by k_ipm_save
    int ncomp, hits, acc_hits, save, bad;
};

// Programmatic dependent launch: a step's grid may be scheduled while the previous step still runs (the launch latency
// and its index loads leave the critical path); it must not touch W, 1/d, the pivots or the right-hand side before
// pdl_wait(), which returns when the previous grid has completed and its stores are visible.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// the ranges of the launched step come as arguments, not from the step tables: one dependent load less on the critical path
struct KktStepRange {
    int s0, s1, m0, m1;   // single-term items [s0, s1), multi-term chunks [m0, m1)
};

struct KktDev {
    const KktTerm *terms;
    const KktRange *fmchunk;
    const KktFwdItem *fwd;
    const KktRange *wmchunk;
    const KktBwdItem *bwd;
    const KktRange *bmchunk;
    const KktPanel *panels;
    const KktPanelTask *ptasks;
    const int *perm, *inv, *kmap;
    double *W, *invd, *diag0;
    double *PB;   // factorised diagonal blocks of the supernodes (KktPanel::off)
    int nnzL, N;
};

struct IpmView {
    // columns
    double *x, *zlx, *zux, *rdx, *Dx, *dzlx, *dzux, *clx, *cux;
    // rows
    double *w, *y, *zlw, *zuw, *rp, *rdw, *Ew, *dw, *dzlw, *dzuw, *clw, *cuw;
    // KKT vectors (node order: columns then rows)
    double *rhs0, *sol, *work;
    IpmState *ist;
    int *need_refine;     // counts LPs that sit at the acceptable level without reaching the target (see k_ipm_decide)
    const double *c0;     // objective constants (the termination test is relative to the objective the caller sees)
    double delta, prox;
    double eps, eps_acc;  // target tolerance; acceptable tolerance (kept as a fall-back result when the target is not reached)
    double mu_target;     // complementarity (scaled units) at which a converged LP stops
    int extra_hits, verbose;
};

__device__ __forceinline__ bool ipm_fin(double v) { return fabs(v) < 1.79e308; }
// distance to a bound; below the resolution of the difference it is floored (the complementarity products stay finite)
__device__ __forceinline__ double ipm_slack(double d) { return fmax(d, 1e-30); }

// =================================== numeric L D L' ============================================================
// Step l applies the updates of the columns of level l to their targets (fan-out).  A chunk = the terms of one target
// in this step.  Nine chunks in ten are a single term: they are stored first, and a warp keeps four of them in flight
// (the kernel is bound by the latency of its dependent loads -- index, then operands -- not by bandwidth: ncu shows
// 40 long-scoreboard stall cycles per issue without the pipelining).  BATCH: a warp owns a chunk and its lanes are 32
// scenarios (index loads warp-uniform, value loads coalesced); single LP: a thread owns a chunk.  Exactly one thread
// writes a target in a step and the terms of a chunk are added in ascending k: bit-reproducible.  One launch per step.
__device__ __forceinline__ void ldl_apply(const KktDev &d, int tflag, double acc, int B, int s) {
    const int t = tflag & ~kLastBit;
    if (t >= d.nnzL) {
        const int64_t e = (int64_t)(t - d.nnzL) * B + s;
        const double piv = d.diag0[e] - acc;
        d.diag0[e] = piv;
        if (tflag & kLastBit) d.invd[e] = 1.0 / piv;
    } else {
        d.W[(int64_t)t * B + s] -= acc;
    }
}
// sum of the terms [q0, q1) of one chunk in ascending order, four terms in flight (with supernodes a chunk holds up to
// kSnMax terms per source supernode: without the unrolling every term would cost a dependent index -> operand round trip)
__device__ __forceinline__ double chunk_sum(const KktDev &d, int q0, int q1, int B, int s, int &tflag, double &tv) {
    KktTerm u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) u[i] = d.terms[q0 + i < q1 ? q0 + i : q0];
    tflag = u[0].t;
    {   // the target travels with the first operands
        const int t = tflag & ~kLastBit;
        tv = t >= d.nnzL ? d.diag0[(int64_t)(t - d.nnzL) * B + s] : d.W[(int64_t)t * B + s];
    }
    double acc = 0.0;
    for (int q = q0; q < q1; q += 4) {
        double a[4], b[4], c[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            a[i] = d.W[(int64_t)u[i].a * B + s];
            b[i] = d.W[(int64_t)u[i].b * B + s];
            c[i] = d.invd[(int64_t)u[i].k * B + s];
        }
        const int qn = q + 4;
        if (qn < q1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = d.terms[qn + i < q1 ? qn + i : qn];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (q + i < q1) acc += a[i] * b[i] * c[i];
    }
    return acc;
}
template <class Item>
__device__ __forceinline__ double chunk_sum_vec(const KktDev &d, const Item *items, const double *v, int q0, int q1, int B, int s, int &dst, double &tv) {
    Item u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) u[i] = items[q0 + i < q1 ? q0 + i : q0];
    dst = u[0].dst;
    tv = v[(int64_t)dst * B + s];
    double acc = 0.0;
    for (int q = q0; q < q1; q += 4) {
        double a[4], x[4], c[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            a[i] = d.W[(int64_t)u[i].pos * B + s];
            x[i] = v[(int64_t)u[i].src * B + s];
            c[i] = d.invd[(int64_t)u[i].k * B + s];
        }
        const int qn = q + 4;
        if (qn < q1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = items[qn + i < q1 ? qn + i : qn];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (q + i < q1) acc += a[i] * x[i] * c[i];
    }
    return acc;
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads, 4) k_ldl_factor(KktDev d, int B, const ScenState *st, KktStepRange rg) {
    pdl_trigger();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = BATCH ? blockIdx.y * 32 + lane : 0;
    const bool live = st[s].status < 0;
    const int first = BATCH ? blockIdx.x * kWarps + warp : blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = BATCH ? gridDim.x * kWarps : gridDim.x * blockDim.x;
    // loads are never gated on the scenario's status (it would put one more dependent load on the critical path); stores are
    const int q0 = rg.s0, q1 = rg.s1;
    pdl_wait();
    if (BATCH) {
        for (int q = q0 + 4 * first; q < q1; q += 4 * stride) {
            KktTerm u[4];
            double a[4], b[4], c[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = d.terms[q + i < q1 ? q + i : q];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                a[i] = d.W[(int64_t)u[i].a * B + s];
                b[i] = d.W[(int64_t)u[i].b * B + s];
                c[i] = d.invd[(int64_t)u[i].k * B + s];
            }
            double tv[4];
            int64_t te[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int t = u[i].t & ~kLastBit;
                const bool piv = t >= d.nnzL;
                te[i] = (int64_t)(piv ? t - d.nnzL : t) * B + s;
                tv[i] = piv ? d.diag0[te[i]] : d.W[te[i]];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (q + i >= q1 || !live) break;
                const double r = tv[i] - a[i] * b[i] * c[i];
                if ((u[i].t & ~kLastBit) >= d.nnzL) {
                    d.diag0[te[i]] = r;
                    if (u[i].t & kLastBit) d.invd[te[i]] = 1.0 / r;
                } else {
                    d.W[te[i]] = r;
                }
            }
        }
    } else {
        for (int q = q0 + first; q < q1; q += stride) {
            const KktTerm u = d.terms[q];
            if (live) ldl_apply(d, u.t, d.W[u.a] * d.W[u.b] * d.invd[u.k], 1, 0);
        }
    }
    for (int c = rg.m0 + first; c < rg.m1; c += stride) {
        const KktRange r = d.fmchunk[c];
        int tflag;
        double tv;
        const double acc = chunk_sum(d, r.begin, r.end, B, s, tflag, tv);
        if (live) {
            const int t = tflag & ~kLastBit;
            const double r2 = tv - acc;
            if (t >= d.nnzL) {
                const int64_t e = (int64_t)(t - d.nnzL) * B + s;
                d.diag0[e] = r2;
                if (tflag & kLastBit) d.invd[e] = 1.0 / r2;
            } else {
                d.W[(int64_t)t * B + s] = r2;
            }
        }
    }
}

// forward substitution  v <- L^-1 v  (fan-out, laid out like the factorisation; v indexed by node id, in place)
template <bool BATCH>
__global__ void __launch_bounds__(kThreads, 4) k_ldl_fwd(KktDev d, double *v, int B, const ScenState *st, KktStepRange rg) {
    pdl_trigger();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = BATCH ? blockIdx.y * 32 + lane : 0;
    const bool live = st[s].status < 0;
    const int first = BATCH ? blockIdx.x * kWarps + warp : blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = BATCH ? gridDim.x * kWarps : gridDim.x * blockDim.x;
    // loads are never gated on the scenario's status (it would put one more dependent load on the critical path); stores are
    const int q0 = rg.s0, q1 = rg.s1;
    if (BATCH) {
        int q = q0 + 4 * first;
        KktFwdItem u[4];
        if (q < q1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = d.fwd[q + i < q1 ? q + i : q];
        }
        pdl_wait();
        while (q < q1) {
            double a[4], x[4], c[4], t[4];
            int dst[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                a[i] = d.W[(int64_t)u[i].pos * B + s];
                x[i] = v[(int64_t)u[i].src * B + s];
                c[i] = d.invd[(int64_t)u[i].k * B + s];
                t[i] = v[(int64_t)u[i].dst * B + s];
                dst[i] = u[i].dst;
            }
            const int qn = q + 4 * stride;
            if (qn < q1) {
#pragma unroll
                for (int i = 0; i < 4; ++i) u[i] = d.fwd[qn + i < q1 ? qn + i : qn];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (q + i < q1 && live) v[(int64_t)dst[i] * B + s] = t[i] - a[i] * x[i] * c[i];
            q = qn;
        }
    } else {
        pdl_wait();
        for (int q = q0 + first; q < q1; q += stride) {
            const KktFwdItem u = d.fwd[q];
            if (live) v[u.dst] -= d.W[u.pos] * v[u.src] * d.invd[u.k];
        }
    }
    for (int c = rg.m0 + first; c < rg.m1; c += stride) {
        const KktRange r = d.wmchunk[c];
        int dst;
        double tv;
        const double acc = chunk_sum_vec(d, d.fwd, v, r.begin, r.end, B, s, dst, tv);
        if (live) v[(int64_t)dst * B + s] = tv - acc;
    }
}
// v <- D^-1 v
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ldl_diag(KktDev d, double *v, int B, const ScenState *st) {
    Map<BATCH> mp;
    if (st[mp.s].status >= 0) return;
    for (int64_t k = mp.first; k < d.N; k += mp.stride) v[(int64_t)d.perm[k] * B + mp.s] *= d.invd[k * B + mp.s];
}
// backward substitution  v <- L'^-1 v : the rows of a column are its ancestors in the elimination tree; without
// supernodes they sit on distinct levels and every item of a step has its own target, with supernodes a column can have
// several rows in one step (a chunk).  Steps are launched downwards
template <bool BATCH>
__global__ void __launch_bounds__(kThreads, 4) k_ldl_bwd(KktDev d, double *v, int B, const ScenState *st, KktStepRange rg) {
    pdl_trigger();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int s = BATCH ? blockIdx.y * 32 + lane : 0;
    const bool live = st[s].status < 0;
    const int first = BATCH ? blockIdx.x * kWarps + warp : blockIdx.x * blockDim.x + threadIdx.x;
    const int stride = BATCH ? gridDim.x * kWarps : gridDim.x * blockDim.x;
    // loads are never gated on the scenario's status (it would put one more dependent load on the critical path); stores are
    const int q0 = rg.s0, q1 = rg.s1;
    if (BATCH) {
        int q = q0 + 4 * first;
        KktBwdItem u[4];
        if (q < q1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = d.bwd[q + i < q1 ? q + i : q];
        }
        pdl_wait();
        while (q < q1) {
            double a[4], x[4], c[4], t[4];
            int dst[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                a[i] = d.W[(int64_t)u[i].pos * B + s];
                x[i] = v[(int64_t)u[i].src * B + s];
                c[i] = d.invd[(int64_t)u[i].k * B + s];
                t[i] = v[(int64_t)u[i].dst * B + s];
                dst[i] = u[i].dst;
            }
            const int qn = q + 4 * stride;
            if (qn < q1) {
#pragma unroll
                for (int i = 0; i < 4; ++i) u[i] = d.bwd[qn + i < q1 ? qn + i : qn];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (q + i < q1 && live) v[(int64_t)dst[i] * B + s] = t[i] - c[i] * a[i] * x[i];
            q = qn;
        }
    } else {
        pdl_wait();
        for (int q = q0 + first; q < q1; q += stride) {
            const KktBwdItem u = d.bwd[q];
            if (live) v[u.dst] -= d.invd[u.k] * d.W[u.pos] * v[u.src];
        }
    }
    for (int c = rg.m0 + first; c < rg.m1; c += stride) {
        const KktRange r = d.bmchunk[c];
        int dst;
        double tv;
        const double acc = chunk_sum_vec(d, d.bwd, v, r.begin, r.end, B, s, dst, tv);
        if (live) v[(int64_t)dst * B + s] = tv - acc;
    }
}

// =================================== supernode panels ===========================================================
// A supernode = w <= kSnMax columns c_0 < ... < c_w-1 with nested patterns: a dense w x w diagonal block and nr dense
// rows below it ("panel").  At the start of its step every update from outside has been applied.  The diagonal block is
// factorised right-looking (W = L D convention, as everywhere); its strictly lower part goes, scaled to L = W / d, to
// a buffer of its own (PB, KktPanel::off) that the rows and the substitutions read.  Then every row below is solved:
//     w[t,k] final  ->  w[t,i] -= w[t,k] * L[i,k]  for i > k        (right-looking: the dependent chain is w long)
// rows are independent of each other and every entry of the panel is read and written once.  Lanes are scenarios, as
// in the step kernels (a single LP runs the same kernels on one lane: the panels are a small part of its work).
//   k_sn_diag : panels wider than kSnSmall -- a block per (panel, 32 scenarios), diagonal block in shared memory;
//               narrow panels (most: separators of two or three buses) -- a warp per task, block AND rows, in registers
//   k_sn_rows : the rows of the wide panels, a block per kPanelRowsWide rows, a warp per row
//   k_sn_solve: the supernode's part of a substitution, a warp per panel
// Block-cooperative fetches use cp.async: a loop of load -> shared store would serialise one L2 round trip per entry.
__device__ __forceinline__ int sn_tri(int j, int i) { return j * (j + 1) / 2 + i; }   // j >= i
constexpr int kSnTri = kSnMax * (kSnMax + 1) / 2;
constexpr int kPanelThreads = 256;
__device__ __forceinline__ void cp_async8(double *smem, const double *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
__global__ void __launch_bounds__(kPanelThreads, 2) k_sn_diag(KktDev d, int B, int p0, int nwide, int t0n, int nnarrow, const ScenState *st) {
    pdl_trigger();
    __shared__ double S[kSnTri][32];
    __shared__ double Iv[kSnMax][32];
    __shared__ int pc[kSnMax], pl[kSnMax];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int nw = kPanelThreads / 32;
    const int s = min((int)blockIdx.y * 32 + lane, B - 1);   // single LP (B == 1): lane 0 works, the others shadow it
    const bool live = (int)blockIdx.y * 32 + lane < B && st[s].status < 0;
    if ((int)blockIdx.x >= nwide) {   // ---- narrow panels: block and rows
        const int ti = ((int)blockIdx.x - nwide) * nw + warp;
        if (ti >= nnarrow) return;
        const KktPanelTask task = d.ptasks[t0n + ti];
        const KktPanel *P = d.panels + task.panel;
        const int w = P->w, nr = P->nr;
        int c[kSnSmall], lp[kSnSmall];
#pragma unroll
        for (int i = 0; i < kSnSmall; ++i) {
            c[i] = P->col[i];
            lp[i] = P->lp[i];
        }
        pdl_wait();
        double A[kSnSmall][kSnSmall], iv[kSnSmall];
#pragma unroll
        for (int j = 0; j < kSnSmall; ++j)
#pragma unroll
            for (int i = 0; i <= j; ++i)
                if (j < w) A[j][i] = i == j ? d.diag0[(int64_t)c[j] * B + s] : d.W[(int64_t)(lp[i] + j - i - 1) * B + s];
        const int t1 = min(task.r0 + kPanelRows, nr);
        double a[4][kSnSmall];   // the first four rows travel with the block
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int i = 0; i < kSnSmall; ++i)
                if (i < w && t1 > task.r0) a[r][i] = d.W[(int64_t)(lp[i] + w - 1 - i + min(task.r0 + r, t1 - 1)) * B + s];
#pragma unroll
        for (int i = 0; i < kSnSmall; ++i) {
            if (i < w) {
                iv[i] = 1.0 / A[i][i];
#pragma unroll
                for (int k = i + 1; k < kSnSmall; ++k) {
                    if (k < w) {
                        const double f = A[k][i] * iv[i];
#pragma unroll
                        for (int j = k; j < kSnSmall; ++j)
                            if (j < w) A[j][k] -= A[j][i] * f;
                    }
                }
            }
        }
#pragma unroll
        for (int j = 1; j < kSnSmall; ++j)   // L = W / d
#pragma unroll
            for (int i = 0; i < j; ++i)
                if (j < w) A[j][i] *= iv[i];
        if (task.r0 == 0 && live) {
            const int64_t off = P->off;
#pragma unroll
            for (int j = 0; j < kSnSmall; ++j) {
                if (j < w) {
                    d.invd[(int64_t)c[j] * B + s] = iv[j];
#pragma unroll
                    for (int i = 0; i < j; ++i) d.PB[(off + sn_tri(j, i)) * B + s] = A[j][i];
                }
            }
        }
        for (int t = task.r0; t < t1; t += 4) {   // four rows in flight
            if (t > task.r0) {
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int i = 0; i < kSnSmall; ++i)
                        if (i < w) a[r][i] = d.W[(int64_t)(lp[i] + w - 1 - i + min(t + r, t1 - 1)) * B + s];
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                if (t + r < t1) {
#pragma unroll
                    for (int k = 0; k < kSnSmall; ++k) {
                        if (k < w) {
                            if (k > 0 && live) d.W[(int64_t)(lp[k] + w - 1 - k + t + r) * B + s] = a[r][k];
#pragma unroll
                            for (int i = k + 1; i < kSnSmall; ++i)
                                if (i < w) a[r][i] -= a[r][k] * A[i][k];
                        }
                    }
                }
            }
        }
        return;
    }
    // ---- wide panels: the diagonal block
    const KktPanel *P = d.panels + p0 + blockIdx.x;
    const int w = P->w;
    if (threadIdx.x < kSnMax) {
        pc[threadIdx.x] = P->col[threadIdx.x];
        pl[threadIdx.x] = P->lp[threadIdx.x];
    }
    __syncthreads();
    pdl_wait();
    {   // entries e = warp, warp + nw, ... of the packed lower triangle
        int j = 0, i = warp;
        while (i > j) i -= ++j;
        while (j < w) {
            cp_async8(&S[sn_tri(j, i)][lane], i == j ? d.diag0 + (int64_t)pc[j] * B + s : d.W + (int64_t)(pl[i] + j - i - 1) * B + s);
            i += nw;
            while (i > j) i -= ++j;
        }
        cp_async_wait_all();
    }
    __syncthreads();
    for (int i = 0; i < w; ++i) {
        const double iv = 1.0 / S[sn_tri(i, i)][lane];
        if (warp == 0) Iv[i][lane] = iv;
        // rows i+1 .. w-1 of the trailing block, a long and a short one per warp
#pragma unroll
        for (int pass = 0; pass < 2; ++pass) {
            const int ja = i + 1 + warp, jb = w - 1 - warp;
            const int j = pass == 0 ? ja : jb;
            if (pass == 0 ? ja <= jb : jb > ja) {
                const double g = S[sn_tri(j, i)][lane] * iv;
#pragma unroll 4
                for (int k = i + 1; k <= j; ++k) S[sn_tri(j, k)][lane] -= g * S[sn_tri(k, i)][lane];
            }
        }
        __syncthreads();
    }
    if (live) {
        const int64_t off = P->off;
        int j = 0, i = warp;
        while (i > j) i -= ++j;
        while (j < w) {
            if (i == j)
                d.invd[(int64_t)pc[j] * B + s] = Iv[j][lane];
            else
                d.PB[(off + sn_tri(j, i)) * B + s] = S[sn_tri(j, i)][lane] * Iv[i][lane];
            i += nw;
            while (i > j) i -= ++j;
        }
    }
}
__global__ void __launch_bounds__(kPanelThreads, 2) k_sn_rows(KktDev d, int B, int t0, const ScenState *st) {
    pdl_trigger();
    __shared__ double L[kSnTri][32];
    __shared__ int pl[kSnMax];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int nw = kPanelThreads / 32;
    const int s = min((int)blockIdx.y * 32 + lane, B - 1);   // single LP (B == 1): lane 0 works, the others shadow it
    const bool live = (int)blockIdx.y * 32 + lane < B && st[s].status < 0;
    const KktPanelTask task = d.ptasks[t0 + blockIdx.x];
    const KktPanel *P = d.panels + task.panel;
    const int w = P->w, nr = P->nr;
    const int64_t off = P->off;
    if (threadIdx.x < kSnMax) pl[threadIdx.x] = P->lp[threadIdx.x];
    __syncthreads();
    pdl_wait();
    {   // strictly lower entries of the factorised block
        int j = 1, i = warp;
        while (i >= j) i -= j++;
        while (j < w) {
            cp_async8(&L[sn_tri(j, i)][lane], d.PB + (off + sn_tri(j, i)) * B + s);
            i += nw;
            while (i >= j) i -= j++;
        }
    }
    const int t1 = min(task.r0 + kPanelRowsWide, nr);
    const int t = task.r0 + warp;   // kPanelRowsWide == 2 * nw: two rows per warp
    double a[2][kSnMax];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < kSnMax; ++i)
            if (i < w) a[r][i] = d.W[(int64_t)(pl[i] + w - 1 - i + min(t + r * nw, nr - 1)) * B + s];
    cp_async_wait_all();
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kSnMax; ++k) {
        if (k < w) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (k > 0 && live && t + r * nw < t1) d.W[(int64_t)(pl[k] + w - 1 - k + t + r * nw) * B + s] = a[r][k];
            }
#pragma unroll
            for (int i = k + 1; i < kSnMax; ++i) {
                if (i < w) {
                    const double l = L[sn_tri(i, k)][lane];
                    a[0][i] -= a[0][k] * l;
                    a[1][i] -= a[1][k] * l;
                }
            }
        }
    }
}
// the supernode's part of a substitution: v_S <- L_SS^-1 v_S (FWD, before the step's fan-out) or L_SS'^-1 v_S (after
// the contributions of the higher steps, before the fan-out to the descendants).  Wide panels: a block per panel, the
// factorised block goes to shared memory in one asynchronous sweep, the first warp walks it (w dependent steps);
// narrow panels: a warp each, in registers
constexpr int kPanelSolveThreads = 128;
template <bool FWD>
__global__ void __launch_bounds__(kPanelSolveThreads) k_sn_solve(KktDev d, double *v, int B, int p0, int nwide, int npanels, const ScenState *st) {
    pdl_trigger();
    __shared__ double S[kSnTri][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int nw = kPanelSolveThreads / 32;
    const int s = min((int)blockIdx.y * 32 + lane, B - 1);   // single LP (B == 1): lane 0 works, the others shadow it
    const bool live = (int)blockIdx.y * 32 + lane < B && st[s].status < 0;
    if ((int)blockIdx.x >= nwide) {   // ---- narrow panels
        const int pi = nwide + ((int)blockIdx.x - nwide) * nw + warp;
        if (pi >= npanels) return;
        const KktPanel *P = d.panels + p0 + pi;
        const int w = P->w;
        const int64_t off = P->off;
        int nd[kSnSmall];
#pragma unroll
        for (int i = 0; i < kSnSmall; ++i) nd[i] = P->node[i];
        pdl_wait();
        double L[kSnSmall][kSnSmall], x[kSnSmall];
#pragma unroll
        for (int j = 0; j < kSnSmall; ++j) {
            if (j < w) {
                x[j] = v[(int64_t)nd[j] * B + s];
#pragma unroll
                for (int i = 0; i < j; ++i) L[j][i] = d.PB[(off + sn_tri(j, i)) * B + s];
            }
        }
        if (FWD) {
#pragma unroll
            for (int j = 1; j < kSnSmall; ++j) {
                if (j < w) {
#pragma unroll
                    for (int i = 0; i < j; ++i) x[j] -= L[j][i] * x[i];
                    if (live) v[(int64_t)nd[j] * B + s] = x[j];
                }
            }
        } else {
#pragma unroll
            for (int i = kSnSmall - 2; i >= 0; --i) {
                if (i < w - 1) {
#pragma unroll
                    for (int j = i + 1; j < kSnSmall; ++j)
                        if (j < w) x[i] -= L[j][i] * x[j];
                    if (live) v[(int64_t)nd[i] * B + s] = x[i];
                }
            }
        }
        return;
    }
    // ---- wide panels
    const KktPanel *P = d.panels + p0 + blockIdx.x;
    const int w = P->w;
    const int64_t off = P->off;
    pdl_wait();
    {
        int j = 1, i = warp;
        while (i >= j) i -= j++;
        while (j < w) {
            cp_async8(&S[sn_tri(j, i)][lane], d.PB + (off + sn_tri(j, i)) * B + s);
            i += nw;
            while (i >= j) i -= j++;
        }
    }
    double x[kSnMax];
    if (warp == 0) {
#pragma unroll
        for (int j = 0; j < kSnMax; ++j)
            if (j < w) x[j] = v[(int64_t)P->node[j] * B + s];
    }
    cp_async_wait_all();
    __syncthreads();
    if (warp != 0) return;
    if (FWD) {
#pragma unroll
        for (int i = 0; i < kSnMax; ++i) {
            if (i < w) {
                if (i > 0 && live) v[(int64_t)P->node[i] * B + s] = x[i];
#pragma unroll
                for (int j = i + 1; j < kSnMax; ++j)
                    if (j < w) x[j] -= S[sn_tri(j, i)][lane] * x[i];
            }
        }
    } else {
#pragma unroll
        for (int j = kSnMax - 1; j >= 0; --j) {
            if (j < w) {
                if (j < w - 1 && live) v[(int64_t)P->node[j] * B + s] = x[j];
#pragma unroll
                for (int i = 0; i < j; ++i) x[i] -= S[sn_tri(j, i)][lane] * x[j];
            }
        }
    }
}

// assembled lower triangle: the scaled Jacobian values at their place in L, zero on the fill
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_kkt_scatter(LpView v, KktDev d, int64_t nnz) {
    Map<BATCH> mp;
    const int B = v.B;
    for (int64_t q = mp.first; q < nnz; q += mp.stride) d.W[(int64_t)d.kmap[q] * B + mp.s] = v.A[q * B + mp.s];
}

// =================================== barrier iteration ==========================================================
struct ColFlags {
    bool fx, hl, hu;
};
__device__ __forceinline__ ColFlags col_flags(double l, double u) {
    ColFlags f;
    f.fx = (l == u);
    f.hl = ipm_fin(l) && !f.fx;
    f.hu = ipm_fin(u) && !f.fx;
    return f;
}
struct RowFlags {
    bool eq, gl, gu;
};
__device__ __forceinline__ RowFlags row_flags(double l, double u) {
    RowFlags f;
    f.eq = (l == u);
    f.gl = ipm_fin(l) && !f.eq;
    f.gu = ipm_fin(u) && !f.eq;
    return f;
}

// starting point: x inside its box (0 where the box allows), w = Kx pushed inside the row bounds, z = 1 / slack, y = 0
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_init_cols(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    double acc[3] = {0.0, 0.0, 0.0};  // complementarity pairs, inconsistent boxes, |x|^2 unscaled
    const double inv_sb = 1.0 / v.state[mp.s].sb;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double l = v.lbs[e], u = v.ubs[e];
        const ColFlags f = col_flags(l, u);
        double x0 = 0.0;
        if (f.fx)
            x0 = l;
        else if (f.hl && f.hu)
            x0 = fmin(fmax(0.0, l + 0.1 * (u - l)), u - 0.1 * (u - l));
        else if (f.hl)
            x0 = fmax(0.0, l + 1.0);
        else if (f.hu)
            x0 = fmin(0.0, u - 1.0);
        g.x[e] = x0;
        // centred start: every complementarity product is 1, whatever the width of the box (a collapsed trust region
        // gives boxes of 1e-6 next to row slacks of order one)
        g.zlx[e] = f.hl ? 1.0 / (x0 - l) : 0.0;
        g.zux[e] = f.hu ? 1.0 / (u - x0) : 0.0;
        acc[0] += (f.hl ? 1.0 : 0.0) + (f.hu ? 1.0 : 0.0);
        if (l > u) acc[1] += 1.0;
        const double xu = x0 * v.dc[e] * inv_sb;
        acc[2] += xu * xu;
    }
    block_reduce_store<BATCH, 3>(acc, 0u, v.partials, 0, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_init_rows(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    double acc[2] = {0.0, 0.0};
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        const double l = v.rls[e], u = v.rus[e];
        const RowFlags f = row_flags(l, u);
        const double ax = spmv_row(v.A, v.col_idx, g.x, v.row_ptr[i], v.row_ptr[i + 1], B, mp.s);
        double w0 = ax;
        if (f.eq)
            w0 = l;
        else if (f.gl && f.gu)
            w0 = fmin(fmax(ax, l + 0.1 * (u - l)), u - 0.1 * (u - l));
        else if (f.gl)
            w0 = fmax(ax, l + 1.0);
        else if (f.gu)
            w0 = fmin(ax, u - 1.0);
        g.w[e] = w0;
        g.y[e] = 0.0;
        g.zlw[e] = f.gl ? 1.0 / (w0 - l) : 0.0;
        g.zuw[e] = f.gu ? 1.0 / (u - w0) : 0.0;
        acc[0] += (f.gl ? 1.0 : 0.0) + (f.gu ? 1.0 : 0.0);
        if (l > u) acc[1] += 1.0;
    }
    block_reduce_store<BATCH, 2>(acc, 0u, v.partials, 3, B);
}
__global__ void __launch_bounds__(kFinalThreads) k_ipm_init_state(LpView v, IpmView g) {
    const int s = blockIdx.x, B = v.B;
    const double nc = final_reduce(v.partials, 0, v.nbx_cols, B, s, false);
    const double badc = final_reduce(v.partials, 1, v.nbx_cols, B, s, false);
    const double xn2 = final_reduce(v.partials, 2, v.nbx_cols, B, s, false);
    const double nr = final_reduce(v.partials, 3, v.nbx_rows, B, s, false);
    const double badr = final_reduce(v.partials, 4, v.nbx_rows, B, s, false);
    if (threadIdx.x) return;
    ScenState *st = v.state + s;
    IpmState it;
    it.mu = 1.0;
    it.smu = 0.0;
    it.ap = it.ad = 0.0;
    {
        const double xn = fmax(1.0, sqrt(xn2));
        it.q_un = g.prox * fmin(0.5 * (1.0 + st->nc_un) / xn, 1.0 / (xn * xn));
    }
    it.qs = it.q_un * st->sc / st->sb;
    it.ncomp = (int)(nc + nr + 0.5);
    it.hits = 0;
    it.acc_hits = 0;
    it.save = 0;
    it.ray_obj = -1.0;
    it.ray_kty = 1.0;
    for (double &k : it.kept) k = 0.0;
    it.bad = (badc + badr) > 0.0;
    g.ist[s] = it;
    if (st->status < 0 && it.bad) {  // lb > ub or rl > ru: nothing to iterate on
        st->status = ASM_LP_INFEASIBLE;
        st->total = 0;
        atomicSub(v.n_active, 1);
    }
}

// residuals of the barrier system and everything the termination / Farkas tests need
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_res_cols(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const bool live = st->status < 0;
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (live) {
        const double inv_sc = 1.0 / st->sc, inv_sb = 1.0 / st->sb, qs = g.ist[mp.s].qs;
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            const double l = v.lbs[e], u = v.ubs[e], c = v.cs[e], x = g.x[e], d = v.dc[e];
            const ColFlags f = col_flags(l, u);
            const double aty = spmv_row(v.AT, v.row_idx, g.y, v.col_ptr[j], v.col_ptr[j + 1], B, mp.s);
            const double Q = f.fx ? 0.0 : qs * d * d;
            const double zl = g.zlx[e], zu = g.zux[e];
            const double rlp = c - aty - zl + zu;
            const double r = rlp + Q * x;
            g.rdx[e] = r;
            if (!f.fx) {
                const double ru = r * inv_sc / d, rl2 = rlp * inv_sc / d;
                acc[I_RDX2] += ru * ru;
                acc[I_RLP2] += rl2 * rl2;
            }
            acc[I_POBJ] += c * x;
            acc[I_QT] += 0.5 * Q * x * x;
            acc[I_DOBJC] += (f.hl ? l * zl : 0.0) - (f.hu ? u * zu : 0.0) + (f.fx ? l * (c - aty) : 0.0);
            acc[I_MUC] += (f.hl ? zl * (x - l) : 0.0) + (f.hu ? zu * (u - x) : 0.0);
            const double xu = x * d * inv_sb;
            acc[I_XN2] += xu * xu;
            const double t = -aty;
            acc[I_RAYC] += t > 0.0 ? t * l : (t < 0.0 ? t * u : 0.0);
            acc[I_KTY] = fmax(acc[I_KTY], fabs(aty / d));
        }
    }
    block_reduce_store<BATCH, 9>(acc, 1u << I_KTY, v.partials, 0, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_res_rows(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const ScenState *st = v.state + mp.s;
    const bool live = st->status < 0;
    double acc[6] = {0, 0, 0, 0, 0, 0};
    if (live) {
        const double inv_sc = 1.0 / st->sc, inv_sb = 1.0 / st->sb;
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            const double l = v.rls[e], u = v.rus[e], d = v.dr[e], y = g.y[e];
            const RowFlags f = row_flags(l, u);
            const double ax = spmv_row(v.A, v.col_idx, g.x, v.row_ptr[i], v.row_ptr[i + 1], B, mp.s);
            const double w = f.eq ? l : g.w[e];
            const double zl = g.zlw[e], zu = g.zuw[e];
            const double rp = ax - w;
            const double rd = f.eq ? 0.0 : y - zl + zu;
            g.rp[e] = rp;
            g.rdw[e] = rd;
            const double rpu = rp * inv_sb / d, rdu = rd * d * inv_sc;
            acc[0] += rpu * rpu;
            acc[1] += rdu * rdu;
            acc[2] += f.eq ? l * y : ((f.gl ? l * zl : 0.0) - (f.gu ? u * zu : 0.0));
            acc[3] += (f.gl ? zl * (w - l) : 0.0) + (f.gu ? zu * (u - w) : 0.0);
            acc[4] += y > 0.0 ? l * y : (y < 0.0 ? u * y : 0.0);
            acc[5] = fmax(acc[5], fabs(y * d));
        }
    }
    block_reduce_store<BATCH, 6>(acc, 1u << 5, v.partials, I_RP2, B);
}

// one block per LP: termination, Farkas test, proximal weight of the next step
__global__ void __launch_bounds__(kFinalThreads) k_ipm_decide(LpView v, IpmView g, int iter, int last) {
    const int s = blockIdx.x, B = v.B;
    ScenState *sp = v.state + s;
    if (sp->status >= 0) return;
    double q[I_COUNT];
    for (int i = 0; i < I_COUNT; ++i)
        q[i] = final_reduce(v.partials, i, i >= I_RP2 ? v.nbx_rows : v.nbx_cols, B, s, i == I_KTY || i == I_YMAX);
    if (threadIdx.x) return;
    ScenState st = *sp;
    IpmState it = g.ist[s];
    const double unit = 1.0 / (st.sb * st.sc);
    const double pq = (q[I_POBJ] + q[I_QT]) * unit, dq = (q[I_DOBJC] + q[I_DOBJR] - q[I_QT]) * unit;
    const double pres = sqrt(q[I_RP2]), dres = sqrt(q[I_RDX2] + q[I_RDW2]);
    const double gapq = fabs(pq - dq);
    it.mu = it.ncomp > 0 ? (q[I_MUC] + q[I_MUR]) / it.ncomp : 0.0;
    // what is reported is measured against the LP itself (no proximal term)
    st.pobj = q[I_POBJ] * unit;
    st.dobj = (q[I_DOBJC] + q[I_DOBJR]) * unit;
    st.pres = pres;
    st.dres = sqrt(q[I_RLP2] + q[I_RDW2]);
    st.gap = fabs(st.pobj - st.dobj);
    st.total = iter;
    const double c0 = g.c0[s];
    const double gden = 1.0 + fabs(pq + c0) + fabs(dq + c0);
    auto within = [&](double e) {
        return pres <= e * (1.0 + st.nq_un) && dres <= e * (1.0 + st.nc_un) && gapq <= e * gden;
    };
    const bool nan = !(pres == pres) || !(dres == dres) || !(gapq == gapq) || !(it.mu == it.mu);
    const bool conv = !nan && within(g.eps), acc = !nan && within(g.eps_acc);
    int status = -1;
    it.save = 0;
    if (conv) {
        // a few more steps drive the complementarity down until the variables on a bound reach it to machine precision
        // (what a vertex solver returns, and what the reference's == tests on bounds expect, subproblem.jl:522-529)
        // and sharpen the least-norm selection
        it.hits += 1;
        it.save = 1;
        if ((it.hits > g.extra_hits && it.mu <= g.mu_target) || it.hits > g.extra_hits + 4 || it.mu <= 1e-26)
            status = ASM_LP_OPTIMAL;
    } else if (it.hits > 0) {
        status = ASM_LP_OPTIMAL;  // the point saved at the previous step stands
    } else if (acc) {
        // acceptable but not at the target: keep the point as fall-back result.  When that lasts, the accuracy of the
        // linear solves is what holds the last digits back (the gap inherits |x| times the dual residual): ask the host
        // for one more refinement pass after 5 and after 8 such steps, and settle for the acceptable point after 12.
        it.acc_hits += 1;
        it.save = 1;
        if (it.acc_hits == 5 || it.acc_hits == 8) atomicAdd(g.need_refine, 1);
        if (it.acc_hits >= 12) status = ASM_LP_OPTIMAL;
    } else if (nan) {
        status = it.acc_hits > 0 ? ASM_LP_OPTIMAL : ASM_LP_NUMERICAL_ERROR;
    } else {
        // Farkas certificate from y itself and from the last step direction dy (the one that grows when the LP is
        // infeasible); both normalised to |ray|_inf = 1 in unscaled units
        const double nr = q[I_YMAX] / st.sc;
        if (nr > 0.0 && iter > 0) {
            const double robj = (q[I_RAYR] + q[I_RAYC]) * unit / nr;
            const double kty = q[I_KTY] / st.sc / nr;
            if (robj > v.prm->eps_infeas * fmax(1.0, kty)) status = ASM_LP_INFEASIBLE;
        }
        if (status < 0 && it.acc_hits == 0 && it.ray_obj > v.prm->eps_infeas * fmax(1.0, it.ray_kty)) status = ASM_LP_INFEASIBLE;
    }
    // safety net: an LP that is still short of the acceptable level after 40 (60) Newton steps is most likely held
    // back by the accuracy of the linear solves as well
    if (status < 0 && it.acc_hits == 0 && (iter == 40 || iter == 60)) atomicAdd(g.need_refine, 1);
    if (status < 0 && last) {
        status = it.acc_hits > 0 ? ASM_LP_OPTIMAL : ASM_LP_ITERATION_LIMIT;
        if (it.acc_hits == 0) it.save = 1;
    }
    if (it.save) {
        it.kept[0] = st.pobj;
        it.kept[1] = st.dobj;
        it.kept[2] = st.pres;
        it.kept[3] = st.dres;
        it.kept[4] = st.gap;
    } else if (status == ASM_LP_OPTIMAL) {  // the result is the point kept earlier: report its numbers
        st.pobj = it.kept[0];
        st.dobj = it.kept[1];
        st.pres = it.kept[2];
        st.dres = it.kept[3];
        st.gap = it.kept[4];
    }
    if (g.verbose && s == 0)
        printf("[ipm] it %3d pres %.3e dres %.3e gap %.3e mu %.3e pobj %.12e q %.3e ap %.3f ad %.3f ray %.2e%s%s\n", iter,
               pres / (1.0 + st.nq_un), dres / (1.0 + st.nc_un), gapq / gden, it.mu, st.pobj + c0, it.q_un, it.ap, it.ad,
               it.ray_obj, acc ? " a" : "", status >= 0 ? " *" : "");
    // proximal weight of the next step: the dual residual q |x| it leaves in the LP stays below prox (1 + |c|) / 2 and
    // the duality gap q |x|^2 below prox (1 + 2 |c'x|)
    {
        const double xn = fmax(1.0, sqrt(q[I_XN2]));
        const double qn = g.prox * fmin(0.5 * (1.0 + st.nc_un) / xn, (1.0 + 2.0 * fabs(st.pobj)) / (xn * xn));
        // hysteresis: a weight that drifts by a percent per step re-introduces a dual residual of that size at every
        // step and the last digits never settle (seen on restoration LPs: the gap stalled at 8e-8)
        if (!(qn > 0.5 * it.q_un && qn < 2.0 * it.q_un)) it.q_un = qn;
        it.qs = it.q_un * st.sc / st.sb;
    }
    g.ist[s] = it;
    if (status >= 0) {
        st.status = status;
        atomicSub(v.n_active, 1);
    }
    *sp = st;
}

// keep the current point as the result (xp, yp, reduced costs in gyp -- what k_finalize reads); variables that sit
// strictly complementary on a bound go exactly onto it
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_save(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    if (!g.ist[mp.s].save) return;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double l = v.lbs[e], u = v.ubs[e];
        const ColFlags f = col_flags(l, u);
        double x = g.x[e];
        const double zl = g.zlx[e], zu = g.zux[e];
        if (f.fx) {
            x = l;
        } else {
            const double span = (f.hl && f.hu) ? u - l : 1.0;
            // strictly complementary and closer than 1e-9 relative: moving it onto the bound changes no row by more
            // than the feasibility tolerance
            if (f.hl && x - l < zl && x - l <= 1e-9 * fmax(span, fabs(l))) x = l;
            if (f.hu && u - x < zu && u - x <= 1e-9 * fmax(span, fabs(u))) x = u;
        }
        v.xp[e] = x;
        v.gyp[e] = f.fx ? g.rdx[e] : zl - zu;
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        v.yp[e] = g.y[e];
    }
}

// objective of the returned (snapped) point, so that the reported number is the one of the point the caller receives
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_final_obj(LpView v) {
    Map<BATCH> mp;
    const int B = v.B;
    double acc[1] = {0.0};
    for (int64_t j = mp.first; j < v.n; j += mp.stride) acc[0] += v.cs[j * B + mp.s] * v.xp[j * B + mp.s];
    block_reduce_store<BATCH, 1>(acc, 0u, v.partials, 0, B);
}
__global__ void __launch_bounds__(kFinalThreads) k_ipm_final_state(LpView v, int Buser) {
    const int s = blockIdx.x, B = v.B;
    const double q = final_reduce(v.partials, 0, v.nbx_cols, B, s, false);
    if (threadIdx.x || s >= Buser) return;
    ScenState *st = v.state + s;
    if (st->status == ASM_LP_OPTIMAL || st->status == ASM_LP_ITERATION_LIMIT) {
        const double pobj = q / (st->sb * st->sc);
        st->gap = fabs(pobj - st->dobj);
        st->pobj = pobj;
    }
}

// diagonal blocks of the Newton system
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_diag(LpView v, IpmView g, KktDev d) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    const double qs = g.ist[mp.s].qs;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double l = v.lbs[e], u = v.ubs[e], x = g.x[e], dc = v.dc[e];
        const ColFlags f = col_flags(l, u);
        double D = (f.hl ? g.zlx[e] / ipm_slack(x - l) : 0.0) + (f.hu ? g.zux[e] / ipm_slack(u - x) : 0.0) + qs * dc * dc;
        if (f.fx) D = 1e20;
        g.Dx[e] = D;
        d.diag0[(int64_t)d.inv[j] * B + mp.s] = -(D + g.delta);
        d.invd[(int64_t)d.inv[j] * B + mp.s] = -1.0 / (D + g.delta);
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        const double l = v.rls[e], u = v.rus[e], w = g.w[e];
        const RowFlags f = row_flags(l, u);
        const double D = (f.gl ? g.zlw[e] / ipm_slack(w - l) : 0.0) + (f.gu ? g.zuw[e] / ipm_slack(u - w) : 0.0);
        const double E = f.eq ? 0.0 : fmin(1.0 / fmax(D, 1e-300), 1e20);
        g.Ew[e] = E;
        d.diag0[(int64_t)d.inv[v.n + i] * B + mp.s] = E + g.delta;
        d.invd[(int64_t)d.inv[v.n + i] * B + mp.s] = 1.0 / (E + g.delta);
    }
}

// right-hand side of the reduced system; CORR adds the centring target sigma*mu and the second-order products
template <bool BATCH, bool CORR>
__global__ void __launch_bounds__(kThreads) k_ipm_rhs(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    const double smu = CORR ? g.ist[mp.s].smu : 0.0;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double l = v.lbs[e], u = v.ubs[e], x = g.x[e];
        const ColFlags f = col_flags(l, u);
        const double tl = f.hl ? (smu - (CORR ? g.clx[e] : 0.0)) / ipm_slack(x - l) - g.zlx[e] : 0.0;
        const double tu = f.hu ? (smu - (CORR ? g.cux[e] : 0.0)) / ipm_slack(u - x) - g.zux[e] : 0.0;
        const double r = f.fx ? 0.0 : -(-g.rdx[e] + tl - tu);
        g.rhs0[e] = r;
        g.sol[e] = r;
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        const double l = v.rls[e], u = v.rus[e], w = g.w[e];
        const RowFlags f = row_flags(l, u);
        const double tl = f.gl ? (smu - (CORR ? g.clw[e] : 0.0)) / ipm_slack(w - l) - g.zlw[e] : 0.0;
        const double tu = f.gu ? (smu - (CORR ? g.cuw[e] : 0.0)) / ipm_slack(u - w) - g.zuw[e] : 0.0;
        const double rw = -g.rdw[e] + tl - tu;
        const double r = -g.rp[e] + (f.eq ? 0.0 : g.Ew[e] * rw);
        const int64_t en = ((int64_t)v.n + i) * B + mp.s;
        g.rhs0[en] = r;
        g.sol[en] = r;
    }
}

// iterative refinement: work = rhs0 - M0 sol with the unregularised blocks
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_kkt_res_cols(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    const double *s2 = g.sol + (int64_t)v.n * B;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        const double a = spmv_row(v.AT, v.row_idx, s2, v.col_ptr[j], v.col_ptr[j + 1], B, mp.s);
        g.work[e] = g.rhs0[e] - (a - g.Dx[e] * g.sol[e]);
    }
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_kkt_res_rows(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t en = ((int64_t)v.n + i) * B + mp.s;
        const double a = spmv_row(v.A, v.col_idx, g.sol, v.row_ptr[i], v.row_ptr[i + 1], B, mp.s);
        g.work[en] = g.rhs0[en] - (a + g.Ew[i * B + mp.s] * g.sol[en]);
    }
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_kkt_add(LpView v, IpmView g, int64_t N) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    for (int64_t i = mp.first; i < N; i += mp.stride) g.sol[i * B + mp.s] += g.work[i * B + mp.s];
}

// directions of the eliminated variables and the ratio tests (as max of -d/s, no division by a small slack)
template <bool BATCH, bool CORR>
__global__ void __launch_bounds__(kThreads) k_ipm_dirs_cols(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};
    if (live) {
        const double smu = CORR ? g.ist[mp.s].smu : 0.0;
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            const double l = v.lbs[e], u = v.ubs[e], x = g.x[e];
            const ColFlags f = col_flags(l, u);
            if (f.fx) g.sol[e] = 0.0;
            const double dx = f.fx ? 0.0 : g.sol[e];
            double dl = 0.0, du = 0.0;
            if (f.hl) {
                const double sl = ipm_slack(x - l), z = fmax(g.zlx[e], 1e-300);
                dl = (smu - (CORR ? g.clx[e] : 0.0)) / sl - z - z / sl * dx;
                acc[0] = fmax(acc[0], -dx / sl);
                acc[1] = fmax(acc[1], -dl / z);
            }
            if (f.hu) {
                const double su = ipm_slack(u - x), z = fmax(g.zux[e], 1e-300);
                du = (smu - (CORR ? g.cux[e] : 0.0)) / su - z + z / su * dx;
                acc[0] = fmax(acc[0], dx / su);
                acc[1] = fmax(acc[1], -du / z);
            }
            g.dzlx[e] = dl;
            g.dzux[e] = du;
        }
    }
    block_reduce_store<BATCH, 2>(acc, 3u, v.partials, J_AP, B);
}
template <bool BATCH, bool CORR>
__global__ void __launch_bounds__(kThreads) k_ipm_dirs_rows(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};
    if (live) {
        const double smu = CORR ? g.ist[mp.s].smu : 0.0;
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            const double l = v.rls[e], u = v.rus[e], w = g.w[e];
            const RowFlags f = row_flags(l, u);
            const double dy = g.sol[((int64_t)v.n + i) * B + mp.s];
            const double tl = f.gl ? (smu - (CORR ? g.clw[e] : 0.0)) / ipm_slack(w - l) - g.zlw[e] : 0.0;
            const double tu = f.gu ? (smu - (CORR ? g.cuw[e] : 0.0)) / ipm_slack(u - w) - g.zuw[e] : 0.0;
            const double dw = f.eq ? 0.0 : g.Ew[e] * (-g.rdw[e] + tl - tu - dy);
            double dl = 0.0, du = 0.0;
            if (f.gl) {
                const double sl = ipm_slack(w - l), z = fmax(g.zlw[e], 1e-300);
                dl = tl - z / sl * dw;
                acc[0] = fmax(acc[0], -dw / sl);
                acc[1] = fmax(acc[1], -dl / z);
            }
            if (f.gu) {
                const double su = ipm_slack(u - w), z = fmax(g.zuw[e], 1e-300);
                du = tu + z / su * dw;
                acc[0] = fmax(acc[0], dw / su);
                acc[1] = fmax(acc[1], -du / z);
            }
            g.dw[e] = dw;
            g.dzlw[e] = dl;
            g.dzuw[e] = du;
        }
    }
    block_reduce_store<BATCH, 2>(acc, 3u, v.partials, J_AP_R, B);
}
// complementarity after the affine step and the second-order products of the corrector
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_muaff(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};  // columns, rows
    if (live) {
        const double ap = g.ist[mp.s].ap, ad = g.ist[mp.s].ad;
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            const double l = v.lbs[e], u = v.ubs[e], x = g.x[e];
            const ColFlags f = col_flags(l, u);
            const double dx = g.sol[e];
            if (f.hl) {
                acc[0] += (x - l + ap * dx) * (g.zlx[e] + ad * g.dzlx[e]);
                g.clx[e] = dx * g.dzlx[e];
            }
            if (f.hu) {
                acc[0] += (u - x - ap * dx) * (g.zux[e] + ad * g.dzux[e]);
                g.cux[e] = -dx * g.dzux[e];
            }
        }
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            const double l = v.rls[e], u = v.rus[e], w = g.w[e];
            const RowFlags f = row_flags(l, u);
            const double dw = g.dw[e];
            if (f.gl) {
                acc[1] += (w - l + ap * dw) * (g.zlw[e] + ad * g.dzlw[e]);
                g.clw[e] = dw * g.dzlw[e];
            }
            if (f.gu) {
                acc[1] += (u - w - ap * dw) * (g.zuw[e] + ad * g.dzuw[e]);
                g.cuw[e] = -dw * g.dzuw[e];
            }
        }
    }
    block_reduce_store<BATCH, 2>(acc, 0u, v.partials, J_MUC, B);
}
// Farkas quantities of the step direction dy = sol[n:], projected on the sign cone of the one-sided rows
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_ray(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};  // row part, |ray|_inf
    if (live) {
        double *ray = g.work + (int64_t)v.n * B;   // the refinement buffer is free at this point
        for (int64_t i = mp.first; i < v.m; i += mp.stride) {
            const int64_t e = i * B + mp.s;
            const double l = v.rls[e], u = v.rus[e];
            double d = g.sol[((int64_t)v.n + i) * B + mp.s];
            if (!ipm_fin(l)) d = fmin(d, 0.0);
            if (!ipm_fin(u)) d = fmax(d, 0.0);
            ray[e] = d;
            acc[0] += d > 0.0 ? l * d : (d < 0.0 ? u * d : 0.0);
            acc[1] = fmax(acc[1], fabs(d * v.dr[e]));
        }
    }
    block_reduce_store<BATCH, 2>(acc, 2u, v.partials, J_RAY, B);
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_ray_cols(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    const bool live = v.state[mp.s].status < 0;
    double acc[2] = {0.0, 0.0};  // column part (box support of -K'ray), |K'ray|_inf
    if (live) {
        const double *ray = g.work + (int64_t)v.n * B;
        for (int64_t j = mp.first; j < v.n; j += mp.stride) {
            const int64_t e = j * B + mp.s;
            const double a = spmv_row(v.AT, v.row_idx, ray, v.col_ptr[j], v.col_ptr[j + 1], B, mp.s);
            const double t = -a;
            acc[0] += t > 0.0 ? t * v.lbs[e] : (t < 0.0 ? t * v.ubs[e] : 0.0);
            acc[1] = fmax(acc[1], fabs(a / v.dc[e]));
        }
    }
    block_reduce_store<BATCH, 2>(acc, 2u, v.partials, J_RAY + 2, B);
}
// one block per LP.  mode 0: affine step lengths; 1: sigma from the affine complementarity; 2: damped final lengths
__global__ void __launch_bounds__(kFinalThreads) k_ipm_scalars(LpView v, IpmView g, int mode, int nbx_both) {
    const int s = blockIdx.x, B = v.B;
    if (v.state[s].status >= 0) return;
    if (mode == 1) {
        const double mc = final_reduce(v.partials, J_MUC, nbx_both, B, s, false);
        const double mr = final_reduce(v.partials, J_MUR, nbx_both, B, s, false);
        if (threadIdx.x) return;
        IpmState it = g.ist[s];
        const double mu_aff = it.ncomp > 0 ? (mc + mr) / it.ncomp : 0.0;
        double sg = it.mu > 0.0 ? mu_aff / it.mu : 0.0;
        sg = fmin(fmax(sg, 0.0), 1.0);
        it.smu = sg * sg * sg * it.mu;
        g.ist[s] = it;
        return;
    }
    const double pc = final_reduce(v.partials, J_AP, v.nbx_cols, B, s, true);
    const double dc = final_reduce(v.partials, J_AD, v.nbx_cols, B, s, true);
    const double pr = final_reduce(v.partials, J_AP_R, v.nbx_rows, B, s, true);
    const double dr = final_reduce(v.partials, J_AD_R, v.nbx_rows, B, s, true);
    double rr = 0.0, rm = 0.0, rc = 0.0, rk = 0.0;
    if (mode == 2) {
        rr = final_reduce(v.partials, J_RAY, v.nbx_rows, B, s, false);
        rm = final_reduce(v.partials, J_RAY + 1, v.nbx_rows, B, s, true);
        rc = final_reduce(v.partials, J_RAY + 2, v.nbx_cols, B, s, false);
        rk = final_reduce(v.partials, J_RAY + 3, v.nbx_cols, B, s, true);
    }
    if (threadIdx.x) return;
    const double damp = mode == 2 ? 0.995 : 1.0;
    const double ip = fmax(pc, pr), id = fmax(dc, dr);
    IpmState it = g.ist[s];
    if (mode == 2) {
        const ScenState *st = v.state + s;
        const double nr = rm / st->sc;
        it.ray_obj = nr > 0.0 ? (rr + rc) / (st->sb * st->sc) / nr : -1.0;
        it.ray_kty = nr > 0.0 ? rk / st->sc / nr : 1.0;
    }
    it.ap = ip > damp ? damp / ip : 1.0;
    it.ad = id > damp ? damp / id : 1.0;
    g.ist[s] = it;
}
template <bool BATCH>
__global__ void __launch_bounds__(kThreads) k_ipm_update(LpView v, IpmView g) {
    Map<BATCH> mp;
    const int B = v.B;
    if (v.state[mp.s].status >= 0) return;
    const double ap = g.ist[mp.s].ap, ad = g.ist[mp.s].ad;
    for (int64_t j = mp.first; j < v.n; j += mp.stride) {
        const int64_t e = j * B + mp.s;
        g.x[e] += ap * g.sol[e];
        g.zlx[e] += ad * g.dzlx[e];
        g.zux[e] += ad * g.dzux[e];
    }
    for (int64_t i = mp.first; i < v.m; i += mp.stride) {
        const int64_t e = i * B + mp.s;
        g.w[e] += ap * g.dw[e];
        g.y[e] += ad * g.sol[((int64_t)v.n + i) * B + mp.s];
        g.zlw[e] += ad * g.dzlw[e];
        g.zuw[e] += ad * g.dzuw[e];
    }
}

// =================================== host side ================================================================
struct IpmEngine {
    KktSymbolic sym;
    bool ready = false;
    int B = 0;
    DBuf<int> perm, inv, kmap;
    DBuf<KktRange> fmchunk, wmchunk, bmchunk;
    DBuf<KktPanel> panels;
    DBuf<KktPanelTask> ptasks;
    DBuf<KktTerm> terms;
    DBuf<KktFwdItem> fwd;
    DBuf<KktBwdItem> bwd;
    DBuf<double> W, invd, diag0, PB;
    DBuf<double> colv[9], rowv[12], kktv[3];
    DBuf<IpmState> ist;
    cudaGraphExec_t g_factor = nullptr, g_solve_sol = nullptr, g_solve_work = nullptr;
    int64_t launches_factor = 0, launches_solve = 0;
    double symbolic_ms = 0.0;
    int last_newton = 0;
    int64_t last_pairs = 0, last_factorisations = 0;   // substitution pairs / factorisations of the last solve
    int64_t n_fchunks = 0;
    float last_factor_ms = 0.f, last_solve_ms = 0.f;

    ~IpmEngine() {
        if (g_factor) cudaGraphExecDestroy(g_factor);
        if (g_solve_sol) cudaGraphExecDestroy(g_solve_sol);
        if (g_solve_work) cudaGraphExecDestroy(g_solve_work);
    }

    template <class T>
    static int up(DBuf<T> &dst, const std::vector<T> &src) {
        ASM_TRY(dst.alloc(std::max<size_t>(src.size(), 1)));
        if (!src.empty()) ASM_CK(cudaMemcpy(dst.p, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
        return ASM_OK;
    }

    int init(int n, int m, const std::vector<int> &row_ptr, const std::vector<int> &col_idx, int B_) {
        B = B_;
        for (int i = 0; i < m; ++i) {   // the assembly writes one value per entry of L: no duplicate (row, column) pairs
            std::vector<int> cols(col_idx.begin() + row_ptr[i], col_idx.begin() + row_ptr[i + 1]);
            std::sort(cols.begin(), cols.end());
            if (std::adjacent_find(cols.begin(), cols.end()) != cols.end())
                return fail(ASM_E_INVALID, "duplicate (row, column) entries in the pattern: the barrier engine needs a deduplicated CSR");
        }
        const auto t0 = std::chrono::steady_clock::now();
        if (sym.build(n, m, row_ptr.data(), col_idx.data(), kkt_supernode_width()))
            return fail(ASM_E_INVALID, "KKT symbolic analysis failed (index out of range or more than 2^31 update terms)");
        symbolic_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        ASM_TRY(up(terms, sym.terms));
        ASM_TRY(up(fmchunk, sym.fmchunk));
        ASM_TRY(up(fwd, sym.fwd));
        ASM_TRY(up(wmchunk, sym.wmchunk));
        ASM_TRY(up(bwd, sym.bwd));
        ASM_TRY(up(bmchunk, sym.bmchunk));
        ASM_TRY(up(panels, sym.panels));
        ASM_TRY(up(ptasks, sym.ptasks));
        ASM_TRY(up(perm, sym.perm));
        ASM_TRY(up(inv, sym.inv));
        ASM_TRY(up(kmap, sym.kmap));
        // the big host lists are not needed any more
        std::vector<KktTerm>().swap(sym.terms);
        std::vector<KktFwdItem>().swap(sym.fwd);
        std::vector<KktBwdItem>().swap(sym.bwd);
        std::vector<KktRange>().swap(sym.fmchunk);
        std::vector<KktRange>().swap(sym.wmchunk);
        std::vector<KktRange>().swap(sym.bmchunk);
        n_fchunks = sym.n_fchunks;
        const size_t N = sym.N;
        ASM_TRY(W.alloc(std::max<size_t>(sym.nnzL, 1) * B));
        ASM_TRY(invd.alloc(N * B));
        ASM_TRY(diag0.alloc(N * B));
        ASM_TRY(PB.alloc(std::max<size_t>(sym.panel_slots, 1) * B));
        for (auto &b : colv) ASM_TRY(b.alloc((size_t)n * B));
        for (auto &b : rowv) ASM_TRY(b.alloc((size_t)std::max(m, 1) * B));
        for (auto &b : kktv) ASM_TRY(b.alloc(N * B));
        ASM_TRY(ist.alloc(B));
        ready = true;
        return ASM_OK;
    }

    KktDev dev() const {
        KktDev d;
        d.terms = terms.p;
        d.fmchunk = fmchunk.p;
        d.fwd = fwd.p;
        d.wmchunk = wmchunk.p;
        d.bwd = bwd.p;
        d.bmchunk = bmchunk.p;
        d.panels = panels.p;
        d.ptasks = ptasks.p;
        d.perm = perm.p;
        d.inv = inv.p;
        d.kmap = kmap.p;
        d.W = W.p;
        d.invd = invd.p;
        d.diag0 = diag0.p;
        d.PB = PB.p;
        d.nnzL = (int)sym.nnzL;
        d.N = sym.N;
        return d;
    }
    IpmView iview(const asm_lp_params &P) {
        IpmView g;
        double **c[] = {&g.x, &g.zlx, &g.zux, &g.rdx, &g.Dx, &g.dzlx, &g.dzux, &g.clx, &g.cux};
        for (int i = 0; i < 9; ++i) *c[i] = colv[i].p;
        double **r[] = {&g.w, &g.y, &g.zlw, &g.zuw, &g.rp, &g.rdw, &g.Ew, &g.dw, &g.dzlw, &g.dzuw, &g.clw, &g.cuw};
        for (int i = 0; i < 12; ++i) *r[i] = rowv[i].p;
        g.rhs0 = kktv[0].p;
        g.sol = kktv[1].p;
        g.work = kktv[2].p;
        g.ist = ist.p;
        g.delta = P.ipm_reg > 0.0 ? P.ipm_reg : 1e-8;
        g.prox = P.ipm_prox >= 0.0 ? P.ipm_prox : 1e-7;
        g.eps = std::min(P.eps_rel, 1e-8);
        g.eps_acc = std::max(P.eps_rel, 1e-7);
        g.extra_hits = 2;
        g.mu_target = 1e-19;
        g.verbose = P.verbose;
        return g;
    }

    // launch of a step kernel, as a programmatic dependent of the previous one (see pdl_wait)
    bool use_pdl = getenv("ASM_NO_PDL") == nullptr;
    template <class... KArgs, class... Args>
    void launch_step(void (*kern)(KArgs...), dim3 grid, int block, cudaStream_t st, Args... args) const {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(block);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = use_pdl ? 1 : 0;
        cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
    }
    // grid of a step kernel.  Batch: a warp per item, scenarios over blockIdx.y; single LP: a thread per item
    dim3 level_grid(int items, int multi) const {
        const int per_block = B == 1 ? kThreads : kWarps;
        const int gy = B == 1 ? 1 : B / 32;
        const int64_t cap = std::max<int64_t>(1, (int64_t)kMaxBlocksX * 4 / gy);
        // batch: four single-term chunks per warp pass, one multi-term chunk per warp pass
        const int64_t units = B == 1 ? items : (items - multi + 3) / 4 + multi + 1;
        return dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>((units + per_block - 1) / per_block, cap)), gy);
    }
    void enqueue_factor(LpView &v, cudaStream_t st, int64_t &count) {
        KktDev d = dev();
        cudaMemsetAsync(W.p, 0, W.n * sizeof(double), st);
        const int64_t nz = (int64_t)sym.kmap.size();
        if (nz) {
            const Geo gz = geo_for(nz, B);
            if (B > 1)
                k_kkt_scatter<true><<<gz.grid, gz.block, 0, st>>>(v, d, nz);
            else
                k_kkt_scatter<false><<<gz.grid, gz.block, 0, st>>>(v, d, nz);
        }
        count += 2;
        const int gy = (B + 31) / 32;
        for (int l = 0; l < sym.n_levels; ++l) {   // per step: the panels of its supernodes, then the updates that leave them
            // wide tasks (rows of the wide panels) come first in the step's task range, then the narrow tasks
            const int np = sym.pstep[l + 1] - sym.pstep[l], npw = sym.pwide[l];
            const int nt = sym.ptstep[l + 1] - sym.ptstep[l], ntw = sym.ptwide[l];
            if (np > 0) {
                const int per = kPanelThreads / 32;
                launch_step(k_sn_diag, dim3(npw + (nt - ntw + per - 1) / per, gy), kPanelThreads, st, d, B, sym.pstep[l], npw,
                            sym.ptstep[l] + ntw, nt - ntw, v.state);
                ++count;
            }
            if (ntw > 0) {
                launch_step(k_sn_rows, dim3(ntw, gy), kPanelThreads, st, d, B, sym.ptstep[l], v.state);
                ++count;
            }
            const KktStepRange rg = {sym.fs_beg[l], sym.fs_end[l], sym.fmstep[l], sym.fmstep[l + 1]};
            const int multi = rg.m1 - rg.m0, items = rg.s1 - rg.s0 + multi;
            if (items > 0) {
                launch_step(B > 1 ? k_ldl_factor<true> : k_ldl_factor<false>, level_grid(items, multi), kThreads, st, d, B, v.state, rg);
                ++count;
            }
        }
    }
    void enqueue_solve(LpView &v, double *vec, cudaStream_t st, int64_t &count) {
        KktDev d = dev();
        const int gy = (B + 31) / 32;
        for (int l = 0; l < sym.n_levels; ++l) {
            const int np = sym.pstep[l + 1] - sym.pstep[l], nwide = sym.pwide[l];
            if (np > 0) {
                const int per = kPanelSolveThreads / 32;
                launch_step(k_sn_solve<true>, dim3(nwide + (np - nwide + per - 1) / per, gy), kPanelSolveThreads, st, d, vec, B, sym.pstep[l], nwide, np, v.state);
                ++count;
            }
            const KktStepRange rg = {sym.ws_beg[l], sym.ws_end[l], sym.wmstep[l], sym.wmstep[l + 1]};
            const int multi = rg.m1 - rg.m0, items = rg.s1 - rg.s0 + multi;
            if (items > 0) {
                launch_step(B > 1 ? k_ldl_fwd<true> : k_ldl_fwd<false>, level_grid(items, multi), kThreads, st, d, vec, B, v.state, rg);
                ++count;
            }
        }
        const Geo gN = geo_for(sym.N, B);
        if (B > 1)
            k_ldl_diag<true><<<gN.grid, gN.block, 0, st>>>(d, vec, B, v.state);
        else
            k_ldl_diag<false><<<gN.grid, gN.block, 0, st>>>(d, vec, B, v.state);
        ++count;
        for (int l = sym.n_levels - 1; l >= 0; --l) {
            const int np = sym.pstep[l + 1] - sym.pstep[l], nwide = sym.pwide[l];
            if (np > 0) {
                const int per = kPanelSolveThreads / 32;
                launch_step(k_sn_solve<false>, dim3(nwide + (np - nwide + per - 1) / per, gy), kPanelSolveThreads, st, d, vec, B, sym.pstep[l], nwide, np, v.state);
                ++count;
            }
            const KktStepRange rg = {sym.bs_beg[l], sym.bs_end[l], sym.bmstep[l], sym.bmstep[l + 1]};
            const int multi = rg.m1 - rg.m0, items = rg.s1 - rg.s0 + multi;
            if (items > 0) {
                launch_step(B > 1 ? k_ldl_bwd<true> : k_ldl_bwd<false>, level_grid(items, multi), kThreads, st, d, vec, B, v.state, rg);
                ++count;
            }
        }
    }
    // the level sequences never change for a handle: captured once, replayed every Newton step
    template <class F>
    int capture(cudaStream_t st, cudaGraphExec_t *exec, int64_t &count, F body) {
        if (*exec) return ASM_OK;
        cudaGraph_t graph = nullptr;
        count = 0;
        ASM_CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        body(count);
        ASM_CK(cudaStreamEndCapture(st, &graph));
        ASM_CK(cudaGraphInstantiate(exec, graph, 0));
        ASM_CK(cudaGraphDestroy(graph));
        return ASM_OK;
    }
};

}  // namespace asmb
