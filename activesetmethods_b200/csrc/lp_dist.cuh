// Row-partitioned single LP across GPUs (SURVEY.md 8(e), BASELINE.json config 4): rank g owns a contiguous block
// of rows of K with its duals y_g and row bounds; x, c and the column bounds are replicated.  K_g xbar is local;
// K_g' y_g is a partial column vector that one ncclAllReduce(sum, f64, n) per PDHG iteration completes, after
// which every rank applies the identical primal update.  The column norms of the preconditioner and the row-side
// KKT / restart sums travel the same way.  NCCL returns bit-identical sums on every rank, so all ranks take the
// same restart / termination decisions without further agreement.
//
// NCCL is bound at run time (dlopen of libnccl.so.2 -- the copy torch already loaded when there is one), so the
// library has no link-time dependency on it and single-GPU users never touch it.
#pragma once
#include <dlfcn.h>

#include "lp_solver.cuh"

namespace asmb {

// ---- minimal NCCL binding -----------------------------------------------------------------------------------
struct NcclApi {
    typedef struct {
        char internal[128];
    } UniqueId;
    typedef void *Comm;
    int (*GetUniqueId)(UniqueId *) = nullptr;
    int (*CommInitRank)(Comm *, int, UniqueId, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    void *lib = nullptr;
    static constexpr int kDouble = 8, kSum = 0, kMax = 2;  // ncclDouble, ncclSum, ncclMax (nccl.h)
    int load() {
        if (lib) return ASM_OK;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return fail(ASM_E_CUDA, std::string("cannot load NCCL: ") + dlerror());
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy || !GetErrorString)
            return fail(ASM_E_CUDA, "libnccl lacks a required symbol");
        return ASM_OK;
    }
};
inline NcclApi &nccl() {
    static NcclApi api;
    return api;
}
#define ASM_NCCL(call)                                                                           \
    do {                                                                                         \
        int r__ = (call);                                                                        \
        if (r__ != 0) {                                                                          \
            char b__[512];                                                                       \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, nccl().GetErrorString(r__)); \
            return ::asmb::fail(ASM_E_CUDA, b__);                                                \
        }                                                                                        \
    } while (0)

// ---- kernels of the partitioned iteration (single LP: B = 1) ----------------------------------------------------
// column norms of the local row block (max or sum of |dr_i K_ij dc_j|), completed by an all-reduce
// out[j] = scaled norm, out[n + j] = max |K_ij| of the original column (local rows)
template <bool SUM>
__global__ void __launch_bounds__(kThreads) k_col_norm_partial(LpView v, double *__restrict__ out) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < v.n; j += (int64_t)gridDim.x * blockDim.x) {
        const double dcj = v.dc[j];
        double a = 0.0, a0 = 0.0;
        for (int k = v.col_ptr[j]; k < v.col_ptr[j + 1]; ++k) {
            const double val = v.vals[v.csc_src[k]];
            const double t = fabs(val * v.dr[v.row_idx[k]] * dcj);
            a = SUM ? a + t : fmax(a, t);
            a0 = fmax(a0, fabs(val));
        }
        out[j] = a;
        out[v.n + j] = a0;
    }
}
// column scale factor from the completed norms; numerically empty columns keep scale 1 (see kTinyRel)
__global__ void k_inv_sqrt(const double *__restrict__ a, const double *__restrict__ a0, const double *__restrict__ gmax,
                           double *__restrict__ out, int64_t n) {
    const double tiny = kTinyRel * gmax[0];
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
        out[t] = (a[t] > 0.0 && a0[t] > tiny) ? 1.0 / sqrt(a[t]) : 1.0;
}
// t = K_g' w  (partial over the local rows); w is y, yp or the ray
__global__ void __launch_bounds__(kThreads) k_aty(LpView v, const double *__restrict__ w, double *__restrict__ t) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < v.n; j += (int64_t)gridDim.x * blockDim.x)
        t[j] = spmv_row(v.AT, v.row_idx, w, v.col_ptr[j], v.col_ptr[j + 1], 1, 0);
}
// primal half with the completed K'y in `aty`
template <bool CHECK>
__global__ void __launch_bounds__(kThreads) k_primal_t(LpView v, const double *__restrict__ aty, int jit) {
    const ScenState *st = v.state;
    const double tau = st->eta / st->omega;
    const double w = pdhg_halpern_weight(st->k0 + jit + 1);
    double acc[3] = {0.0, 0.0, 0.0};
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < v.n; j += (int64_t)gridDim.x * blockDim.x) {
        const double cj = v.cs[j], g = cj - aty[j], xv = v.x[j];
        const double xpv = pdhg_primal_step(xv, g, tau, v.lbs[j], v.ubs[j]);
        const double xb = pdhg_reflect(xpv, xv);
        v.xbar[j] = xb;
        if (CHECK) {
            v.xp[j] = xpv;
            pdhg_col_terms(xpv, xv, v.xa[j], cj, acc[0], acc[1], acc[2]);
        } else {
            v.x[j] = pdhg_halpern(w, xb, v.xa[j]);
        }
    }
    if (CHECK) block_reduce_store<false, 3>(acc, 0u, v.partials, Q_DX2, 1);
}
// reduced costs from the completed K'yp
__global__ void __launch_bounds__(kThreads) k_dual_resid_t(LpView v, const double *__restrict__ atyp) {
    const double inv_sc = 1.0 / v.state->sc;
    double acc[2] = {0.0, 0.0};
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < v.n; j += (int64_t)gridDim.x * blockDim.x) {
        const double rc = v.cs[j] - atyp[j];
        v.gyp[j] = rc;
        pdhg_rc_terms(rc, v.xp[j], v.lbs[j], v.ubs[j], inv_sc, v.dc[j], acc[0], acc[1]);
    }
    block_reduce_store<false, 2>(acc, 0u, v.partials, Q_DRES2, 1);
}
__global__ void __launch_bounds__(kThreads) k_ray_cols_t(LpView v, const double *__restrict__ atr) {
    double acc[2] = {0.0, 0.0};
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < v.n; j += (int64_t)gridDim.x * blockDim.x)
        pdhg_ray_col_terms(atr[j], v.lbs[j], v.ubs[j], v.dc[j], acc[0], acc[1]);
    block_reduce_store<false, 2>(acc, 2u, v.partials, Q_RAY_COL, 1);
}
// second stage of the check reductions into qsum[Q_COUNT] / qmax[2]; column-side sums are replicated on every
// rank, so only rank 0 contributes them to the all-reduce
__global__ void __launch_bounds__(kFinalThreads) k_reduce_q(LpView v, int rank, double *qsum, double *qmax) {
    for (int i = 0; i < Q_COUNT; ++i) {
        const bool rows = (kQRows >> i) & 1u, is_max = (kQMax >> i) & 1u;
        const double q = final_reduce(v.partials, i, rows ? v.nbx_rows : v.nbx_cols, 1, 0, is_max);
        if (threadIdx.x == 0) {
            if (is_max) {
                qmax[i == Q_RAY_MAX ? 0 : 1] = q;
                qsum[i] = 0.0;
            } else {
                qsum[i] = (rows || rank == 0) ? q : 0.0;
            }
        }
    }
}
__global__ void k_merge_q(double *qsum, const double *qmax) {
    qsum[Q_RAY_MAX] = qmax[0];
    qsum[Q_KTY_MAX] = qmax[1];
}
// the check decision on the completed sums (single LP)
__global__ void k_decide_q(LpView v, const double *q, int jit, int steps) {
    ScenState st = *v.state;
    if (st.status >= 0) return;
    pdhg_decide(st, *v.prm, q, jit, steps, "pdhg-rows");
    *v.state = st;
}
// norms for k_start_q: psum = {c2, cun2 (replicated), q2, qun2 (local)}
__global__ void __launch_bounds__(kFinalThreads) k_reduce_prep(LpView v, int rank, double *psum) {
    const double c2 = final_reduce(v.partials, P_C2, v.nbx_cols, 1, 0, false);
    const double cun2 = final_reduce(v.partials, P_CUN2, v.nbx_cols, 1, 0, false);
    const double q2 = final_reduce(v.partials, P_Q2, v.nbx_rows, 1, 0, false);
    const double qun2 = final_reduce(v.partials, P_QUN2, v.nbx_rows, 1, 0, false);
    if (threadIdx.x == 0) {
        psum[0] = rank == 0 ? c2 : 0.0;
        psum[1] = rank == 0 ? cun2 : 0.0;
        psum[2] = q2;
        psum[3] = qun2;
    }
}
__global__ void k_start_q(LpView v, const double *psum) { *v.state = pdhg_start(psum[0], psum[1], psum[2], psum[3]); }

// ---- host ------------------------------------------------------------------------------------------------------
class DistLp {
   public:
    LpSolver lp;  // local row block: n columns, m_local rows
    int rank = 0, world = 1, device = 0;
    NcclApi::Comm comm = nullptr;
    DBuf<double> t_part, t_full, a0_full, qsum, qmax, psum;
    int64_t allreduces = 0;

    ~DistLp() {
        if (comm) nccl().CommDestroy(comm);
    }

    int init(int n, int m_local, int64_t nnz_local, const int64_t *rp, const int32_t *ci, int rank_, int world_,
             const char *unique_id, int dev) {
        rank = rank_;
        world = world_;
        device = dev;
        if (world < 1 || rank < 0 || rank >= world || !unique_id) return fail(ASM_E_INVALID, "bad rank / world / id");
        ASM_TRY(nccl().load());
        ASM_CK(cudaSetDevice(dev));
        ASM_TRY(lp.init(n, m_local, nnz_local, rp, ci, 1, nullptr));
        NcclApi::UniqueId id;
        memcpy(id.internal, unique_id, sizeof id.internal);
        ASM_NCCL(nccl().CommInitRank(&comm, world, id, rank));
        ASM_TRY(t_part.alloc(2 * (size_t)n));
        ASM_TRY(t_full.alloc(2 * (size_t)n));
        ASM_TRY(a0_full.alloc(n));
        ASM_TRY(qsum.alloc(Q_COUNT));
        ASM_TRY(qmax.alloc(2));
        ASM_TRY(psum.alloc(4));
        return ASM_OK;
    }

    int allreduce(const double *src, double *dst, size_t cnt, int op) {
        ASM_NCCL(nccl().AllReduce(src, dst, cnt, NcclApi::kDouble, op, comm, lp.stream));
        ++allreduces;
        return ASM_OK;
    }

    int precondition(int ruiz_iters, int warm) {
        LpSolver &L = lp;
        LpView v = L.view();
        cudaStream_t stream = L.stream;
        int64_t &launches = L.launches;
        const int n = L.n, m = L.m;
        const Geo gr = geo_for(m, 1), gc = geo_for(n, 1), gm = geo_for(std::max(n, m), 1);
        ASM_KL(k_fill<<<LpSolver::ew_grid(std::max(m, 1)), 1024, 0, stream>>>(L.dr.p, 1.0, m));
        ASM_KL(k_fill<<<LpSolver::ew_grid(n), 1024, 0, stream>>>(L.dc.p, 1.0, n));
        {   // largest coefficient of the whole matrix (all ranks) and of every column
            const Geo gz = geo_for(std::max<int64_t>(L.nnz, 1), 1);
            ASM_KL(k_absmax<false><<<gz.grid, gz.block, 0, stream>>>(v, L.nnz));
            ASM_KL(k_final_max<<<1, kFinalThreads, 0, stream>>>(L.partials.p, (int)gz.grid.x, 1, L.gmax.p, L.tiny_rel / kTinyRel));
            ASM_TRY(allreduce(L.gmax.p, L.gmax.p, 1, NcclApi::kMax));
            ASM_KL(k_col_norm_partial<false><<<gc.grid, gc.block, 0, stream>>>(v, t_part.p));
            ASM_TRY(allreduce(t_part.p + n, a0_full.p, n, NcclApi::kMax));
        }
        for (int it = 0; it <= ruiz_iters; ++it) {
            const bool pc = it == ruiz_iters;  // last pass: Pock-Chambolle (alpha = 1): 1-norms
            if (pc) {
                ASM_KL(k_ruiz_rows<false, true><<<gr.grid, gr.block, 0, stream>>>(v));
                ASM_KL(k_col_norm_partial<true><<<gc.grid, gc.block, 0, stream>>>(v, t_part.p));
            } else {
                ASM_KL(k_ruiz_rows<false, false><<<gr.grid, gr.block, 0, stream>>>(v));
                ASM_KL(k_col_norm_partial<false><<<gc.grid, gc.block, 0, stream>>>(v, t_part.p));
            }
            ASM_TRY(allreduce(t_part.p, t_full.p, n, pc ? NcclApi::kSum : NcclApi::kMax));
            ASM_KL(k_inv_sqrt<<<LpSolver::ew_grid(n), 1024, 0, stream>>>(t_full.p, a0_full.p, L.gmax.p, L.scf.p, n));
            if (m) ASM_KL(k_mul_inplace<<<LpSolver::ew_grid(m), 1024, 0, stream>>>(L.dr.p, L.sr.p, m));
            ASM_KL(k_mul_inplace<<<LpSolver::ew_grid(n), 1024, 0, stream>>>(L.dc.p, L.scf.p, n));
        }
        ASM_KL(k_build_scaled_csr<false><<<gr.grid, gr.block, 0, stream>>>(v));
        ASM_KL(k_build_scaled_csc<false><<<gc.grid, gc.block, 0, stream>>>(v));
        ASM_TRY(L.partials.zero(stream));
        ASM_KL(k_prepare_cols<false><<<gc.grid, gc.block, 0, stream>>>(v));
        ASM_KL(k_prepare_rows<false><<<gr.grid, gr.block, 0, stream>>>(v));
        ASM_KL(k_reduce_prep<<<1, kFinalThreads, 0, stream>>>(v, rank, psum.p));
        ASM_TRY(allreduce(psum.p, psum.p, 4, NcclApi::kSum));
        ASM_KL(k_start_q<<<1, 1, 0, stream>>>(v, psum.p));
        ASM_KL(k_prepare_finish<false><<<gm.grid, gm.block, 0, stream>>>(v, warm, (const int *)(warm ? L.d_prev_ok.p : nullptr)));
        ASM_CK(cudaGetLastError());
        return ASM_OK;
    }

    // K' w over all ranks -> t_full
    int aty(const double *w) {
        LpView v = lp.view();
        const Geo gc = geo_for(lp.n, 1);
        k_aty<<<gc.grid, gc.block, 0, lp.stream>>>(v, w, t_part.p);
        ++lp.launches;
        return allreduce(t_part.p, t_full.p, lp.n, NcclApi::kSum);
    }

    int solve(const asm_lp_params &P, asm_lp_info *info) {
        LpSolver &L = lp;
        cudaStream_t stream = L.stream;
        int64_t &launches = L.launches;
        ASM_CK(cudaSetDevice(device));
        DevParams dp = dev_params(P);
        dp.verbose = P.verbose && rank == 0;
        ASM_CK(cudaMemcpyAsync(L.prm.p, &dp, sizeof dp, cudaMemcpyHostToDevice, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        L.tiny_rel = P.tiny_rel > 0.0 ? P.tiny_rel : kTinyRel;
        const int warm = (P.warm_start && L.has_solution) ? (int)P.warm_start : 0;
        if (warm) ASM_TRY(L.upload_start_ok());   // the single-GPU rule: every rank holds the same decision
        ASM_TRY(precondition(P.ruiz_iters, warm));
        const int steps = std::max(2, (int)P.check_every);
        LpView v = L.view();
        const int n = L.n, m = L.m;
        const Geo gr = geo_for(m, 1), gc = geo_for(n, 1), gm = geo_for(std::max(n, m), 1);
        ASM_CK(cudaEventRecord(L.ev0, stream));
        ScenState hs;
        int64_t it = 0;
        bool done = false;
        while (!done && it < P.max_iter) {
            for (int j = 0; j < steps; ++j) {
                const bool check = (j == 0 || j == steps - 1);
                ASM_TRY(aty(L.y.p));
                if (!check) {
                    ASM_KL(k_primal_t<false><<<gc.grid, gc.block, 0, stream>>>(v, t_full.p, j));
                    ASM_KL(k_dual<false, false><<<gr.grid, gr.block, 0, stream>>>(v, j));
                    continue;
                }
                ASM_TRY(L.partials.zero(stream));
                ASM_KL(k_primal_t<true><<<gc.grid, gc.block, 0, stream>>>(v, t_full.p, j));
                ASM_KL(k_dual<false, true><<<gr.grid, gr.block, 0, stream>>>(v, j));
                ASM_TRY(aty(L.yp.p));
                ASM_KL(k_dual_resid_t<<<gc.grid, gc.block, 0, stream>>>(v, t_full.p));
                ASM_KL(k_ray_rows<false><<<gr.grid, gr.block, 0, stream>>>(v));
                ASM_TRY(aty(L.ray.p));
                ASM_KL(k_ray_cols_t<<<gc.grid, gc.block, 0, stream>>>(v, t_full.p));
                ASM_KL(k_store_kstep<<<1, 32, 0, stream>>>(L.state.p, L.kstep.p, j, 1));
                ASM_KL(k_reduce_q<<<1, kFinalThreads, 0, stream>>>(v, rank, qsum.p, qmax.p));
                ASM_TRY(allreduce(qsum.p, qsum.p, Q_COUNT, NcclApi::kSum));
                ASM_TRY(allreduce(qmax.p, qmax.p, 2, NcclApi::kMax));
                ASM_KL(k_merge_q<<<1, 1, 0, stream>>>(qsum.p, qmax.p));
                ASM_KL(k_decide_q<<<1, 1, 0, stream>>>(v, qsum.p, j, steps));
                ASM_KL(k_apply<false><<<gm.grid, gm.block, 0, stream>>>(v, L.kstep.p));
                ASM_KL(k_after_apply<<<1, 32, 0, stream>>>(L.state.p, 1));
            }
            it += steps;
            ASM_CK(cudaMemcpyAsync(&hs, L.state.p, sizeof hs, cudaMemcpyDeviceToHost, stream));
            ASM_CK(cudaStreamSynchronize(stream));
            done = hs.status >= 0;
        }
        ASM_CK(cudaEventRecord(L.ev1, stream));
        ASM_KL(k_finalize<false><<<gm.grid, gm.block, 0, stream>>>(v));
        ASM_CK(cudaMemcpyAsync(&hs, L.state.p, sizeof hs, cudaMemcpyDeviceToHost, stream));
        double hc0 = 0.0;
        ASM_CK(cudaMemcpyAsync(&hc0, L.c0.p, sizeof(double), cudaMemcpyDeviceToHost, stream));
        ASM_CK(cudaStreamSynchronize(stream));
        float ms = 0.f;
        ASM_CK(cudaEventElapsedTime(&ms, L.ev0, L.ev1));
        L.last_loop_ms = ms;
        if (hs.status < 0) hs.status = ASM_LP_ITERATION_LIMIT;
        L.last_iters = hs.total;
        L.host_state[0] = hs;
        L.start_ok[0] = hs.status == ASM_LP_OPTIMAL;
        if (info) lp_info(hs, hc0, *info);
        L.has_solution = true;
        return ASM_OK;
    }
};

}  // namespace asmb
