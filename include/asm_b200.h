/*
 * asm_b200.h — C ABI of the B200-native sub-LP engine for sequential linear programming.
 *
 * This is the drop-in boundary for the hot path of exanauts/ActiveSetMethods (reference tree
 * /root/reference, all citations relative to it).  The reference reaches its LP solver through the
 * `"external_optimizer"` MathOptInterface hook (src/parameters.jl:7, instantiated at
 * src/algorithms/slp.jl:32) and pushes / reads the sub-LP one scalar at a time
 * (src/algorithms/subproblem.jl:51-215, :229-542).  A Julia MOI shim binds the functions below with
 * `ccall` (see INTEGRATION.md); Python/ctypes binds them for the tests.
 *
 * Conventions
 *   - plain pointers and sizes only; all arrays are caller-owned host memory unless a name says `dev`;
 *   - every function returns 0 on success or a negative ASM_E_* code; no C++ exception crosses the ABI;
 *     `asm_last_error()` returns a thread-local message for the last failure;
 *   - +-infinity bounds are IEEE infinities;
 *   - batch: a handle created with `batch = B` holds B independent LPs that share one sparsity pattern.
 *     Host arrays of a batch are laid out scenario-major, `a[s * len + i]` (B contiguous vectors);
 *   - one CUDA stream and one host thread per handle; calls on a handle block until the result is in
 *     host memory unless stated otherwise.
 *
 * There is no CPU fallback: every entry point that computes fails with ASM_E_CUDA when no sm_100-class
 * device is available.
 */
#ifndef ASM_B200_H
#define ASM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes ------------------------------------------------------------------------------------ */
#define ASM_OK 0
#define ASM_E_INVALID (-1)  /* bad argument (null pointer, negative size, index out of range)            */
#define ASM_E_CUDA (-2)     /* CUDA runtime error / no device                                            */
#define ASM_E_FREE_ROW (-3) /* a row with both bounds infinite: the reference builder pushes no row for  */
                            /* it and breaks (subproblem.jl:143-197), so it is rejected here             */
#define ASM_E_STATE (-4)    /* call out of order (e.g. solve before update)                              */

/* ---- LP termination status (the subset of MOI.TerminationStatus the reference branches on,
 *      subproblem.jl:491-539) ------------------------------------------------------------------------- */
#define ASM_LP_OPTIMAL 0
#define ASM_LP_INFEASIBLE 1
#define ASM_LP_DUAL_INFEASIBLE 2
#define ASM_LP_ITERATION_LIMIT 3
#define ASM_LP_NUMERICAL_ERROR 4
#define ASM_LP_SKIPPED 5 /* the scenario was masked out of this solve (asm_slp_set_active) */

const char *asm_last_error(void);
/* number of visible CUDA devices (0 if none); never fails */
int asm_device_count(void);
const char *asm_version(void);

/* ---- solver parameters ------------------------------------------------------------------------------- */
typedef struct asm_lp_params {
    double eps_rel;        /* relative KKT tolerance: primal residual, dual residual and gap (default 1e-8) */
    double eps_infeas;     /* Farkas-certificate tolerance (default 1e-9)                                   */
    int64_t max_iter;      /* PDHG iteration limit per LP (default 2 000 000)                               */
    int32_t check_every;   /* KKT / restart evaluation period in iterations (default 64)                   */
    int32_t ruiz_iters;    /* Ruiz equilibration passes before Pock-Chambolle (default 10)                 */
    int32_t warm_start;    /* start from the previous solve of this handle: 1 = (x, y), 2 = y only; 0 = cold */
    int32_t verbose;       /* 1: print one line per restart check of scenario 0 to stderr                  */
    double restart_sufficient; /* 0.2  */
    double restart_necessary;  /* 0.8  */
    double restart_artificial; /* 0.36 */
    double pid_kp, pid_ki, pid_kd; /* primal-weight controller on log(w |dx|/|dy|); (0.5, 0, 0) = PDLP rule  */
    int32_t engine;        /* 0 auto (the barrier engine; PDHG hybrid if the pattern is refused);            */
                           /* 1 PDHG streaming kernels (one launch per half iteration, CUDA graph);          */
                           /* 2 PDHG persistent group kernel (LP resident in the shared memory of G blocks)  */
                           /* 4 barrier method: Mehrotra predictor-corrector on a fixed-pattern L D L'       */
                           /* 5 PDHG hybrid: stream, compact, hand the stragglers to the group kernel        */
    int32_t group_size;    /* blocks per LP for engine 2 (0 = auto)                                          */
    double hand_over;      /* engine 0 on a batch: fraction of the batch still running at which the          */
                           /* streaming kernels hand the stragglers to the group kernel (default 0.5)        */
    double weight_balance; /* > 0: at restarts move the primal weight by (relative primal residual / relative dual  */
                           /* residual)^weight_balance instead of the PDLP rule (0 = PDLP rule, the default)          */
    double tiny_rel;       /* rows / columns whose largest coefficient is below tiny_rel * max|K| are treated as     */
                           /* empty by the equilibration (0 = default 1e-8)                                            */
    /* barrier engine (engine 0 / 4) */
    int32_t ipm_max_iter;  /* Newton steps per LP (default 200)                                                        */
    int32_t ipm_refine;    /* iterative-refinement passes per linear solve to start with (default 0: the barrier       */
                           /* method tolerates the 1e-8 regularisation error); one more, at most two more, when LPs    */
                           /* sit between the acceptable and the target tolerance                                      */
    double ipm_reg;        /* static regularisation d of the quasi-definite system (default 1e-8, scaled units)        */
    double ipm_prox;       /* least-norm selection: proximal weight q = ipm_prox (1 + |c|) / (2 max(1, |x|)), i.e. the */
                           /* relative dual residual it may leave in the LP (default 1e-7; 0 = pure LP)                */
} asm_lp_params;
void asm_lp_default_params(asm_lp_params *p);

/* per-LP solve report (arrays of length batch) */
typedef struct asm_lp_info {
    int32_t status;     /* ASM_LP_*                                  */
    int32_t restarts;
    int64_t iterations;
    double objective;   /* c'x + c0 at the returned point            */
    double dual_objective;
    double primal_residual; /* ||Kx - proj(Kx)||_2, unscaled         */
    double dual_residual;   /* ||c - K'y - r||_2, unscaled           */
    double gap;             /* |pobj - dobj|                         */
} asm_lp_info;

/* =======================================================================================================
 * 1. Generic LP handle:   min c'x + c0   s.t.  rl <= K x <= ru,  lb <= x <= ub.
 *    What a GLPK-replacing MOI optimizer needs (the MOI calls listed in SURVEY.md App. B,
 *    subproblem.jl:54-213 build, :252-483 update, :490 solve, :491-520 read-back).
 * ===================================================================================================== */
typedef struct asm_lp asm_lp;

/* pattern is 0-based CSR, uploaded once (MOI add_variables/add_constraint, subproblem.jl:75-213) */
int asm_lp_create(int32_t n_cols, int32_t n_rows, int64_t nnz, const int64_t *row_ptr, const int32_t *col_idx,
                  int32_t batch, int32_t device, asm_lp **out);
void asm_lp_destroy(asm_lp *h);
/* MOI.modify(row, ScalarCoefficientChange) for the whole pattern (subproblem.jl:438-457); vals[batch][nnz] */
int asm_lp_set_matrix_values(asm_lp *h, const double *vals);
/* MOI.modify(ObjectiveFunction, ...) (subproblem.jl:252-272, :385-405); c[batch][n_cols], c0[batch] */
int asm_lp_set_objective(asm_lp *h, const double *c, const double *c0);
/* MOI.set(ConstraintSet, bound ci) (subproblem.jl:427-434) */
int asm_lp_set_col_bounds(asm_lp *h, const double *lb, const double *ub);
/* MOI.set(ConstraintSet, row ci) (subproblem.jl:461-484) */
int asm_lp_set_row_bounds(asm_lp *h, const double *rl, const double *ru);
/* MOI.optimize! (subproblem.jl:490); info[batch] */
int asm_lp_solve(asm_lp *h, const asm_lp_params *params, asm_lp_info *info);
/* MOI.get(VariablePrimal) (subproblem.jl:502-505); x[batch][n_cols] */
int asm_lp_get_primal(asm_lp *h, double *x);
/* MOI.get(ConstraintDual) on rows (subproblem.jl:510-515): >=0 lower side active, <=0 upper side */
int asm_lp_get_row_dual(asm_lp *h, double *y);
/* MOI.get(ConstraintDual) on the two bound constraints of every column (subproblem.jl:519-520):
 * dual_lb >= 0 (GreaterThan), dual_ub <= 0 (LessThan); either pointer may be NULL */
int asm_lp_get_col_dual(asm_lp *h, double *dual_lb, double *dual_ub);
/* warm start for the next solve (used when params.warm_start = 1); either pointer may be NULL */
int asm_lp_set_start(asm_lp *h, const double *x, const double *y);

/* ---- row-partitioned single LP (SURVEY.md 8(e): one very large instance over several GPUs) -----------------
 * One process per GPU.  Rank g passes the CSR pattern of its contiguous row block (all n_cols columns); the
 * setters above then take the local rows' values / row bounds and the replicated objective / column bounds;
 * asm_lp_solve is collective (one ncclAllReduce of the partial K'y per PDHG iteration); asm_lp_get_primal returns
 * the replicated x, asm_lp_get_row_dual the local rows' duals.  `id128` is a 128-byte NCCL unique id made by
 * rank 0 with asm_dist_unique_id and handed to the other ranks by the host (torch.distributed / MPI / files). */
int asm_dist_unique_id(char *id128);
int asm_lp_dist_create(int32_t n_cols, int32_t n_rows_local, int64_t nnz_local, const int64_t *row_ptr,
                       const int32_t *col_idx, int32_t rank, int32_t world, const char *id128, int32_t device,
                       asm_lp **out);

/* =======================================================================================================
 * 2. SLP fast path: the whole per-iteration sub-LP of the reference in three calls.
 *    Replaces compute_jacobian_matrix (common.jl:12-20), LpData (slp.jl:8-21), create_model!
 *    (subproblem.jl:51-215) and sub_optimize! (subproblem.jl:229-542).
 * ===================================================================================================== */
typedef struct asm_slp asm_slp;

/* Model (model.jl:1-61) + create_model!: bounds, and the COO Jacobian pattern j_str as 1-based
 * (row, col) pairs with duplicates allowed (model.jl:10).  The pattern is analysed and uploaded once.
 * x_L/x_U [n], g_L/g_U [m] are shared by all `batch` scenarios unless `per_scenario_bounds` != 0, in
 * which case they are [batch][n] / [batch][m]. */
int asm_slp_create(int32_t n, int32_t m, int64_t nnz_coo, const int64_t *j_row, const int64_t *j_col,
                   const double *x_L, const double *x_U, const double *g_L, const double *g_U, int32_t batch,
                   int32_t per_scenario_bounds, int32_t device, asm_slp **out);
void asm_slp_destroy(asm_slp *h);

/* sizes of the assembled (deduplicated) Jacobian and of the LP in reference form
 * (subproblem.jl:75-112: n + slacks columns; m + |adj| rows) */
int asm_slp_sizes(asm_slp *h, int64_t *nnz_csr, int32_t *lp_cols, int32_t *lp_rows);
/* the CSR pattern and, after an update, the values of the assembled Jacobian of scenario `s`
 * (bit-exact restatement of common.jl:12-20; duplicates summed in j_str order from 0.0).
 * row_ptr[m+1], col_idx[nnz_csr] 0-based, vals[nnz_csr]; any pointer may be NULL */
int asm_slp_get_csr(asm_slp *h, int32_t s, int64_t *row_ptr, int32_t *col_idx, double *vals);
/* the sub-LP of the last update as the engine holds it, for scenario s.  Normal phase: n columns, m rows (range rows
 * two-sided), the Jacobian CSR; restoration: the reference layout of asm_slp_sizes (n + slacks, m + |adj|).
 * cols, rows, nnz, row_ptr[rows+1], col_idx[nnz], vals[nnz], c[cols], c0, lb/ub[cols], rl/ru[rows];
 * after a solve also the LP's own solution, before the read-back of subproblem.jl:500-536:
 * x[cols], y[rows], dual_lb/dual_ub[cols] and the raw status of the scenario's solve (-1: still running when the
 * solve stopped).  Any pointer may be NULL.  ASM_E_STATE before an update, and for the solution outputs before a
 * solve; the handle's state is left as it is (no solve, no read-back). */
int asm_slp_get_lp(asm_slp *h, int32_t s, int32_t *cols, int32_t *rows, int64_t *nnz, int64_t *row_ptr,
                   int32_t *col_idx, double *vals, double *c, double *c0, double *lb, double *ub, double *rl,
                   double *ru, double *x, double *y, double *dual_lb, double *dual_ub, int32_t *status);

/* eval_functions! hand-over (slp.jl:186-191) + the data push of sub_optimize! (subproblem.jl:248-484):
 * x_k[batch][n], f[batch], df[batch][n], E[batch][m], dE[batch][nnz_coo] (j_str order), delta[batch],
 * feasibility (shared flag: 0 normal phase, 1 feasibility restoration).
 * Host -> device: straight from the caller's arrays when they are pinned (cudaHostRegister / cudaHostAlloc), else
 * through the handle's own ring of two pinned 8 MB chunks (memcpy overlapping the DMA); then the CSR is assembled and
 * the column / row / slack bounds are built on the device. */
int asm_slp_update(asm_slp *h, const double *x_k, const double *f, const double *df, const double *E,
                   const double *dE, const double *delta, int32_t feasibility);
/* MOI.optimize! on the current sub-LP (subproblem.jl:490); device-resident, no host copies except the
 * convergence flags.  info[batch] may be NULL. */
int asm_slp_solve(asm_slp *h, const asm_lp_params *params, asm_lp_info *info);
/* read-back of subproblem.jl:491-541: p[batch][n] (Xsol), lambda[batch][m] (row duals, range rows
 * summed), mult_x_U/mult_x_L[batch][n] (bound duals masked to the original bounds, :522-529),
 * p_slack[batch][m][2] (second entry 0 for one-slack rows; all 0 in the normal phase), status[batch].
 * INFEASIBLE => zeros (:532-536).  Any output pointer may be NULL. */
int asm_slp_extract(asm_slp *h, double *p, double *lambda, double *mult_x_U, double *mult_x_L,
                    double *p_slack, int32_t *status);
/* update + solve + extract in one call: the reference's sub_optimize!(slp, delta) (slp.jl:23-47) */
int asm_slp_sub_optimize(asm_slp *h, const double *x_k, const double *f, const double *df, const double *E,
                         const double *dE, const double *delta, int32_t feasibility,
                         const asm_lp_params *params, double *p, double *lambda, double *mult_x_U,
                         double *mult_x_L, double *p_slack, int32_t *status, asm_lp_info *info);

/* ---- merit / KKT reductions on the device (they use x_k, df, E, J of the last asm_slp_update and the
 *      multipliers / step of the last solve unless host arrays are given) ------------------------------ */
/* norm_violations (common.jl:75-98): p_norm = 0 -> infinity norm, 1 -> 1-norm, 2 -> 2-norm.
 * E[batch][m], x[batch][n] host arrays; out[batch] */
int asm_slp_norm_violations(asm_slp *h, const double *E, const double *x, int32_t p_norm, double *out);
/* KT_residuals (common.jl:35-44) with the Jacobian of the last update: df, lambda, mult_x_U, mult_x_L */
int asm_slp_kt_residuals(asm_slp *h, const double *df, const double *lambda, const double *mult_x_U,
                         const double *mult_x_L, double *out);
/* norm_complementarity (common.jl:51-68), infinity norm */
int asm_slp_norm_complementarity(asm_slp *h, const double *E, const double *lambda, double *out);
/* row 2-norms of the assembled Jacobian (used by compute_nu!, slp.jl:54-66, and KT_residuals) */
int asm_slp_row_norms(asm_slp *h, double *out /* [batch][m] */);
/* compute_phi (slp.jl:79-115) constraint part: sum_i nu_i * viol_i(E_trial) in the normal phase;
 * in feasibility restoration the shifted form of :84-103 with the slacks of the last extract.
 * base[batch] is f(x + alpha p) (normal) or prim_infeas (restoration); E_trial is g(x + alpha p) */
int asm_slp_merit_phi(asm_slp *h, const double *base, const double *E_trial, const double *nu,
                      const double *alpha, int32_t feasibility, double *out);
/* compute_derivative (slp.jl:122-147) with the df, E of the last update and the p / slacks of the last solve */
int asm_slp_merit_derivative(asm_slp *h, const double *nu, int32_t feasibility, double *out);

/* ---- device-side ACOPF evaluator (SURVEY.md 8(f)-1) ------------------------------------------------------
 * The role of the NLPEvaluator callbacks (src/MOI_wrapper.jl:1047-1069) and of eval_functions!
 * (src/algorithms/slp.jl:186-191) for the ACP-polar OPF in the variable / row / Jacobian layout of
 * activesetmethods_b200/examples/acopf.py: variables va[nb] vm[nb] pg[ng] qg[ng] p[2nl] q[2nl] pdc[2nd] qdc[2nd];
 * rows angmax[nl] angmin[nl] ref dc[nd] thermal[2nl] balance[2nb] ohm[4nl]; j_str in the same block order.
 * All scenarios of a batch share the network (loads only enter the row bounds). */
typedef struct asm_acopf_desc {
    int32_t nb, ng, nl, nd, ref_bus;
    const int32_t *f_bus, *t_bus;         /* [nl] 0-based bus indices                                              */
    const double *coef;                   /* [12][nl]: a, b, c of p_fr, q_fr, p_to, q_to (acopf.py `_cf` order)     */
    const double *gs, *bs;                /* [nb] shunts                                                           */
    const double *cost2, *cost1, *cost0;  /* [ng]                                                                  */
    const double *dc_loss1;               /* [nd] (may be NULL when nd = 0)                                        */
    const int32_t *bal_ptr;               /* [2nb + 1] CSR over the balance rows of their entries in j_str order   */
    const int32_t *bal_col;               /* [bal_ptr[2nb]] 0-based columns                                        */
    const double *bal_coef;               /* constant coefficients, NaN at the vm^2 (shunt) slots                  */
} asm_acopf_desc;
int asm_slp_attach_acopf(asm_slp *h, const asm_acopf_desc *d);
/* eval_functions! on the device at x[batch][n], then the device part of asm_slp_update */
int asm_slp_eval_acopf(asm_slp *h, const double *x, const double *delta, int32_t feasibility);
/* f[batch], df[batch][n], E[batch][m], dE[batch][nnz_coo] of the last evaluation; any pointer may be NULL */
int asm_slp_get_eval(asm_slp *h, double *f, double *df, double *E, double *dE);
/* compute_phi(x + alpha p) (slp.jl:79-115; the backtracking of slp_line_search.jl:228-241) with f and g evaluated on
 * the device at the trial point; `base` (prim_infeas) is read in feasibility restoration only */
int asm_slp_acopf_trial(asm_slp *h, const double *alpha, const double *nu, const double *base, int32_t feasibility,
                        double *out);

/* ---- instrumentation --------------------------------------------------------------------------------- */
/* kernels launched by this handle's solver since creation (all of them this library's own) */
int64_t asm_slp_launch_count(asm_slp *h);
/* device time (ms, CUDA events on the handle's stream) of the PDHG loop of the last asm_slp_solve and
 * the total PDHG iterations it ran (max over the batch) */
int asm_slp_last_solve_timing(asm_slp *h, double *loop_ms, int64_t *iterations);

/* host-only self-check of the group engine's data layout for groups of G blocks (no device needed): rebuilds
 * every row of the pattern from the sliced-ELL / halo arrays; returns the dynamic shared memory one block needs,
 * whether the matrix values stay resident there, and the padded entry count of the row side */
int asm_plan_check(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx, int32_t G,
                   int64_t *smem_bytes, int32_t *matrix_resident, int64_t *padded_entries);
/* barrier engine (engine 0 / 4) instrumentation.  stats[14]: KKT dimension, nnz(L), update terms outside the supernode
 * panels, steps of the schedule (levels of the elimination tree when supernodes are off), factor chunks,
 * forward-substitution chunks, kernel launches per factorisation, per substitution pair, factorisations and substitution
 * pairs of the last solve, distinct f64 operands read / targets updated per factorisation and per substitution pair
 * (summed over the levels: the compulsory HBM traffic of a batch larger than L2, DESIGN.md 4.4); times[4]: symbolic analysis
 * ms, Newton steps of the last solve, factor / solve ms of the traced step (ASM_TRACE=1).  Either pointer may be NULL.
 * Environment switches read when a handle builds its engine: ASM_IPM_SUPERNODE = widest supernode (default 16, 1 = one
 * column per level), ASM_NO_PDL = plain stream-ordered launches */
int asm_slp_ipm_info(asm_slp *h, int64_t *stats, double *times);
/* average device time (CUDA events on the handle's stream) of one numeric factorisation and one substitution pair of
 * the whole batch, `reps` launches each, on the data of the last solve */
int asm_slp_ipm_timing(asm_slp *h, int32_t reps, double *factor_ms, double *solve_ms);
/* host-only self test of the barrier engine's symbolic analysis (no device needed): factorises
 * [-diag(dx) K'; K diag(ew)] and solves one right-hand side on the host with the lists and the summation order of the
 * device kernels (supernodes as a handle would use them).  rhs_sol[n_cols + n_rows]: right-hand side in, solution out.
 * stats[8]: nnz(L), terms, steps, steps with fan-out items in the factorisation / forward / backward substitution (the
 * step-kernel launches of each), longest chunk, chunks */
int asm_kkt_selftest(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx, const double *vals,
                     const double *dx, const double *ew, double *rhs_sol, int64_t *stats);
/* device self test of the barrier engine's numeric kernels: factorises, for each of `batch` scenarios sharing the
 * m x n CSR pattern, [-diag(dx_s) K_s'; K_s diag(ew_s)] with the engine's captured factor graph and solves
 * rhs_sol[s] with its captured substitution graph.  vals[batch][nnz], dx[batch][n_cols], ew[batch][n_rows],
 * rhs_sol[batch][n_cols + n_rows] (node order: columns then rows; right-hand side in, solution out).
 * active[batch] (NULL = all): masked scenarios are not live and their rhs_sol comes back unchanged.
 * inv_pivots[batch][n_cols + n_rows] (may be NULL): 1/d of every node after the factorisation.
 * stats[10] (may be NULL): nnz(L), steps, narrow panels (2 <= w <= 4), wide panels (w > 4), narrow row tasks that
 * start below the first row (r0 > 0), wide panels with more than one row task, longest factor chunk, step launches
 * whose grid-stride loops take a second pass (capped grid), launches per factorisation, per substitution pair.
 * Reads ASM_IPM_SUPERNODE and ASM_NO_PDL like a handle.  ASM_E_CUDA without a device: there is no host fallback */
int asm_kkt_device_selftest(int32_t n_cols, int32_t n_rows, const int64_t *row_ptr, const int32_t *col_idx,
                            int32_t batch, const double *vals, const double *dx, const double *ew,
                            const int32_t *active, double *rhs_sol, double *inv_pivots, int32_t device,
                            int64_t *stats);

/* Restrict the following solves of a batch to the scenarios with active[s] != 0 (active[batch]; NULL = all again).
 * A lock-step batch of SLP runs calls this every round: scenarios that have terminated, or that are in the other
 * phase, cost nothing and come back with status ASM_LP_SKIPPED and zeroed outputs. */
int asm_slp_set_active(asm_slp *h, const int32_t *active);

/* which engine the last asm_slp_solve used (1 streaming, 2 group, 3 both, 4 barrier), blocks per LP and LPs resident at once */
int asm_slp_engine_info(asm_slp *h, int32_t *engine, int32_t *group_size, int32_t *groups);

/* ---- device-resident variants (bench.py's `value`: inputs already in HBM) ----------------------------- */
/* the device part of asm_slp_update (assembly + bounds, subproblem.jl:248-484) on the x_k, df, E, dE, delta
 * already resident from the last asm_slp_update */
int asm_slp_reassemble(asm_slp *h, int32_t feasibility);
/* the device part of asm_slp_extract (masking / range-row sums of subproblem.jl:500-536), no copy to the host */
int asm_slp_extract_device(asm_slp *h);
/* CUDA-event timer on the handle's own stream: start records an event, stop records another, waits for it
 * and returns the elapsed device time */
int asm_slp_timer_start(asm_slp *h);
int asm_slp_timer_stop(asm_slp *h, double *ms);
/* average duration (ms) of one launch of the two streaming PDHG kernels (A'y + primal update, A xbar + dual
 * update) over `reps` back-to-back launches each, CUDA events on the handle's stream.  Needs a solved LP;
 * the iterate is advanced (benchmark use only) */
int asm_slp_kernel_timing(asm_slp *h, int32_t reps, double *primal_ms, double *dual_ms);

#ifdef __cplusplus
}
#endif
#endif /* ASM_B200_H */
