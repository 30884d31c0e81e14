"""Host-side mirror of the reference's sub-problem objects, on top of the C ABI.

================================  ==========================================================================
here                              reference (relative to /root/reference)
================================  ==========================================================================
``SubLp``                         ``QpModel`` + ``create_model!`` + ``sub_optimize!``
                                  (``src/algorithms/subproblem.jl:16-542``), reached from
                                  ``sub_optimize!(slp, Δ)`` (``src/algorithms/slp.jl:23-47``)
``SubLp.jacobian_csr``            ``compute_jacobian_matrix`` (``src/algorithms/common.jl:12-20``)
``SubLp.norm_violations`` …       ``src/algorithms/common.jl:35-98``, ``src/algorithms/slp.jl:79-147``
``B200LP``                        the ``external_optimizer`` (GLPK.Optimizer in the reference's tests,
                                  ``test/runtests.jl:2``): a general LP solved by PDHG on the GPU
================================  ==========================================================================

All heavy lifting happens in ``libasm_b200.so`` (CUDA, sm_100a).  A handle holds ``batch`` independent
sub-LPs that share the Jacobian sparsity pattern; arrays of a batch are ``[batch, len]``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import LP_OPTIMAL, LP_INFEASIBLE, LP_DUAL_INFEASIBLE, LP_ITERATION_LIMIT, LP_NUMERICAL_ERROR  # noqa: F401

__all__ = ["SubLp", "B200LP", "B200RowPartitionedLP", "LP_OPTIMAL", "LP_INFEASIBLE", "LP_DUAL_INFEASIBLE", "LP_ITERATION_LIMIT",
           "LP_NUMERICAL_ERROR"]


def _info_to_dicts(info, batch):
    return [dict(status=int(i.status), restarts=int(i.restarts), iterations=int(i.iterations),
                 objective=float(i.objective), dual_objective=float(i.dual_objective),
                 primal_residual=float(i.primal_residual), dual_residual=float(i.dual_residual), gap=float(i.gap))
            for i in info[:batch]]


class SubLp:
    """The SLP sub-problem of a (batch of) NLP(s) with a fixed Jacobian pattern.

    Parameters mirror ``Model`` (``src/model.jl:33-60``): ``n, m``, bounds and ``j_str`` — an ``(nnz, 2)``
    array of **1-based** (row, col) pairs, duplicates allowed.  Bounds are ``[n]`` / ``[m]`` (shared by the
    batch) or ``[batch, n]`` / ``[batch, m]``."""

    def __init__(self, n, m, j_str, x_L, x_U, g_L, g_U, batch=1, device=0, **lp_params):
        self._lib = capi.load()
        self.n, self.m, self.batch = int(n), int(m), int(batch)
        j = np.ascontiguousarray(np.asarray(j_str, dtype=np.int64).reshape(-1, 2))
        self.nnz_coo = len(j)
        jr = np.ascontiguousarray(j[:, 0])
        jc = np.ascontiguousarray(j[:, 1])
        x_L, x_U = capi.as_f64(x_L), capi.as_f64(x_U)
        g_L, g_U = capi.as_f64(g_L), capi.as_f64(g_U)
        per = 1 if x_L.ndim == 2 else 0
        if per:
            assert x_L.shape == (batch, n) and x_U.shape == (batch, n)
            assert g_L.shape == (batch, m) and g_U.shape == (batch, m)
        self._h = C.c_void_p()
        capi.check(self._lib.asm_slp_create(
            self.n, self.m, self.nnz_coo, jr.ctypes.data_as(capi.c_int64_p), jc.ctypes.data_as(capi.c_int64_p),
            capi.dptr(x_L), capi.dptr(x_U), capi.dptr(g_L), capi.dptr(g_U), self.batch, per, int(device),
            C.byref(self._h)))
        nnz = C.c_int64()
        cols = C.c_int32()
        rows = C.c_int32()
        capi.check(self._lib.asm_slp_sizes(self._h, C.byref(nnz), C.byref(cols), C.byref(rows)))
        self.nnz_csr, self.lp_cols, self.lp_rows = nnz.value, cols.value, rows.value
        self.params = capi.default_params(**lp_params)
        self.last_info = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.asm_slp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers --------------------------------------------------------------------------------------------
    def _vec(self, a, length):
        return capi.as_f64(a, (self.batch, length)) if length else np.zeros((self.batch, 0))

    def _scal(self, a):
        a = np.asarray(a, dtype=np.float64)
        if a.ndim == 0:
            a = np.full(self.batch, float(a))
        return capi.as_f64(a, (self.batch,))

    def _out(self, a):
        return a[0] if self.batch == 1 and self._squeeze else a

    _squeeze = True

    # -- the hot path -----------------------------------------------------------------------------------------
    def update(self, x_k, f, df, E, dE, delta, feasibility=False):
        """``eval_functions!`` hand-over + the data push of ``sub_optimize!`` (subproblem.jl:248-484)."""
        capi.check(self._lib.asm_slp_update(
            self._h, capi.dptr(self._vec(x_k, self.n)), capi.dptr(self._scal(f)), capi.dptr(self._vec(df, self.n)),
            capi.dptr(self._vec(E, self.m)), capi.dptr(self._vec(dE, self.nnz_coo)), capi.dptr(self._scal(delta)),
            1 if feasibility else 0))

    def set_active(self, mask=None):
        """Restrict the following solves to the scenarios with ``mask[s]`` true (``None``: all again).  Masked
        scenarios come back with status ``LP_SKIPPED`` (5) and zeroed outputs."""
        if mask is None:
            capi.check(self._lib.asm_slp_set_active(self._h, None))
            return
        m = np.ascontiguousarray(np.asarray(mask).astype(bool), dtype=np.int32)
        assert m.shape == (self.batch,)
        capi.check(self._lib.asm_slp_set_active(self._h, m.ctypes.data_as(capi.c_int32_p)))

    def solve(self):
        info = (capi.LpInfo * self.batch)()
        capi.check(self._lib.asm_slp_solve(self._h, C.byref(self.params), info))
        self.last_info = _info_to_dicts(info, self.batch)
        return self.last_info

    def extract(self):
        B, n, m = self.batch, self.n, self.m
        p = np.empty((B, n)); lam = np.empty((B, m)); mu_u = np.empty((B, n)); mu_l = np.empty((B, n))
        slack = np.empty((B, m, 2)); status = np.empty(B, dtype=np.int32)
        capi.check(self._lib.asm_slp_extract(self._h, capi.dptr(p), capi.dptr(lam), capi.dptr(mu_u), capi.dptr(mu_l),
                                             capi.dptr(slack), status.ctypes.data_as(capi.c_int32_p)))
        return p, lam, mu_u, mu_l, slack, status

    def solve_extract(self):
        """``MOI.optimize!`` + read-back (subproblem.jl:490-541) on the data of the last ``update``."""
        self.solve()
        p, lam, mu_u, mu_l, slack, status = self.extract()
        if self.batch == 1:
            return p[0], lam[0], mu_u[0], mu_l[0], slack[0], int(status[0])
        return p, lam, mu_u, mu_l, slack, status

    def sub_optimize(self, x_k, f, df, E, dE, delta=1000.0, feasibility=False):
        """``sub_optimize!(slp, Δ)`` (slp.jl:23-47): returns ``(Xsol, lambda, mult_x_U, mult_x_L, p_slack,
        status)`` like subproblem.jl:541 — arrays are ``[batch, ...]`` (squeezed when ``batch == 1``);
        ``p_slack`` is ``[m, 2]`` with a zero second entry for one-slack rows."""
        B, n, m = self.batch, self.n, self.m
        p = np.empty((B, n)); lam = np.empty((B, m)); mu_u = np.empty((B, n)); mu_l = np.empty((B, n))
        slack = np.empty((B, m, 2)); status = np.empty(B, dtype=np.int32)
        info = (capi.LpInfo * B)()
        capi.check(self._lib.asm_slp_sub_optimize(
            self._h, capi.dptr(self._vec(x_k, n)), capi.dptr(self._scal(f)), capi.dptr(self._vec(df, n)),
            capi.dptr(self._vec(E, m)), capi.dptr(self._vec(dE, self.nnz_coo)), capi.dptr(self._scal(delta)),
            1 if feasibility else 0, C.byref(self.params), capi.dptr(p), capi.dptr(lam), capi.dptr(mu_u),
            capi.dptr(mu_l), capi.dptr(slack), status.ctypes.data_as(capi.c_int32_p), info))
        self.last_info = _info_to_dicts(info, B)
        if B == 1:
            return p[0], lam[0], mu_u[0], mu_l[0], slack[0], int(status[0])
        return p, lam, mu_u, mu_l, slack, status

    # -- Jacobian storage -------------------------------------------------------------------------------------
    def jacobian_csr(self, scenario=0):
        """(row_ptr, col_idx, vals) of the assembled Jacobian after the last ``update`` — the device result of
        ``compute_jacobian_matrix`` (common.jl:12-20)."""
        rp = np.empty(self.m + 1, dtype=np.int64)
        ci = np.empty(self.nnz_csr, dtype=np.int32)
        v = np.empty(self.nnz_csr)
        capi.check(self._lib.asm_slp_get_csr(self._h, int(scenario), rp.ctypes.data_as(capi.c_int64_p),
                                             ci.ctypes.data_as(capi.c_int32_p), capi.dptr(v)))
        return rp, ci, v

    # -- merit / KKT reductions (device) ----------------------------------------------------------------------
    def _ret(self, out):
        return float(out[0]) if self.batch == 1 else out

    def norm_violations(self, E=None, x=None, p=1):
        """common.jl:75-98; ``p`` in {1, 2, inf}.  ``None`` uses the E / x of the last update."""
        code = {1: 1, 2: 2, np.inf: 0, float("inf"): 0}[p]
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_norm_violations(
            self._h, capi.dptr(None if E is None else self._vec(E, self.m)),
            capi.dptr(None if x is None else self._vec(x, self.n)), code, capi.dptr(out)))
        return self._ret(out)

    def kt_residuals(self, lam, mult_x_U, mult_x_L, df=None):
        """common.jl:35-44 with the Jacobian of the last update."""
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_kt_residuals(
            self._h, capi.dptr(None if df is None else self._vec(df, self.n)), capi.dptr(self._vec(lam, self.m)),
            capi.dptr(self._vec(mult_x_U, self.n)), capi.dptr(self._vec(mult_x_L, self.n)), capi.dptr(out)))
        return self._ret(out)

    def norm_complementarity(self, lam, E=None):
        """common.jl:51-68 (infinity norm)."""
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_norm_complementarity(
            self._h, capi.dptr(None if E is None else self._vec(E, self.m)), capi.dptr(self._vec(lam, self.m)),
            capi.dptr(out)))
        return self._ret(out)

    def row_norms(self):
        out = np.empty((self.batch, self.m))
        capi.check(self._lib.asm_slp_row_norms(self._h, capi.dptr(out)))
        return out[0] if self.batch == 1 else out

    def merit_phi(self, base, E_trial, nu, alpha, feasibility=False):
        """compute_phi (slp.jl:79-115): ``base`` is f(x+αp) (normal) or prim_infeas (restoration)."""
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_merit_phi(
            self._h, capi.dptr(self._scal(base)), capi.dptr(None if E_trial is None else self._vec(E_trial, self.m)),
            capi.dptr(self._vec(nu, self.m)), capi.dptr(self._scal(alpha)), 1 if feasibility else 0, capi.dptr(out)))
        return self._ret(out)

    def merit_derivative(self, nu, feasibility=False):
        """compute_derivative (slp.jl:122-147) with the step / slacks of the last solve."""
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_merit_derivative(self._h, capi.dptr(self._vec(nu, self.m)),
                                                      1 if feasibility else 0, capi.dptr(out)))
        return self._ret(out)

    # -- device-resident variants (inputs of the last ``update`` stay in HBM) -----------------------------------
    def reassemble(self, feasibility=False):
        capi.check(self._lib.asm_slp_reassemble(self._h, 1 if feasibility else 0))

    def extract_device(self):
        capi.check(self._lib.asm_slp_extract_device(self._h))

    def timer_start(self):
        capi.check(self._lib.asm_slp_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_double()
        capi.check(self._lib.asm_slp_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def kernel_timing(self, reps=50):
        """Average device ms of one launch of (A'y + primal update, A xbar + dual update)."""
        a = C.c_double()
        b = C.c_double()
        capi.check(self._lib.asm_slp_kernel_timing(self._h, int(reps), C.byref(a), C.byref(b)))
        return a.value, b.value

    def ipm_info(self):
        """Sizes of the barrier engine's factorisation and the Newton steps of the last solve."""
        st = np.zeros(14, dtype=np.int64)
        tm = np.zeros(4)
        capi.check(self._lib.asm_slp_ipm_info(self._h, st.ctypes.data_as(capi.c_int64_p), capi.dptr(tm)))
        keys = ("kkt_dim", "nnz_L", "terms", "levels", "factor_chunks", "forward_chunks", "launches_factor",
                "launches_substitution", "factorisations", "substitution_pairs", "factor_distinct_reads",
                "factor_targets", "substitution_distinct_reads", "substitution_targets")
        out = {k: int(v) for k, v in zip(keys, st)}
        out.update(symbolic_ms=float(tm[0]), newton_steps=int(tm[1]))
        return out

    def ipm_timing(self, reps=20):
        """(factor_ms, substitution_pair_ms): device time per launch sequence of the whole batch, CUDA events."""
        f = C.c_double()
        s = C.c_double()
        capi.check(self._lib.asm_slp_ipm_timing(self._h, int(reps), C.byref(f), C.byref(s)))
        return f.value, s.value

    def engine_info(self):
        e = C.c_int32()
        g = C.c_int32()
        k = C.c_int32()
        capi.check(self._lib.asm_slp_engine_info(self._h, C.byref(e), C.byref(g), C.byref(k)))
        return dict(engine=e.value, group_size=g.value, groups=k.value)

    # -- device-side ACOPF evaluator (SURVEY.md 8(f)-1) ----------------------------------------------------------
    def attach_acopf(self, model):
        """Hand the network of an ``examples.acopf.AcopfModel`` to the device so that ``eval_acopf`` /
        ``acopf_trial`` replace the host callbacks (``src/MOI_wrapper.jl:1047-1069``).  All scenarios of the batch
        share the network; loads only enter the row bounds given at construction."""
        net = model.net
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)   # noqa: E731
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
        cf = model._cf
        keep = dict(
            f_bus=i32(net.f_bus), t_bus=i32(net.t_bus),
            coef=f64(np.stack([cf[k] for k in ("a_pf", "b_pf", "c_pf", "a_qf", "b_qf", "c_qf", "a_pt", "b_pt", "c_pt",
                                               "a_qt", "b_qt", "c_qt")])),
            gs=f64(net.gs), bs=f64(net.bs), cost2=f64(net.cost2), cost1=f64(net.cost1), cost0=f64(net.cost0),
            dc_loss1=f64(net.dc_loss1 if model.nd else np.zeros(1)),
            bal_ptr=i32(np.concatenate([[0], np.cumsum(np.bincount(model._bal_rows - model.r_bal,
                                                                   minlength=2 * model.nb))])),
            bal_col=i32(model._bal_cols), bal_coef=f64(model._bal_coef))
        d = capi.AcopfDesc()
        d.nb, d.ng, d.nl, d.nd, d.ref_bus = model.nb, model.ng, model.nl, model.nd, int(net.ref_bus)
        for k, a in keep.items():
            setattr(d, k, a.ctypes.data_as(capi.c_int32_p if a.dtype == np.int32 else capi.c_double_p))
        capi.check(self._lib.asm_slp_attach_acopf(self._h, C.byref(d)))

    def eval_acopf(self, x, delta=1000.0, feasibility=False):
        """``eval_functions!`` (slp.jl:186-191) on the device at ``x`` + the device part of ``update``."""
        capi.check(self._lib.asm_slp_eval_acopf(self._h, capi.dptr(self._vec(x, self.n)), capi.dptr(self._scal(delta)),
                                                1 if feasibility else 0))

    def get_eval_f(self):
        """f[batch] of the last evaluation (the only piece the batched driver needs back on the host)."""
        f = np.empty(self.batch)
        capi.check(self._lib.asm_slp_get_eval(self._h, capi.dptr(f), None, None, None))
        return f

    def get_eval_df(self):
        """df[batch, n] of the last evaluation (squeezed when ``batch == 1``): the gradient norm of the trust
        region's first penalty (slp.jl:54-66)."""
        df = np.empty((self.batch, self.n))
        capi.check(self._lib.asm_slp_get_eval(self._h, None, capi.dptr(df), None, None))
        return df[0] if self.batch == 1 and self._squeeze else df

    def get_eval(self):
        """(f, df, E, dE) of the last evaluation, ``[batch, ...]`` (squeezed when ``batch == 1``)."""
        B = self.batch
        f = np.empty(B); df = np.empty((B, self.n)); E = np.empty((B, self.m)); dE = np.empty((B, self.nnz_coo))
        capi.check(self._lib.asm_slp_get_eval(self._h, capi.dptr(f), capi.dptr(df), capi.dptr(E), capi.dptr(dE)))
        if B == 1 and self._squeeze:
            return float(f[0]), df[0], E[0], dE[0]
        return f, df, E, dE

    def acopf_trial(self, alpha, nu, base=None, feasibility=False):
        """``compute_phi(x + alpha p)`` (slp.jl:79-115) with f and g evaluated on the device at the trial point."""
        out = np.empty(self.batch)
        capi.check(self._lib.asm_slp_acopf_trial(
            self._h, capi.dptr(self._scal(alpha)), capi.dptr(self._vec(nu, self.m)),
            capi.dptr(None if base is None else self._scal(base)), 1 if feasibility else 0, capi.dptr(out)))
        return self._ret(out) if self._squeeze else out

    # -- instrumentation ----------------------------------------------------------------------------------------
    def launch_count(self) -> int:
        return int(self._lib.asm_slp_launch_count(self._h))

    def last_solve_timing(self):
        ms = C.c_double()
        it = C.c_int64()
        capi.check(self._lib.asm_slp_last_solve_timing(self._h, C.byref(ms), C.byref(it)))
        return ms.value, it.value


class B200LP:
    """General LP  ``min c'x + c0  s.t. rl <= Kx <= ru, lb <= x <= ub``  on the GPU — the object that takes
    GLPK's place as ``external_optimizer`` (reference ``src/parameters.jl:7``, ``src/algorithms/slp.jl:32``).
    ``K`` is given once as a CSR pattern (the MOI model skeleton of subproblem.jl:51-215); values, objective
    and bounds are replaced wholesale before each ``optimize`` (the modify/set calls of :248-484)."""

    def __init__(self, n_cols, n_rows, row_ptr, col_idx, batch=1, device=0, **lp_params):
        self._lib = capi.load()
        self.n, self.m, self.batch = int(n_cols), int(n_rows), int(batch)
        rp = np.ascontiguousarray(row_ptr, dtype=np.int64)
        ci = np.ascontiguousarray(col_idx, dtype=np.int32)
        self.nnz = int(rp[-1])
        self._h = C.c_void_p()
        capi.check(self._lib.asm_lp_create(self.n, self.m, self.nnz, rp.ctypes.data_as(capi.c_int64_p),
                                           ci.ctypes.data_as(capi.c_int32_p), self.batch, int(device),
                                           C.byref(self._h)))
        self.params = capi.default_params(**lp_params)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.asm_lp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _v(self, a, length):
        return capi.as_f64(a, (self.batch, length))

    def set_matrix_values(self, vals):
        capi.check(self._lib.asm_lp_set_matrix_values(self._h, capi.dptr(self._v(vals, self.nnz))))

    def set_objective(self, c, c0=0.0):
        c0 = np.full(self.batch, c0, dtype=np.float64) if np.ndim(c0) == 0 else capi.as_f64(c0, (self.batch,))
        capi.check(self._lib.asm_lp_set_objective(self._h, capi.dptr(self._v(c, self.n)), capi.dptr(c0)))

    def set_col_bounds(self, lb, ub):
        capi.check(self._lib.asm_lp_set_col_bounds(self._h, capi.dptr(self._v(lb, self.n)),
                                                   capi.dptr(self._v(ub, self.n))))

    def set_row_bounds(self, rl, ru):
        capi.check(self._lib.asm_lp_set_row_bounds(self._h, capi.dptr(self._v(rl, self.m)),
                                                   capi.dptr(self._v(ru, self.m))))

    def set_start(self, x=None, y=None):
        capi.check(self._lib.asm_lp_set_start(self._h, capi.dptr(None if x is None else self._v(x, self.n)),
                                              capi.dptr(None if y is None else self._v(y, self.m))))

    def optimize(self):
        info = (capi.LpInfo * self.batch)()
        capi.check(self._lib.asm_lp_solve(self._h, C.byref(self.params), info))
        self.info = _info_to_dicts(info, self.batch)
        return self.info

    def primal(self):
        x = np.empty((self.batch, self.n))
        capi.check(self._lib.asm_lp_get_primal(self._h, capi.dptr(x)))
        return x[0] if self.batch == 1 else x

    def row_dual(self):
        y = np.empty((self.batch, self.m))
        capi.check(self._lib.asm_lp_get_row_dual(self._h, capi.dptr(y)))
        return y[0] if self.batch == 1 else y

    def col_dual(self):
        lo = np.empty((self.batch, self.n))
        up = np.empty((self.batch, self.n))
        capi.check(self._lib.asm_lp_get_col_dual(self._h, capi.dptr(lo), capi.dptr(up)))
        return (lo[0], up[0]) if self.batch == 1 else (lo, up)


class B200RowPartitionedLP(B200LP):
    """One LP over several GPUs, one process per GPU (SURVEY.md §8e, BASELINE config 4): rank ``rank`` of ``world``
    owns a contiguous block of rows of ``K`` (balanced by nonzeros) with its duals; ``x`` is replicated and one NCCL
    all-reduce of the partial ``K'y`` completes every PDHG iteration.  All ranks pass the *global* pattern and
    data; each keeps its rows.  ``unique_id`` is the 128-byte id from :func:`nccl_unique_id` made on rank 0 and
    shared by the host (e.g. ``torch.distributed.broadcast_object_list``).  ``optimize`` is collective."""

    def __init__(self, n_cols, n_rows, row_ptr, col_idx, rank, world, unique_id, device=0, **lp_params):
        from . import shard
        self._lib = capi.load()
        rp = np.ascontiguousarray(row_ptr, dtype=np.int64)
        ci = np.ascontiguousarray(col_idx, dtype=np.int32)
        cuts = shard.row_blocks(rp, world)
        self.r0, self.r1 = cuts[rank], cuts[rank + 1]
        self.k0, self.k1 = int(rp[self.r0]), int(rp[self.r1])
        self.rank, self.world = int(rank), int(world)
        self.n, self.m, self.batch = int(n_cols), self.r1 - self.r0, 1
        self.m_global, self.nnz_global = int(n_rows), int(rp[-1])
        self.nnz = self.k1 - self.k0
        lrp = np.ascontiguousarray(rp[self.r0:self.r1 + 1] - self.k0)
        lci = np.ascontiguousarray(ci[self.k0:self.k1])
        assert len(unique_id) == 128
        self._h = C.c_void_p()
        capi.check(self._lib.asm_lp_dist_create(self.n, self.m, self.nnz, lrp.ctypes.data_as(capi.c_int64_p),
                                                lci.ctypes.data_as(capi.c_int32_p), self.rank, self.world,
                                                bytes(unique_id), int(device), C.byref(self._h)))
        self.params = capi.default_params(**lp_params)

    def set_matrix_values(self, vals):
        vals = capi.as_f64(vals, (self.nnz_global,))
        super().set_matrix_values(np.ascontiguousarray(vals[self.k0:self.k1]))

    def set_row_bounds(self, rl, ru):
        rl, ru = capi.as_f64(rl, (self.m_global,)), capi.as_f64(ru, (self.m_global,))
        super().set_row_bounds(np.ascontiguousarray(rl[self.r0:self.r1]), np.ascontiguousarray(ru[self.r0:self.r1]))

    def set_start(self, x=None, y=None):
        super().set_start(x, None if y is None else np.ascontiguousarray(capi.as_f64(y)[self.r0:self.r1]))


def nccl_unique_id() -> bytes:
    """128-byte NCCL unique id (call on one rank, share with the others)."""
    buf = C.create_string_buffer(128)
    capi.check(capi.load().asm_dist_unique_id(buf))
    return buf.raw
