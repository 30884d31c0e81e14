"""SLP drivers on top of the GPU sub-LP engine — the host orchestration of the reference, unchanged in
behaviour, with every array-sized operation of the iteration moved behind the C ABI.

================================  ==========================================================================
here                              reference (relative to /root/reference)
================================  ==========================================================================
``Parameters``                    ``src/parameters.jl:1-29``
``Model`` / ``optimize``          ``src/model.jl:1-80`` (problem container, algorithm dispatch)
``SlpLSBatch``                    ``src/algorithms/slp_line_search.jl:78-261``
``SlpTRBatch``                    ``src/algorithms/slp_trust_region.jl:62-251``, ``src/algorithms/slp.jl:54-66``
``SlpLS`` / ``SlpTR``             ``SlpLS`` / ``SlpTR`` ``(model)``, ``run!``, the write-back into ``Model``
                                  (``slp_line_search.jl:207-214``): the one-scenario batch
``STATUS``                        ``src/status.jl:2-22``
================================  ==========================================================================

Each algorithm has one driver, the lock-step batch (``SlpLSBatch``, ``SlpTRBatch``); a single solve is its
one-scenario case.  The NLP callbacks (``eval_f``, ``eval_grad_f``, ``eval_g``, ``eval_jac_g``) stay on the host
exactly like the JuMP ``NLPEvaluator`` of the reference (``src/MOI_wrapper.jl:1047-1069``), unless a device-side
evaluator replaces them: the ACOPF one for ``examples.acopf.AcopfModel``, the QCQP one for
``examples.qcqp.QcqpModel`` (affine and quadratic models such as ``examples.acopf.AcrModel``).  Per round the driver hands ``x, f, df, E, dE`` to ``SubLp.update`` (one H2D
hand-over, assembly + bounds on the device), solves the sub-LPs with ``solve_extract`` and asks the device for the
merit / KKT reductions.
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field, replace
from functools import partial

import numpy as np

from .sublp import SubLp, LP_OPTIMAL, LP_INFEASIBLE

INF = math.inf

# src/status.jl:2-22
STATUS = {
    0: "Solve_Succeeded", 1: "Solved_To_Acceptable_Level", 2: "Infeasible_Problem_Detected",
    3: "Search_Direction_Becomes_Too_Small", 4: "Diverging_Iterates", 5: "User_Requested_Stop",
    6: "Feasible_Point_Found", -1: "Maximum_Iterations_Exceeded", -2: "Restoration_Failed",
    -3: "Error_In_Step_Computation", -4: "Maximum_CpuTime_Exceeded", -5: "Optimize_not_called",
    -10: "Not_Enough_Degrees_Of_Freedom", -11: "Invalid_Problem_Definition", -12: "Invalid_Option",
    -13: "Invalid_Number_Detected", -100: "Unrecoverable_Exception", -101: "NonIpopt_Exception_Thrown",
    -102: "Insufficient_Memory", -199: "Internal_Error",
}


@dataclass
class Parameters:
    """src/parameters.jl:1-29.  ``external_optimizer`` is the hook: a callable
    ``(n, m, j_str, x_L, x_U, g_L, g_U) -> SubLp``-like object, or ``None`` → status -12 (model.jl:64-66).
    The default is the B200 engine."""
    mu_merit: float = 1.0
    external_optimizer: object = "B200LP"
    method: str = "SLP"
    algorithm: str = "Line Search"
    max_mu: float = 1.0e10
    rho: float = 0.8
    eta: float = 0.4
    tau: float = 0.9
    tol_direction: float = 1.0e-6
    tol_residual: float = 0.01
    tol_infeas: float = 0.01
    max_iter: int = 1000
    time_limit: float = INF
    min_alpha: float = 1.0e-6
    tr_size: float = 0.4
    OutputFlag: int = 0
    StatisticsFlag: int = 0
    # engine options forwarded to asm_lp_params (not in the reference)
    lp_options: dict = field(default_factory=dict)
    device: int = 0
    # either algorithm on an examples.acopf.AcopfModel or an examples.qcqp.QcqpModel with the B200 engine: evaluate
    # f, g, the Jacobian and the merit at trial points (backtracking / step quality) with the device-side ACOPF or QCQP
    # evaluator instead of the host callbacks (SURVEY.md 8(f)-1)
    device_evaluator: bool = False


class Model:
    """src/model.jl:1-61: the problem container handed over by the MOI front-end
    (``src/MOI_wrapper.jl:1093-1099``)."""

    def __init__(self, n, m, x_L, x_U, g_L, g_U, j_str, eval_f, eval_g, eval_grad_f, eval_jac_g,
                 parameters: Parameters | None = None, x0=None):
        self.n, self.m = int(n), int(m)
        self.x_L = np.asarray(x_L, dtype=float)
        self.x_U = np.asarray(x_U, dtype=float)
        self.g_L = np.asarray(g_L, dtype=float)
        self.g_U = np.asarray(g_U, dtype=float)
        self.j_str = np.asarray(j_str, dtype=np.int64).reshape(-1, 2)
        self.eval_f, self.eval_g, self.eval_grad_f, self.eval_jac_g = eval_f, eval_g, eval_grad_f, eval_jac_g
        self.parameters = parameters if parameters is not None else Parameters()
        self.x = np.zeros(self.n) if x0 is None else np.array(x0, dtype=float)
        self.g = np.zeros(self.m)
        self.mult_g = np.zeros(self.m)
        self.mult_x_L = np.zeros(self.n)
        self.mult_x_U = np.zeros(self.n)
        self.obj_val = 0.0
        self.status = -5
        self.statistics = {}

    @classmethod
    def from_problem(cls, problem, parameters=None):
        """Wrap an object exposing ``n, m, x_L, x_U, g_L, g_U, j_str, x0`` and the four callbacks."""
        mdl = cls(problem.n, problem.m, problem.x_L, problem.x_U, problem.g_L, problem.g_U, problem.j_str,
                  problem.eval_f, problem.eval_g, problem.eval_grad_f, problem.eval_jac_g, parameters, problem.x0)
        mdl.source = problem         # the device-side evaluator needs the network behind the callbacks
        return mdl

    def add_statistic(self, name, value):                                   # model.jl:82-97
        if self.parameters.StatisticsFlag:
            self.statistics.setdefault(name, []).append(value)


def optimize(model: Model):
    """model.jl:63-80."""
    o = model.parameters
    if o.external_optimizer is None:
        model.status = -12
        return model
    if o.method == "SLP" and o.algorithm == "Line Search":
        SlpLS(model).run()
    elif o.method == "SLP" and o.algorithm == "Trust Region":
        SlpTR(model).run()
    else:
        raise ValueError(f"unknown method/algorithm {o.method}/{o.algorithm}")
    return model


class _SlpBatch:
    """B independent SLP solves that share one Jacobian pattern (load scenarios of one network, BASELINE config 5),
    advanced in lock-step so that every round is one batched call of each operation of the device hot path.
    ``problems`` are objects with the ``Model.from_problem`` interface, or ``Model`` s (which start from ``model.x``).
    Subclasses give the round (``run``) and ``warm_start``, the B200 engine's warm-start flag.

    ``record``: optional ``callable(driver, dict)``, called before every sub-LP solve for each scenario solved, with
    that scenario's linearisation (``x, f, df, E, dE, delta, fr``).  ``lp_log[s]`` lists (status, objective,
    restoration flag, iterations) of every sub-LP solved for scenario ``s``.

    ``lanes``: run ``len(problems)`` scenarios through a handle of only ``lanes`` lanes (continuous batching).  Lane
    ``l`` starts with problem ``l``; a problem whose run ends in a round is retired in that round, and before the next
    round the next queued problems are loaded into the freed lanes with one ``load_lanes`` call (the handle, its
    symbolic analysis and its captured graphs stay).  A loaded lane starts exactly like a lane of a fresh batch.
    During ``run`` the state arrays are indexed by lane; afterwards ``ret``, ``iter``, ``x``, ``obj_val``,
    ``prim_infeas``, ``dual_infeas``, ``compl``, ``lp_solves`` and ``lp_log`` (and ``delta`` for the trust region) are
    indexed by problem.  ``None`` (or ``lanes >= len(problems)``): one lane per problem, one batch."""

    # Line search: every sub-LP starts from the previous one's (p, lambda) -- the analogue of GLPK keeping its basis
    # (one glp_prob per SLP run, slp.jl:24); it halves the PDHG work (case118: 1.03 M -> 0.51 M iterations for the
    # same 14 SLP iterations).  Trust region: cold starts; there a warm start changes which minimiser of the
    # (degenerate) restoration LPs is returned and the runs measured so far ended further from the optimum.
    # ``lp_options={"warm_start": ...}`` overrides either.
    warm_start = 1
    _dev = "acopf"          # the device-side evaluator attached by _instantiate: "acopf" or "qcqp"
    # per-problem results of a queued run (see ``lanes``)
    _outputs = ("ret", "iter", "x", "obj_val", "prim_infeas", "dual_infeas", "compl", "lp_solves")

    def __init__(self, problems, parameters: Parameters | None = None, device_evaluator: bool = False, lanes=None):
        self.device_evaluator = bool(device_evaluator)
        self.problems = list(problems)
        self.options = parameters if parameters is not None else Parameters()
        p0 = self.problems[0]
        self.B, self.n, self.m = len(self.problems), p0.n, p0.m
        for pr in self.problems:
            if pr.n != self.n or pr.m != self.m or not np.array_equal(pr.j_str, p0.j_str):
                raise ValueError("batched scenarios must share the Jacobian pattern")
        self._queue = None                  # all problems of a queued run; None: one lane per problem
        if lanes is not None:
            if int(lanes) < 1:
                raise ValueError(f"lanes must be at least 1, got {lanes}")
            ext = self.options.external_optimizer
            if int(lanes) < self.B:
                if ext != "B200LP" and not hasattr(ext, "load_lanes"):
                    raise ValueError("lanes < len(problems) needs an external_optimizer with load_lanes")
                self._queue = self.problems
                self.problems = self._queue[:int(lanes)]
                self.B = int(lanes)
                self._slot = np.arange(self.B)  # problem held by each lane, -1 once retired with the queue empty
                self._next = self.B             # next problem to load
                self.loads = []                 # lanes loaded before each round that loaded any, (round, lanes)
        B, n, m = self.B, self.n, self.m
        self.x = np.array([np.array(pr.x if isinstance(pr, Model) else pr.x0, dtype=float) for pr in self.problems])
        self.f = np.zeros(B)
        self.df = np.zeros((B, n))
        self.E = np.zeros((B, m))
        self.dE = np.zeros((B, len(p0.j_str)))
        self.p = np.zeros((B, n))
        self.lam = np.zeros((B, m))
        self.mult_x_U = np.zeros((B, n))
        self.mult_x_L = np.zeros((B, n))
        self.nu = np.zeros((B, m))
        self.iter = np.ones(B, dtype=np.int64)
        self.ret = np.full(B, -5, dtype=np.int64)
        self.running = np.ones(B, dtype=bool)
        self.fr = np.zeros(B, dtype=bool)
        self.prim_infeas = np.full(B, INF)
        self.dual_infeas = np.full(B, INF)
        self.compl = np.full(B, INF)
        self.obj_val = np.zeros(B)
        self.rounds = 0
        self.two_phase_rounds = 0       # rounds with scenarios in both phases: two sub-LP batch solves
        self.lp_solves = np.zeros(B, dtype=np.int64)
        self.lp_log = [[] for _ in range(B)]
        self.lp_iterations = 0
        self.lp_time = 0.0
        self.optimizer = None
        self.record = None

    def _instantiate(self):
        o = self.options
        prs = self.problems
        arr = lambda name: np.array([np.asarray(getattr(pr, name), dtype=float) for pr in prs])  # noqa: E731
        if o.external_optimizer == "B200LP":
            qcqp = self.device_evaluator and self._is_qcqp(prs[0])
            if qcqp:
                # the QCQP evaluator holds one set of term lists for the batch: scenarios differ in bounds and start
                # only.  A queued run checks every problem up front, so that a mismatch fails before any solve.
                models = self._acopf(self._queue or prs)
                for k, pr in enumerate(models[1:], 1):
                    if not self._is_qcqp(pr):
                        raise ValueError(f"device_evaluator: scenario {k} is not a QcqpModel like scenario 0")
                    diff = models[0].same_terms(pr)
                    if diff is not None:
                        raise ValueError(f"device_evaluator: scenario {k} differs from scenario 0 in its terms ({diff})")
            opt = SubLp(self.n, self.m, prs[0].j_str, arr("x_L"), arr("x_U"), arr("g_L"), arr("g_U"), batch=self.B,
                        device=o.device, **{"warm_start": self.warm_start, **o.lp_options})
            opt._squeeze = False
            if qcqp:
                opt.attach_qcqp(models[0])
                self._dev = "qcqp"
            elif self.device_evaluator:
                # the device evaluator holds one topology, shunts, costs, dc-line losses and reference bus for the
                # batch; branch data (impedances, taps, shifts, outages) may differ per scenario, and loads, generator
                # outages and relaxed angle rows only enter the bounds.  A Model hands over the problem it was built from.
                acopf = self._acopf(prs)
                n0 = acopf[0].net
                # a queued run checks every problem up front, so that a mismatch fails before any solve
                for k, pr in enumerate(self._acopf(self._queue or prs)[1:], 1):
                    for name in ("f_bus", "t_bus", "gs", "bs", "cost2", "cost1", "cost0", "gen_bus", "dc_loss1"):
                        if not np.array_equal(getattr(pr.net, name), getattr(n0, name)):
                            raise ValueError(f"device_evaluator: scenario {k} differs from scenario 0 in network.{name}")
                    if pr.net.ref_bus != n0.ref_bus:
                        raise ValueError(f"device_evaluator: scenario {k} has another reference bus")
                opt.attach_acopf(acopf)
                self._dev = "acopf"
            return opt
        if self.device_evaluator:
            raise ValueError("device_evaluator needs the B200 engine")
        return o.external_optimizer(self.n, self.m, prs[0].j_str, arr("x_L"), arr("x_U"), arr("g_L"), arr("g_U"),
                                    batch=self.B)

    @staticmethod
    def _is_qcqp(pr):
        return hasattr(pr.source if isinstance(pr, Model) else pr, "qcqp_desc")

    def _dev_eval(self, delta, feasibility):
        """The device-side evaluation at ``self.x`` + the device part of ``update``, with the attached evaluator."""
        if self._dev == "qcqp":
            self.optimizer.eval_qcqp(self.x, delta, feasibility)
        else:
            self.optimizer.eval_acopf(self.x, delta, feasibility)

    def _dev_trial(self, alpha, fr):
        """compute_phi(x + alpha p) for the batch with the attached device-side evaluator."""
        trial = self.optimizer.qcqp_trial if self._dev == "qcqp" else self.optimizer.acopf_trial
        return np.atleast_1d(trial(alpha, self.nu, self.prim_infeas if fr else None, fr))

    @staticmethod
    def _acopf(prs):
        """The ACOPF models behind ``prs`` (a Model hands over the problem it was built from)."""
        return [pr.source if isinstance(pr, Model) else pr for pr in prs]

    def _clip_starts(self):
        for s, pr in enumerate(self.problems):
            self._clip_start(s, pr)

    def _clip_start(self, s, pr):                                           # slp_line_search.jl:96-105
        lo = pr.x_L > -INF
        self.x[s][lo] = np.maximum(self.x[s][lo], pr.x_L[lo])
        up = pr.x_U > -INF
        self.x[s][up] = np.minimum(self.x[s][up], pr.x_U[up])

    def _reset_lane(self, s, pr):
        """Lane ``s`` starts problem ``pr`` exactly like lane ``s`` of a fresh batch."""
        self.x[s] = np.array(pr.x if isinstance(pr, Model) else pr.x0, dtype=float)
        self._clip_start(s, pr)
        for a in (self.f, self.df, self.E, self.dE, self.p, self.lam, self.mult_x_U, self.mult_x_L, self.nu):
            a[s] = 0.0
        self.prim_infeas[s] = self.dual_infeas[s] = self.compl[s] = INF
        self.iter[s] = 1
        self.ret[s] = -5
        self.fr[s] = False
        self.running[s] = True
        self.lp_solves[s] = 0
        self.lp_log[s] = []

    def _refill(self):
        """Continuous batching, at the end of a round: retire the problems whose runs ended in it (their results are
        stored by problem), then load the next queued problems into the freed lanes with one ``load_lanes`` call."""
        if not hasattr(self, "_res"):
            N = len(self._queue)
            self._res = {name: np.zeros((N,) + getattr(self, name).shape[1:], getattr(self, name).dtype)
                         for name in self._outputs}
            self._res_log = [None] * N
        done = np.nonzero(~self.running & (self._slot >= 0))[0]
        for s in done:
            q = self._slot[s]
            self.obj_val[s] = self.problems[s].eval_f(self.x[s])
            for name in self._outputs:
                self._res[name][q] = getattr(self, name)[s]
            self._res_log[q] = self.lp_log[s]
            self._slot[s] = -1
        load = done[:max(0, len(self._queue) - self._next)]
        if not len(load):
            return
        new = self._queue[self._next:self._next + len(load)]
        for s, pr in zip(load, new):
            self._slot[s] = self._next
            self._next += 1
            self.problems[s] = pr
            self._reset_lane(s, pr)
        bounds = [np.array([np.asarray(getattr(pr, name), dtype=float) for pr in new])
                  for name in ("x_L", "x_U", "g_L", "g_U")]
        if self.device_evaluator and self._dev == "acopf":
            self.optimizer.load_lanes(load, *bounds, acopf=self._acopf(new))
        else:
            self.optimizer.load_lanes(load, *bounds)
        self.loads.append((self.rounds, load.copy()))

    def _eval(self, s):
        pr = self.problems[s]
        self.f[s] = pr.eval_f(self.x[s])
        pr.eval_grad_f(self.x[s], self.df[s])
        pr.eval_g(self.x[s], self.E[s])
        pr.eval_jac_g(self.x[s], "eval", None, None, self.dE[s])

    def _solve_phase(self, fr, sel, delta):
        """Sub-LP batch of one phase (``delta``: the trust-region radius, scalar or per scenario).  ``sel``: the
        scenarios that are running in this phase -- the others (terminated, or in the other phase, whose normal LP is
        infeasible by construction) are masked out of the solve instead of being re-solved every round."""
        opt = self.optimizer
        if hasattr(opt, "set_active"):
            opt.set_active(sel)
        if fr and self.device_evaluator:
            self._dev_eval(delta, True)
        elif fr:                    # the normal-phase data push was done at the start of this round
            opt.update(self.x, self.f, self.df, self.E, self.dE, delta, True)
        idx = np.nonzero(sel)[0]
        if self.record is not None:
            radius = np.broadcast_to(delta, (self.B,))
            for s in idx:
                self.record(self, dict(x=self.x[s].copy(), f=float(self.f[s]), df=self.df[s].copy(),
                                       E=self.E[s].copy(), dE=self.dE[s].copy(), delta=float(radius[s]), fr=fr))
        t0 = time.time()
        p, lam, mu_u, mu_l, slack, status = opt.solve_extract()
        self.lp_time = time.time() - t0
        status = np.atleast_1d(status)
        self.lp_solves[sel] += 1
        info = getattr(opt, "last_info", None) or [{}] * self.B
        self.lp_iterations += int(sum(i.get("iterations") or 0 for i in info))
        for s in idx:
            self.lp_log[s].append((int(status[s]), info[s].get("objective"), fr, info[s].get("iterations")))
        return [np.atleast_2d(a) if np.ndim(a) < 2 else a for a in (p, lam, mu_u, mu_l)] + [slack, status]

    def _print(self, s, phi, derivative, alpha, extra=""):
        if self.options.OutputFlag:
            print(f"{s:4d}  {self.iter[s]:6d}  {self.f[s]: .8e}  {phi: .8e}  {derivative: .4e}  "
                  f"{float(np.max(np.abs(self.p[s]))):.4e}  {alpha:.4e}  {self.prim_infeas[s]:.4e}  "
                  f"{self.dual_infeas[s]:.4e}  {self.compl[s]:.4e}  {self.lp_time:7.2f}{extra}")

    def _finish(self):
        if self._queue is None:
            for s, pr in enumerate(self.problems):
                self.obj_val[s] = pr.eval_f(self.x[s])
            return
        # every problem was retired by _refill in the round its run ended: publish the results by problem
        self.problems = self._queue
        for name in self._outputs:
            setattr(self, name, self._res[name])
        self.lp_log = self._res_log


class SlpLSBatch(_SlpBatch):
    """B independent line-search SLP solves in lock-step (see ``_SlpBatch``): every round is one `update`, the KKT
    reductions, one sub-LP batch solve (two when some scenarios are in feasibility restoration), and one batched merit
    evaluation per backtracking round.  Per scenario the control flow is exactly ``run!`` of the reference
    (``slp_line_search.jl:78-215``) — a scenario that terminates simply stops moving while the others go on.  A
    single solve (``SlpLS``) is the one-scenario batch.

    ``device_evaluator=True`` (ACOPF scenarios of one network, or QCQP scenarios that share their terms; B200
    engine): the NLP callbacks are not called at all — f, g and the Jacobian are evaluated by the device-side evaluator
    (``SubLp.eval_acopf`` / ``SubLp.eval_qcqp``) and every backtracking trial is one ``SubLp.acopf_trial`` /
    ``SubLp.qcqp_trial`` call for the whole batch."""

    def __init__(self, problems, parameters: Parameters | None = None, device_evaluator: bool = False, lanes=None):
        super().__init__(problems, parameters, device_evaluator, lanes)
        self.alpha = np.zeros(self.B)

    def _reset_lane(self, s, pr):
        super()._reset_lane(s, pr)
        self.alpha[s] = 0.0

    def run(self):
        o = self.options
        B = self.B
        self._clip_starts()
        if self.optimizer is None:
            self.optimizer = self._instantiate()
        opt = self.optimizer
        while self.running.any():
            self.rounds += 1
            run = np.nonzero(self.running)[0]
            # KKT metrics with last round's multipliers on this round's Jacobian (App. C-7)
            if self.device_evaluator:
                self._dev_eval(1000.0, False)
                self.f[:] = opt.get_eval_f()
            else:
                for s in run:
                    self._eval(s)
                opt.update(self.x, self.f, self.df, self.E, self.dE, 1000.0, False)
            self.prim_infeas[run] = np.atleast_1d(opt.norm_violations(None, None, INF))[run]
            self.dual_infeas[run] = np.atleast_1d(opt.kt_residuals(self.lam, self.mult_x_U, self.mult_x_L))[run]
            self.compl[run] = np.atleast_1d(opt.norm_complementarity(self.lam))[run]
            need = {False: self.running & ~self.fr, True: self.running & self.fr}
            self.two_phase_rounds += int(need[False].any() and need[True].any())
            status = np.zeros(B, dtype=np.int64)
            phi0 = np.zeros(B)
            deriv = np.zeros(B)
            for fr in (False, True):
                sel = need[fr]
                if not sel.any():
                    continue
                p, lam, mu_u, mu_l, slack, st = self._solve_phase(fr, sel, 1000.0)
                idx = np.nonzero(sel)[0]
                self.p[idx], self.lam[idx], self.mult_x_U[idx], self.mult_x_L[idx] = p[idx], lam[idx], mu_u[idx], mu_l[idx]
                status[idx] = st[idx]
                ok = idx[st[idx] == LP_OPTIMAL]
                # compute_nu! (:251-261) then phi(0) and D with this phase's device state
                first = ok[self.iter[ok] == 1]
                later = ok[self.iter[ok] != 1]
                self.nu[first] = np.abs(self.lam[first])
                self.nu[later] = np.maximum(self.nu[later], np.abs(self.lam[later]))
                base = self.prim_infeas if fr else self.f
                phi0[sel] = np.atleast_1d(opt.merit_phi(base, None, self.nu, np.zeros(B), fr))[sel]
                deriv[sel] = np.atleast_1d(opt.merit_derivative(self.nu, fr))[sel]
                self._line_search(fr, ok, phi0, deriv)
            # ---- per-scenario control flow of run! (:127-205)
            for s in run:
                st = status[s]
                if st not in (LP_OPTIMAL, LP_INFEASIBLE):
                    # Deviation from slp_line_search.jl:129, whose `slp.ret == -3` is a comparison, not an assignment:
                    # the run would end as -5 "Optimize_not_called" after a full solve.  -3 (Error_In_Step_Computation)
                    # is the evident intent.
                    self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else -3
                    self.running[s] = False
                    continue
                if st == LP_INFEASIBLE:
                    if self.fr[s]:
                        self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else 2
                        self.running[s] = False
                    else:
                        self.fr[s] = True                                   # re-solved next round, iter unchanged
                    continue
                self._print(s, phi0[s], deriv[s], self.alpha[s])
                if self.iter[s] >= o.max_iter:
                    self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else -1
                    self.running[s] = False
                    continue
                if (self.prim_infeas[s] <= o.tol_infeas and self.compl[s] <= o.tol_residual) or \
                        float(np.max(np.abs(self.p[s]))) <= o.tol_direction:
                    if self.fr[s]:
                        self.fr[s] = False
                        self.iter[s] += 1
                        continue
                    elif self.dual_infeas[s] <= o.tol_residual:
                        self.ret[s] = 0
                        self.running[s] = False
                        continue
                if not self._valid[s]:
                    if self._ret3[s]:
                        self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else 2
                        self.running[s] = False
                    else:
                        self.fr[s] = True
                        self.iter[s] += 1
                    continue
                self.x[s] = self.x[s] + self.alpha[s] * self.p[s]
                self.iter[s] += 1
            if self._queue is not None:
                self._refill()
        self._finish()
        return self

    def _line_search(self, fr, idx, phi0, deriv):
        """compute_alpha (:222-244) for the scenarios ``idx`` of one phase, one batched merit call per trial round."""
        o = self.options
        B = self.B
        if not hasattr(self, "_valid"):
            self._valid = np.ones(B, dtype=bool)
            self._ret3 = np.zeros(B, dtype=bool)
        self._valid[idx] = True
        self._ret3[idx] = False
        self.alpha[idx] = 1.0
        searching = np.zeros(B, dtype=bool)
        searching[idx] = True
        base = np.zeros(B)
        Et = self.E.copy()
        while searching.any():
            act = np.nonzero(searching)[0]
            if self.device_evaluator:
                phi = self._dev_trial(self.alpha, fr)
            else:
                for s in act:
                    pr = self.problems[s]
                    xt = self.x[s] + self.alpha[s] * self.p[s]
                    pr.eval_g(xt, Et[s])
                    base[s] = self.prim_infeas[s] if fr else pr.eval_f(xt)
                phi = np.atleast_1d(self.optimizer.merit_phi(base, Et, self.nu, self.alpha, fr))
            for s in act:
                if phi[s] > phi0[s] + o.eta * self.alpha[s] * deriv[s]:
                    if self.alpha[s] < o.min_alpha:
                        if fr:
                            self._ret3[s] = True
                        self._valid[s] = False
                        searching[s] = False
                    else:
                        self.alpha[s] *= o.tau
                else:
                    searching[s] = False


class SlpTRBatch(_SlpBatch):
    """B independent trust-region SLP solves in lock-step (see ``_SlpBatch``).  Per scenario the control flow is
    exactly ``run!`` of the reference (``slp_trust_region.jl:87-206``) — a scenario that terminates simply stops moving
    while the others go on.  A single solve (``SlpTR``) is the one-scenario batch.  Each scenario has its own radius
    ``delta[s]``, which also bounds its restoration LPs (``sub_optimize!(slp, Δ)`` passes Δ in both phases).

    A round is one evaluation + `update`, then for each phase that has running scenarios: one masked sub-LP batch
    solve, ν, the KKT metrics with the new multipliers, and one batched ϕ(x + p), ϕ(x) and predicted reduction for
    ``step_quality``.  All of a phase runs before the next phase's push, which overwrites the step and slacks on the
    device that the merit calls read.

    ``device_evaluator=True``: as for ``SlpLSBatch``; ϕ(x + p) is one ``SubLp.acopf_trial`` / ``SubLp.qcqp_trial``
    call for the batch."""

    warm_start = 0      # see _SlpBatch.warm_start
    _outputs = _SlpBatch._outputs + ("delta",)

    def __init__(self, problems, parameters: Parameters | None = None, device_evaluator: bool = False, lanes=None):
        super().__init__(problems, parameters, device_evaluator, lanes)
        self.delta = np.full(self.B, float(self.options.tr_size))           # slp_trust_region.jl:62-65
        self.delta_max = 2.0
        self.alpha1 = 0.1
        self.alpha2 = 0.25

    def _reset_lane(self, s, pr):
        super()._reset_lane(s, pr)
        self.delta[s] = float(self.options.tr_size)

    def run(self):                                                          # :87-206
        self._clip_starts()
        if self.optimizer is None:
            self.optimizer = self._instantiate()
        opt = self.optimizer
        while self.running.any():
            self.rounds += 1
            if self.device_evaluator:
                self._dev_eval(self.delta, False)
                self.f[:] = opt.get_eval_f()
            else:
                for s in np.nonzero(self.running)[0]:
                    self._eval(s)
                opt.update(self.x, self.f, self.df, self.E, self.dE, self.delta, False)
            need = {False: self.running & ~self.fr, True: self.running & self.fr}
            self.two_phase_rounds += int(need[False].any() and need[True].any())
            for fr in (False, True):
                if need[fr].any():
                    self._phase(fr, need[fr])
            if self._queue is not None:
                self._refill()
        self._finish()
        return self

    def _phase(self, fr, sel):
        """One iteration of ``run!`` (:117-205) for the scenarios ``sel``, all in phase ``fr``."""
        o = self.options
        opt = self.optimizer
        p, lam, mu_u, mu_l, _, status = self._solve_phase(fr, sel, self.delta)
        idx = np.nonzero(sel)[0]
        self.p[idx], self.lam[idx], self.mult_x_U[idx], self.mult_x_L[idx] = p[idx], lam[idx], mu_u[idx], mu_l[idx]
        ok = idx[status[idx] == LP_OPTIMAL]
        if len(ok):
            self._compute_nu(fr, ok)
            self.prim_infeas[ok] = np.atleast_1d(opt.norm_violations(None, None, INF))[ok]
            self.dual_infeas[ok] = np.atleast_1d(opt.kt_residuals(self.lam, self.mult_x_U, self.mult_x_L))[ok]
            self.compl[ok] = np.atleast_1d(opt.norm_complementarity(self.lam))[ok]
        viol1 = None
        quality = []
        for s in idx:
            st = status[s]
            if st not in (LP_OPTIMAL, LP_INFEASIBLE):
                if viol1 is None:   # 1-norm at x: E and x of this phase's push are g(x) and x
                    viol1 = np.atleast_1d(opt.norm_violations(None, None, 1))
                self.ret[s] = 6 if viol1[s] <= o.tol_infeas else -3           # see SlpLSBatch.run (:131)
                self.running[s] = False
                continue
            if st == LP_INFEASIBLE:
                if fr:
                    self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else 2
                    self.running[s] = False
                else:
                    self.fr[s] = True                                       # re-solved next round, iter unchanged
                continue
            if self.prim_infeas[s] <= o.tol_infeas and self.compl[s] <= o.tol_residual and \
                    float(np.max(np.abs(self.p[s]))) <= o.tol_direction:
                if fr:
                    self.fr[s] = False
                    self.iter[s] += 1
                    # Deviation from slp_trust_region.jl:163-170, which `continue`s here without ever reaching its
                    # max_iter test: once the trust region has collapsed (delta ~ 1e-7) at a point that is feasible to
                    # tolerance but whose linearisation is infeasible inside the tiny box, the reference alternates
                    # normal LP (INFEASIBLE) / restoration LP forever.  Stop as its own max_iter branch (:177-183)
                    # would.
                    if self.iter[s] >= o.max_iter:
                        self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else -1
                        self.running[s] = False
                    continue
                if self.dual_infeas[s] <= o.tol_residual:
                    self.ret[s] = 0
                    self.running[s] = False
                    continue
            if self.iter[s] >= o.max_iter:
                self.ret[s] = 6 if self.prim_infeas[s] <= o.tol_infeas else -1
                self.running[s] = False
                continue
            quality.append(s)
        if quality:
            self._step_quality(fr, np.array(quality))

    def _compute_nu(self, fr, ok):                                          # slp.jl:54-66
        first = ok[self.iter[ok] == 1]
        later = ok[self.iter[ok] != 1]
        if len(first):
            rn = np.atleast_2d(self.optimizer.row_norms())
            df = None
            if not fr:
                df = self.optimizer.get_eval_df() if self.device_evaluator else self.df
            for s in first:
                norm_df = 1.0 if fr else float(np.linalg.norm(df[s]))
                self.nu[s] = np.maximum(1.0, norm_df / np.maximum(1.0, rn[s]))
        self.nu[later] = np.maximum(self.nu[later], np.abs(self.lam[later]))

    def _step_quality(self, fr, idx):                                       # :213-251
        """step_quality for the scenarios ``idx`` of phase ``fr``, then the step acceptance of run! (:195-204)."""
        o = self.options
        opt = self.optimizer
        B = self.B
        base = self.prim_infeas if fr else self.f
        if self.device_evaluator:
            phi1 = self._dev_trial(np.ones(B), fr)
        else:
            base1 = base.copy()
            Et = self.E.copy()
            for s in idx:
                pr = self.problems[s]
                xt = self.x[s] + self.p[s]
                pr.eval_g(xt, Et[s])
                if not fr:
                    base1[s] = pr.eval_f(xt)
            phi1 = np.atleast_1d(opt.merit_phi(base1, Et, self.nu, np.ones(B), fr))
        phi0 = np.atleast_1d(opt.merit_phi(base, None, self.nu, np.zeros(B), fr))
        phi_pre = np.atleast_1d(opt.merit_derivative(self.nu, fr))
        for s in idx:
            phi = phi1[s] - phi0[s]
            if abs(phi_pre[s]) > 0.0:
                rho = phi / phi_pre[s]
                if rho <= 0:
                    self.delta[s] *= self.alpha1
                elif rho <= 0.25:
                    self.delta[s] *= self.alpha2
                elif rho > 0.75:
                    self.delta[s] = min(2 * self.delta[s], self.delta_max)
            else:
                rho = -phi
                if abs(phi) < 1.0e-8:
                    if fr:
                        self.fr[s] = False
                    elif self.prim_infeas[s] <= o.tol_infeas:
                        ok = self.dual_infeas[s] <= o.tol_residual and self.compl[s] <= o.tol_residual
                        self.ret[s] = 0 if ok else 6
                    else:
                        self.ret[s] = 2
            self._print(s, phi, phi_pre[s], 1.0, f"  rho {rho: .3e} delta {self.delta[s]:.3e}")
            if self.ret[s] in (0, 2, 6):
                self.running[s] = False
                continue
            if rho >= 0:
                self.x[s] = self.x[s] + self.p[s]
            self.iter[s] += 1


class _OneLp:
    """A single-LP ``external_optimizer`` -- the reference's one-LP optimizer: ``factory(n, m, j_str, x_L, x_U, g_L,
    g_U)`` with 1-D bounds, scalar results and 1-D arrays -- presented to the batch drivers as a batch of one: every
    argument loses its leading axis and every result gains one.  It has no ``set_active``: there is nothing to mask."""

    def __init__(self, factory, n, m, j_str, x_L, x_U, g_L, g_U, batch):
        self.lp = factory(n, m, j_str, x_L[0], x_U[0], g_L[0], g_U[0])

    @property
    def last_info(self):
        return self.lp.last_info

    def _call(self, name, *args):
        return getattr(self.lp, name)(*(a[0] if np.ndim(a) else a for a in args))

    def _batched(self, name, *args):
        return np.asarray(self._call(name, *args))[None]

    def update(self, *args):
        self._call("update", *args)

    def solve_extract(self):
        return tuple(np.asarray(a)[None] for a in self.lp.solve_extract())

    def norm_violations(self, *args):
        return self._batched("norm_violations", *args)

    def kt_residuals(self, *args):
        return self._batched("kt_residuals", *args)

    def norm_complementarity(self, *args):
        return self._batched("norm_complementarity", *args)

    def row_norms(self):
        return self._batched("row_norms")

    def merit_phi(self, *args):
        return self._batched("merit_phi", *args)

    def merit_derivative(self, *args):
        return self._batched("merit_derivative", *args)


class _Slp:
    """A single SLP solve of ``model`` (``SlpLS(model)`` / ``SlpTR(model)``, slp_line_search.jl:4-71,
    slp_trust_region.jl:10-80): ``run`` solves it as the one-scenario batch of ``_batch``, copies scenario 0 back
    into this object (scalars and 1-D arrays) and writes the result into the model (slp_line_search.jl:207-214).
    ``record`` (see ``_SlpBatch``) and the ``_inputs`` may be set between construction and ``run``."""

    _inputs = ("x",)

    def __init__(self, model: Model):
        self.problem = model
        self.options = model.parameters
        self.x = model.x.copy()
        self.record = None
        self.optimizer = None

    def run(self):
        pr, o = self.problem, self.options
        if o.external_optimizer != "B200LP":
            o = replace(o, external_optimizer=partial(_OneLp, o.external_optimizer))
        b = self._batch([pr], o, device_evaluator=o.device_evaluator)
        for name in self._inputs:
            getattr(b, name)[0] = getattr(self, name)
        b.record = self.record
        b.run()
        for name in self._inputs + ("p", "lam", "mult_x_U", "mult_x_L", "nu", "ret", "iter", "f", "prim_infeas",
                                    "dual_infeas", "compl", "obj_val"):
            v = getattr(b, name)[0]
            setattr(self, name, v.item() if v.ndim == 0 else v)
        self.feasibility_restoration = bool(b.fr[0])
        self.lp_log = b.lp_log[0]
        self.optimizer = b.optimizer
        pr.obj_val = self.obj_val
        pr.status = self.status = self.ret
        pr.x[:] = self.x
        pr.eval_g(self.x, pr.g)
        pr.mult_g[:] = self.lam
        pr.mult_x_U[:] = self.mult_x_U
        pr.mult_x_L[:] = self.mult_x_L
        return self


class SlpLS(_Slp):
    """Line-search SLP (slp_line_search.jl) on one model: the one-scenario ``SlpLSBatch``."""

    _batch = SlpLSBatch


class SlpTR(_Slp):
    """Trust-region SLP (slp_trust_region.jl) on one model: the one-scenario ``SlpTRBatch``, with the radius
    ``delta`` as a second input."""

    _batch = SlpTRBatch
    _inputs = ("x", "delta")

    def __init__(self, model: Model):
        super().__init__(model)
        self.delta = self.options.tr_size                                   # :62-65
