"""Models whose objective and rows are all affine or quadratic (QCQPs), as term lists.

The reference's MOI wrapper evaluates affine and quadratic rows inline and sends only NLP rows through the AD
evaluator (reference ``src/MOI_wrapper.jl:889-918``).  A model made of such rows alone needs no derivative code at all:
f, grad f, g and the Jacobian are sums over fixed term lists.  ``QcqpModel`` holds those lists and provides

  * the tuple the reference's ``Model`` takes (``src/model.jl:33-60``): ``n, m, x_L, x_U, g_L, g_U, j_str, x0``;
  * the four host callbacks computed from the term lists (the runs without the device evaluator, and the oracle);
  * ``qcqp_desc()``: the arrays of ``asm_qcqp_desc`` for ``SubLp.attach_qcqp``, the device-side evaluator.

Term conventions (those of ``asm_qcqp_desc``): indices are 0-based; a quadratic term is ``q * x_i * x_j`` with no 1/2
convention and ``i == j`` allowed; row r is the sum of its affine terms, then of its quadratic terms, each in the given
term order; the objective is ``c0`` plus its affine, then its quadratic terms.

``j_str`` has the reference's layout for affine and quadratic rows (``append_to_jacobian_sparsity!``,
``src/MOI_wrapper.jl:699-713``): row by row, one entry per affine term, then one per distinct variable of each
quadratic term (i, then j), duplicates allowed.  ``RandomNlp`` (``small_nlps.py``) imitates the same layout.

``random_nlp_as_qcqp`` and ``toy_qcqp`` restate two problems of ``small_nlps`` in this form.
"""
from __future__ import annotations

import numpy as np

__all__ = ["QcqpModel", "random_nlp_as_qcqp", "toy_qcqp"]


def _i(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int64).reshape(-1))


def _f(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(-1))


class QcqpModel:
    """A QCQP as term lists.

    ``n``: variables; ``x_L, x_U`` [n], ``g_L, g_U`` [m] bounds and ``x0`` [n] start.  ``obj_aff = (col, coef)``,
    ``obj_quad = (i, j, coef)``, ``aff = (row, col, coef)``, ``quad = (row, i, j, coef)``: parallel arrays, 0-based.
    Models that differ only in bounds and start (load scenarios, generator outages) share the term lists and can run
    as one batch on the device evaluator (``same_terms``)."""

    def __init__(self, n, x_L, x_U, g_L, g_U, x0, *, obj_const=0.0, obj_aff=((), ()), obj_quad=((), (), ()),
                 aff=((), (), ()), quad=((), (), (), ())):
        self.n = int(n)
        self.x_L, self.x_U = _f(x_L).copy(), _f(x_U).copy()
        self.g_L, self.g_U = _f(g_L).copy(), _f(g_U).copy()
        self.m = len(self.g_L)
        self.x0 = _f(x0).copy()
        self.c0 = float(obj_const)
        self.oa_col, self.oa_coef = _i(obj_aff[0]), _f(obj_aff[1])
        self.oq_i, self.oq_j, self.oq_coef = _i(obj_quad[0]), _i(obj_quad[1]), _f(obj_quad[2])
        self.a_row, self.a_col, self.a_coef = _i(aff[0]), _i(aff[1]), _f(aff[2])
        self.q_row, self.q_i, self.q_j, self.q_coef = _i(quad[0]), _i(quad[1]), _i(quad[2]), _f(quad[3])
        n, m = self.n, self.m
        for name, a, hi in (("obj_aff col", self.oa_col, n), ("obj_quad i", self.oq_i, n), ("obj_quad j", self.oq_j, n),
                            ("aff row", self.a_row, m), ("aff col", self.a_col, n), ("quad row", self.q_row, m),
                            ("quad i", self.q_i, n), ("quad j", self.q_j, n)):
            if len(a) and (a.min() < 0 or a.max() >= hi):
                raise ValueError(f"QcqpModel: {name} index out of range")
        if not (len(self.x_L) == len(self.x_U) == len(self.x0) == n and len(self.g_U) == m):
            raise ValueError("QcqpModel: bound / start sizes do not match n, m")
        if not (len(self.oa_col) == len(self.oa_coef) and len(self.oq_i) == len(self.oq_j) == len(self.oq_coef)
                and len(self.a_row) == len(self.a_col) == len(self.a_coef)
                and len(self.q_row) == len(self.q_i) == len(self.q_j) == len(self.q_coef)):
            raise ValueError("QcqpModel: term arrays of unequal length")
        self._build_pattern()

    # -- sparsity: the reference's layout -----------------------------------------------------------------------
    def _build_pattern(self):
        m = self.m
        diag = self.q_i == self.q_j
        # entries per row: its affine terms, then 1 or 2 per quadratic term
        per_row = np.bincount(self.a_row, minlength=m) + np.bincount(self.q_row, weights=np.where(diag, 1, 2),
                                                                     minlength=m).astype(np.int64)
        start = np.concatenate([[0], np.cumsum(per_row)])
        nnz = int(start[-1])
        fill = start[:-1].copy()
        rows = np.empty(nnz, dtype=np.int64)
        cols = np.empty(nnz, dtype=np.int64)
        self.aff_pos = np.empty(len(self.a_row), dtype=np.int64)
        self.quad_pos = np.full(2 * len(self.q_row), -1, dtype=np.int64)
        for k, (r, c) in enumerate(zip(self.a_row, self.a_col)):
            p = fill[r]; fill[r] += 1
            rows[p], cols[p] = r, c
            self.aff_pos[k] = p
        for k, (r, i, j) in enumerate(zip(self.q_row, self.q_i, self.q_j)):
            p = fill[r]; fill[r] += 1
            rows[p], cols[p] = r, i
            self.quad_pos[2 * k] = p
            if i != j:
                p = fill[r]; fill[r] += 1
                rows[p], cols[p] = r, j
                self.quad_pos[2 * k + 1] = p
        self.j_str = np.stack([rows + 1, cols + 1], 1)       # 1-based, like the reference
        self.nnz = nnz
        # derivative contributions in the evaluator's order (affine first, then quadratic in term order):
        # Jacobian entry  jac_pos <- jac_coef * x[jac_var]  (jac_var = -1: the constant jac_coef)
        off = ~diag
        qpos = np.stack([self.quad_pos[0::2], self.quad_pos[1::2]], 1)
        qcoef = np.stack([np.where(diag, 2.0 * self.q_coef, self.q_coef), self.q_coef], 1)
        qvar = np.stack([self.q_j, self.q_i], 1)
        keep = np.stack([np.ones(len(diag), dtype=bool), off], 1)
        self._jac_pos = np.concatenate([self.aff_pos, qpos[keep]])
        self._jac_coef = np.concatenate([self.a_coef, qcoef[keep]])
        self._jac_var = np.concatenate([np.full(len(self.a_row), -1), qvar[keep]])
        # gradient entry  grad_col <- grad_coef * x[grad_var]
        odiag = self.oq_i == self.oq_j
        gcol = np.stack([self.oq_i, self.oq_j], 1)
        gcoef = np.stack([np.where(odiag, 2.0 * self.oq_coef, self.oq_coef), self.oq_coef], 1)
        gvar = np.stack([self.oq_j, self.oq_i], 1)
        gkeep = np.stack([np.ones(len(odiag), dtype=bool), ~odiag], 1)
        self._grad_col = np.concatenate([self.oa_col, gcol[gkeep]])
        self._grad_coef = np.concatenate([self.oa_coef, gcoef[gkeep]])
        self._grad_var = np.concatenate([np.full(len(self.oa_col), -1), gvar[gkeep]])

    @staticmethod
    def _contrib(coef, var, x):
        return np.where(var >= 0, coef * x[np.maximum(var, 0)], coef)

    # -- callbacks (src/MOI_wrapper.jl:1047-1069) ---------------------------------------------------------------
    def eval_f(self, x):
        t = np.concatenate([self.oa_coef * x[self.oa_col], self.oq_coef * x[self.oq_i] * x[self.oq_j]])
        return float(self.c0 + np.sum(t))

    def eval_grad_f(self, x, grad):
        grad[:] = 0.0
        np.add.at(grad, self._grad_col, self._contrib(self._grad_coef, self._grad_var, x))
        return grad

    def eval_g(self, x, g):
        g[:] = 0.0
        np.add.at(g, self.a_row, self.a_coef * x[self.a_col])
        np.add.at(g, self.q_row, self.q_coef * x[self.q_i] * x[self.q_j])
        return g

    def eval_jac_g(self, x, mode, rows, cols, values):
        """``mode == "Structure"`` fills 1-based rows / cols; anything else fills ``values`` in ``j_str`` order."""
        if mode == "Structure":
            rows[:] = self.j_str[:, 0]
            cols[:] = self.j_str[:, 1]
            return
        values[:] = 0.0
        np.add.at(values, self._jac_pos, self._contrib(self._jac_coef, self._jac_var, x))
        return values

    # -- the device-side evaluator ----------------------------------------------------------------------------
    def terms(self):
        """Everything the device evaluator holds once for a batch: sizes, pattern and term lists."""
        return dict(n=self.n, m=self.m, j_str=self.j_str, c0=self.c0, oa_col=self.oa_col, oa_coef=self.oa_coef,
                    oq_i=self.oq_i, oq_j=self.oq_j, oq_coef=self.oq_coef, a_row=self.a_row, a_col=self.a_col,
                    a_coef=self.a_coef, q_row=self.q_row, q_i=self.q_i, q_j=self.q_j, q_coef=self.q_coef)

    def same_terms(self, other):
        """The name of the first field in which ``other`` differs from this model's term lists, or None."""
        a, b = self.terms(), other.terms()
        for k, v in a.items():
            if not np.array_equal(np.asarray(v), np.asarray(b[k])):
                return k
        return None

    def qcqp_desc(self):
        """The arrays of ``asm_qcqp_desc`` (int32 indices, int64 positions, float64 coefficients)."""
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)   # noqa: E731
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
        i64 = lambda a: np.ascontiguousarray(a, dtype=np.int64)   # noqa: E731
        return dict(n=self.n, m=self.m, nnz_coo=self.nnz, c0=self.c0,
                    obj_aff_col=i32(self.oa_col), obj_aff_coef=f64(self.oa_coef),
                    obj_quad_i=i32(self.oq_i), obj_quad_j=i32(self.oq_j), obj_quad_coef=f64(self.oq_coef),
                    aff_row=i32(self.a_row), aff_col=i32(self.a_col), aff_coef=f64(self.a_coef),
                    aff_pos=i64(self.aff_pos),
                    quad_row=i32(self.q_row), quad_i=i32(self.q_i), quad_j=i32(self.q_j),
                    quad_coef=f64(self.q_coef), quad_pos=i64(self.quad_pos))


def random_nlp_as_qcqp(p):
    """``small_nlps.RandomNlp`` as a ``QcqpModel``: same n, m, bounds, start and ``j_str`` (its pattern already has the
    reference's layout), 0.5 d_j x_j^2 and 0.5 Q_ij x_j^2 as quadratic terms with coefficient 0.5 d_j, 0.5 Q_ij."""
    rows, cols = np.nonzero(p.A != 0.0)
    qr, qc = np.nonzero(p.Q != 0.0)
    n = p.n
    return QcqpModel(n, p.x_L, p.x_U, p.g_L, p.g_U, p.x0,
                     obj_aff=(np.arange(n), p.c), obj_quad=(np.arange(n), np.arange(n), 0.5 * p.d),
                     aff=(rows, cols, p.A[rows, cols]), quad=(qr, qc, qc, 0.5 * p.Q[qr, qc]))


def toy_qcqp():
    """``small_nlps.ToyNlp`` (reference ``test/ext_solver.jl:13-19``) as a ``QcqpModel``:
    min X^2 + X  s.t.  X >= -2,  X^2 - X == 2,  X*Y == 1,  X*Y >= 0  ->  X = Y = -1."""
    inf = np.inf
    return QcqpModel(2, [-inf, -inf], [inf, inf], [-2.0, 2.0, 1.0, 0.0], [inf, 2.0, 1.0, inf], np.zeros(2),
                     obj_aff=([0], [1.0]), obj_quad=([0], [0], [1.0]),
                     aff=([0, 1], [0, 0], [1.0, -1.0]),
                     quad=([1, 2, 3], [0, 0, 0], [0, 1, 1], [1.0, 1.0, 1.0]))
