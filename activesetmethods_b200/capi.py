"""ctypes binding of ``include/asm_b200.h`` (the C ABI of ``libasm_b200.so``).

This is the Python twin of the Julia ``ccall`` shim shown in INTEGRATION.md: every function below maps 1:1
onto an ``extern "C"`` entry point; nothing here computes.  The library is built in-tree by
``__graft_entry__.build()`` (``activesetmethods_b200/lib/libasm_b200.so``).  There is no fallback: if the
library is missing, or no CUDA device is visible when a handle is created, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libasm_b200.so")

OK, E_INVALID, E_CUDA, E_FREE_ROW, E_STATE = 0, -1, -2, -3, -4
LP_OPTIMAL, LP_INFEASIBLE, LP_DUAL_INFEASIBLE, LP_ITERATION_LIMIT, LP_NUMERICAL_ERROR = 0, 1, 2, 3, 4

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_int32_p = C.POINTER(C.c_int32)


class LpParams(C.Structure):
    _fields_ = [
        ("eps_rel", C.c_double), ("eps_infeas", C.c_double), ("max_iter", C.c_int64),
        ("check_every", C.c_int32), ("ruiz_iters", C.c_int32), ("warm_start", C.c_int32), ("verbose", C.c_int32),
        ("restart_sufficient", C.c_double), ("restart_necessary", C.c_double), ("restart_artificial", C.c_double),
        ("pid_kp", C.c_double), ("pid_ki", C.c_double), ("pid_kd", C.c_double),
        ("engine", C.c_int32), ("group_size", C.c_int32),
        ("hand_over", C.c_double), ("weight_balance", C.c_double), ("tiny_rel", C.c_double),
        ("ipm_max_iter", C.c_int32), ("ipm_refine", C.c_int32), ("ipm_reg", C.c_double), ("ipm_prox", C.c_double),
    ]


class LpInfo(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("restarts", C.c_int32), ("iterations", C.c_int64),
        ("objective", C.c_double), ("dual_objective", C.c_double),
        ("primal_residual", C.c_double), ("dual_residual", C.c_double), ("gap", C.c_double),
    ]


class AcopfDesc(C.Structure):
    _fields_ = [
        ("nb", C.c_int32), ("ng", C.c_int32), ("nl", C.c_int32), ("nd", C.c_int32), ("ref_bus", C.c_int32),
        ("f_bus", c_int32_p), ("t_bus", c_int32_p), ("coef", c_double_p), ("gs", c_double_p), ("bs", c_double_p),
        ("cost2", c_double_p), ("cost1", c_double_p), ("cost0", c_double_p), ("dc_loss1", c_double_p),
        ("bal_ptr", c_int32_p), ("bal_col", c_int32_p), ("bal_coef", c_double_p),
    ]


class QcqpDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("m", C.c_int32), ("nnz_coo", C.c_int64), ("c0", C.c_double),
        ("n_obj_aff", C.c_int32), ("n_obj_quad", C.c_int32),
        ("obj_aff_col", c_int32_p), ("obj_aff_coef", c_double_p),
        ("obj_quad_i", c_int32_p), ("obj_quad_j", c_int32_p), ("obj_quad_coef", c_double_p),
        ("n_aff", C.c_int64), ("n_quad", C.c_int64),
        ("aff_row", c_int32_p), ("aff_col", c_int32_p), ("aff_coef", c_double_p), ("aff_pos", c_int64_p),
        ("quad_row", c_int32_p), ("quad_i", c_int32_p), ("quad_j", c_int32_p), ("quad_coef", c_double_p),
        ("quad_pos", c_int64_p),
    ]


class AsmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"asm_b200 error {code}: {msg}")
        self.code = code


# every symbol include/asm_b200.h declares: name -> (restype, argtypes)
_VP = C.c_void_p
SIGNATURES = {
    "asm_last_error": (C.c_char_p, []),
    "asm_device_count": (C.c_int, []),
    "asm_version": (C.c_char_p, []),
    "asm_lp_default_params": (None, [C.POINTER(LpParams)]),
    "asm_lp_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, c_int64_p, c_int32_p, C.c_int32, C.c_int32,
                                C.POINTER(_VP)]),
    "asm_lp_destroy": (None, [_VP]),
    "asm_lp_set_matrix_values": (C.c_int, [_VP, c_double_p]),
    "asm_lp_set_objective": (C.c_int, [_VP, c_double_p, c_double_p]),
    "asm_lp_set_col_bounds": (C.c_int, [_VP, c_double_p, c_double_p]),
    "asm_lp_set_row_bounds": (C.c_int, [_VP, c_double_p, c_double_p]),
    "asm_lp_solve": (C.c_int, [_VP, C.POINTER(LpParams), C.POINTER(LpInfo)]),
    "asm_lp_get_primal": (C.c_int, [_VP, c_double_p]),
    "asm_lp_get_row_dual": (C.c_int, [_VP, c_double_p]),
    "asm_lp_get_col_dual": (C.c_int, [_VP, c_double_p, c_double_p]),
    "asm_lp_set_start": (C.c_int, [_VP, c_double_p, c_double_p]),
    "asm_dist_unique_id": (C.c_int, [C.c_char_p]),
    "asm_lp_dist_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, c_int64_p, c_int32_p, C.c_int32, C.c_int32,
                                     C.c_char_p, C.c_int32, C.POINTER(_VP)]),
    "asm_slp_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, c_int64_p, c_int64_p, c_double_p, c_double_p,
                                 c_double_p, c_double_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "asm_slp_destroy": (None, [_VP]),
    "asm_slp_sizes": (C.c_int, [_VP, c_int64_p, c_int32_p, c_int32_p]),
    "asm_slp_get_csr": (C.c_int, [_VP, C.c_int32, c_int64_p, c_int32_p, c_double_p]),
    "asm_slp_get_lp": (C.c_int, [_VP, C.c_int32, c_int32_p, c_int32_p, c_int64_p, c_int64_p, c_int32_p, c_double_p,
                                 c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                 c_double_p, c_double_p, c_double_p, c_int32_p]),
    "asm_slp_update": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                 C.c_int32]),
    "asm_slp_solve": (C.c_int, [_VP, C.POINTER(LpParams), C.POINTER(LpInfo)]),
    "asm_slp_extract": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_int32_p]),
    "asm_slp_sub_optimize": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                       C.c_int32, C.POINTER(LpParams), c_double_p, c_double_p, c_double_p,
                                       c_double_p, c_double_p, c_int32_p, C.POINTER(LpInfo)]),
    "asm_slp_norm_violations": (C.c_int, [_VP, c_double_p, c_double_p, C.c_int32, c_double_p]),
    "asm_slp_kt_residuals": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "asm_slp_norm_complementarity": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p]),
    "asm_slp_row_norms": (C.c_int, [_VP, c_double_p]),
    "asm_slp_merit_phi": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p, C.c_int32, c_double_p]),
    "asm_slp_merit_derivative": (C.c_int, [_VP, c_double_p, C.c_int32, c_double_p]),
    "asm_slp_attach_acopf": (C.c_int, [_VP, C.POINTER(AcopfDesc)]),
    "asm_slp_acopf_branch_coef": (C.c_int, [_VP, c_double_p]),
    "asm_slp_eval_acopf": (C.c_int, [_VP, c_double_p, c_double_p, C.c_int32]),
    "asm_slp_get_eval": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, c_double_p]),
    "asm_slp_acopf_trial": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, C.c_int32, c_double_p]),
    "asm_slp_attach_qcqp": (C.c_int, [_VP, C.POINTER(QcqpDesc)]),
    "asm_slp_eval_qcqp": (C.c_int, [_VP, c_double_p, c_double_p, C.c_int32]),
    "asm_slp_qcqp_trial": (C.c_int, [_VP, c_double_p, c_double_p, c_double_p, C.c_int32, c_double_p]),
    "asm_slp_launch_count": (C.c_int64, [_VP]),
    "asm_slp_last_solve_timing": (C.c_int, [_VP, c_double_p, c_int64_p]),
    "asm_plan_check": (C.c_int, [C.c_int32, C.c_int32, c_int64_p, c_int32_p, C.c_int32, c_int64_p, c_int32_p,
                                 c_int64_p]),
    "asm_slp_engine_info": (C.c_int, [_VP, c_int32_p, c_int32_p, c_int32_p]),
    "asm_slp_reassemble": (C.c_int, [_VP, C.c_int32]),
    "asm_slp_extract_device": (C.c_int, [_VP]),
    "asm_slp_timer_start": (C.c_int, [_VP]),
    "asm_slp_timer_stop": (C.c_int, [_VP, c_double_p]),
    "asm_slp_kernel_timing": (C.c_int, [_VP, C.c_int32, c_double_p, c_double_p]),
    "asm_slp_set_active": (C.c_int, [_VP, c_int32_p]),
    "asm_slp_load_lanes": (C.c_int, [_VP, C.c_int32, c_int32_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "asm_slp_acopf_branch_coef_lanes": (C.c_int, [_VP, C.c_int32, c_int32_p, c_double_p]),
    "asm_slp_ipm_info": (C.c_int, [_VP, c_int64_p, c_double_p]),
    "asm_slp_ipm_timing": (C.c_int, [_VP, C.c_int32, c_double_p, c_double_p]),
    "asm_kkt_selftest": (C.c_int, [C.c_int32, C.c_int32, c_int64_p, c_int32_p, c_double_p, c_double_p, c_double_p,
                                   c_double_p, c_int64_p]),
    "asm_kkt_device_selftest": (C.c_int, [C.c_int32, C.c_int32, c_int64_p, c_int32_p, C.c_int32, c_double_p,
                                          c_double_p, c_double_p, c_int32_p, c_double_p, c_double_p, C.c_int32,
                                          c_int64_p]),
}

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load ``libasm_b200.so`` and attach the prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError(f"{_LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != OK:
        raise AsmError(rc, load().asm_last_error().decode())


def dptr(a):
    """Pointer to a C-contiguous float64 array (or NULL for None)."""
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_double_p)


def as_f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def default_params(**overrides) -> LpParams:
    p = LpParams()
    load().asm_lp_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p
