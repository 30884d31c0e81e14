"""The C-ABI library builds, loads and exports every symbol include/asm_b200.h declares (CPU: no compute)."""
import ctypes as C
import os
import re

import pytest

from activesetmethods_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "asm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(asm_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(built_lib):
    syms = header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(built_lib, s), f"{s} declared in include/asm_b200.h but not exported"
    assert sorted(capi.SIGNATURES) == syms, "capi.SIGNATURES and the header disagree"


def test_default_params(built_lib):
    p = capi.default_params()
    assert p.eps_rel == 1e-8 and p.check_every == 64 and p.max_iter == 2000000
    assert C.sizeof(capi.LpParams) == 8 * 2 + 8 + 4 * 4 + 8 * 6 + 8 * 4 + 4 * 2 + 8 * 2
    assert p.ipm_max_iter == 200 and p.ipm_refine == 0 and p.ipm_reg == 1e-8 and p.ipm_prox == 1e-7
    assert C.sizeof(capi.LpInfo) == 4 + 4 + 8 + 8 * 5


def test_no_cpu_fallback(built_lib):
    """Without a device, creating a handle fails loudly (ASM_E_CUDA) instead of computing on the host."""
    if built_lib.asm_device_count() > 0:
        pytest.skip("a GPU is present")
    from activesetmethods_b200.sublp import SubLp
    import numpy as np
    with pytest.raises(capi.AsmError) as e:
        SubLp(2, 1, np.array([[1, 1], [1, 2]]), [-1, -1], [1, 1], [0.0], [0.0])
    assert e.value.code == capi.E_CUDA


def test_kkt_device_selftest_arguments(built_lib):
    """The device self test rejects bad arguments before it looks for a device, and without one it fails with
    ASM_E_CUDA: its host twin is asm_kkt_selftest, not a fallback."""
    import numpy as np
    i64, i32, d = capi.c_int64_p, capi.c_int32_p, capi.dptr
    rp = np.array([0, 2, 3], dtype=np.int64)
    ci = np.array([0, 2, 1], dtype=np.int32)
    vals, dx, ew = np.ones(3), np.ones(3), np.ones(2)
    sol, stats = np.zeros(5), np.zeros(10, dtype=np.int64)

    def call(n=3, m=2, rp=rp, ci=ci, batch=1, vals=vals, dx=dx, ew=ew, sol=sol, device=0):
        return built_lib.asm_kkt_device_selftest(
            n, m, None if rp is None else rp.ctypes.data_as(i64), None if ci is None else ci.ctypes.data_as(i32),
            batch, d(vals), d(dx), d(ew), None, d(sol), None, device, stats.ctypes.data_as(i64))

    bad = [dict(n=0), dict(m=-1), dict(batch=0), dict(rp=None), dict(ci=None), dict(vals=None), dict(dx=None),
           dict(ew=None), dict(sol=None), dict(rp=np.array([1, 2, 3], dtype=np.int64)),
           dict(rp=np.array([0, 3, 2], dtype=np.int64)), dict(ci=np.array([0, 3, 1], dtype=np.int32)),
           dict(ci=np.array([0, -1, 1], dtype=np.int32))]
    for kw in bad:
        assert call(**kw) == capi.E_INVALID, kw
    if built_lib.asm_device_count() > 0:
        assert call(device=-1) == capi.E_INVALID
    else:
        assert call() == capi.E_CUDA
        assert call(device=-1) == capi.E_CUDA


def test_slp_get_lp_arguments(built_lib):
    """asm_slp_get_lp rejects a null handle without touching a device; with a device, a scenario outside [0, batch),
    a read before the first update and a read of the solution before a solve are refused too."""
    import numpy as np
    i32, i64 = capi.c_int32_p, capi.c_int64_p
    cols, rows, st = np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int32)
    nnz = np.zeros(1, np.int64)
    buf = np.zeros(64)

    def call(h, s, x=None, status=None):
        return built_lib.asm_slp_get_lp(h, s, cols.ctypes.data_as(i32), rows.ctypes.data_as(i32),
                                        nnz.ctypes.data_as(i64), None, None, None, None, None, None, None, None, None,
                                        capi.dptr(x), None, None, None, None if status is None else status.ctypes.data_as(i32))

    for s in (-1, 0, 1):
        assert call(None, s) == capi.E_INVALID
        assert call(None, s, x=buf, status=st) == capi.E_INVALID
    if built_lib.asm_device_count() == 0:
        return
    from activesetmethods_b200.sublp import SubLp
    lp = SubLp(2, 1, np.array([[1, 1], [1, 2]]), [-1, -1], [1, 1], [0.0], [1.0], batch=3)
    for s in (-1, 3, 64):
        assert call(lp._h, s) == capi.E_INVALID
    assert call(lp._h, 0) == capi.E_STATE
    lp.update(np.zeros((3, 2)), np.zeros(3), np.ones((3, 2)), np.zeros((3, 1)), np.ones((3, 2)), 1.0)
    assert call(lp._h, 2) == capi.OK and (cols[0], rows[0], nnz[0]) == (2, 1, 2)
    assert call(lp._h, 2, x=buf) == capi.E_STATE and call(lp._h, 2, status=st) == capi.E_STATE
    lp.close()


def test_product_does_not_import_oracle():
    """Only tests/, smoke() and bench.py's cpu_baseline may touch oracle/."""
    pkg = os.path.join(ROOT, "activesetmethods_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(d, f)).read()
                assert "slp_oracle" not in src and "import oracle" not in src and "from oracle" not in src, f
