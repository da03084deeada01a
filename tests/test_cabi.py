"""The C-ABI library loads and exports every symbol include/ghost_cwt.h declares.
No compute calls: there is no GPU in the build container."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from ghost_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "ghost_cwt.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gcwt_[a-z_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_lib.EXPORTS) == names
    assert lib.gcwt_version() == 200


def test_constants_match_header():
    text = open(os.path.join(ROOT, "include", "ghost_cwt.h")).read()
    defs = dict(re.findall(r"#define\s+(GCWT_[A-Z0-9_]+)\s+(-?\d+)", text))
    assert int(defs["GCWT_F32"]) == _lib.F32 and int(defs["GCWT_F64"]) == _lib.F64
    assert int(defs["GCWT_OUT_COMPLEX"]) == _lib.OUT_COMPLEX
    assert int(defs["GCWT_OUT_AMPLITUDE"]) == _lib.OUT_AMPLITUDE
    assert int(defs["GCWT_OUT_POWER"]) == _lib.OUT_POWER
    assert int(defs["GCWT_FLAG_FORCE_GENERIC"]) == _lib.FLAG_FORCE_GENERIC
    assert int(defs["GCWT_FLAG_NO_INTERP"]) == _lib.FLAG_NO_INTERP
    assert int(defs["GCWT_FLAG_NO_GUARD"]) == _lib.FLAG_NO_GUARD
    for name in ("FULL", "BANDED", "INTERP", "WIDE2"):
        assert int(defs["GCWT_KERNEL_" + name]) == getattr(_lib, "KERNEL_" + name)


def test_class_info_layout_matches_header():
    text = open(os.path.join(ROOT, "include", "ghost_cwt.h")).read()
    body = re.search(r"typedef struct gcwt_class_info \{(.*?)\} gcwt_class_info;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"(int32_t|int64_t)\s+(\w+);", body)
    ctypes_of = {"int32_t": C.c_int32, "int64_t": C.c_int64}
    assert [(n, ctypes_of[t]) for t, n in fields] == list(_lib.ClassInfo._fields_)
    assert C.sizeof(_lib.ClassInfo) == 40


def test_plan_classes_null_arguments():
    lib = _lib.load()
    n = C.c_int32(7)
    assert lib.gcwt_plan_classes(None, C.byref(n), None, None) == -1
    assert b"NULL" in lib.gcwt_last_error()
    assert n.value == 7
    assert lib.gcwt_plan_classes(None, None, None, None) == -1


def test_argument_errors_without_device():
    lib = _lib.load()
    handle = C.c_void_p()
    assert lib.gcwt_plan_create(C.byref(handle), None) == -1
    assert b"NULL" in lib.gcwt_last_error()
    desc = _lib.PlanDesc()
    desc.n_scales = 0
    assert lib.gcwt_plan_create(C.byref(handle), C.byref(desc)) == -1
    assert lib.gcwt_plan_destroy(None) == 0


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from ghost_b200 import ContinuousWaveletTransform
    with pytest.raises(_lib.GcwtError, match="no CUDA device"):
        ContinuousWaveletTransform().transform(np.zeros(4000), fs=1000.0)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "ghost_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("cwt_oracle", "oracle") or f == "never", (dirpath, f)


@pytest.mark.parametrize("log2u,T,os_,bound", [(4, 8, 4.0, 5e-6), (6, 8, 5.0, 1e-6), (2, 12, 2.5, 3e-6),
                                               (3, 12, 2.5, 3e-6), (1, 8, 4.0, 5e-6), (10, 8, 4.0, 5e-6)])
def test_interpolator_design_worst_case_bound(log2u, T, os_, bound):
    """Host-side design used on the amplitude / power paths (csrc/fast_path.cu design_interpolator):
    least-squares fractional delay over the band |W|^2 can occupy.  The bound holds for EVERY tone in
    that band (two-tone beats at the band edge included), not just for typical spectra."""
    lib = _lib.load()
    U = 1 << log2u
    taps = np.zeros((U, T), dtype=np.float32)
    rc = lib.gcwt_interp_taps(log2u, T, os_, taps.ctypes.data_as(C.POINTER(C.c_float)))
    assert rc == 0
    assert np.allclose(taps.sum(axis=1), 1.0, atol=2e-6)       # exact DC gain
    assert np.allclose(taps[0], np.eye(T)[T // 2 - 1], atol=1e-6)   # phase 0 copies the coarse sample
    phis = range(U) if U <= 64 else range(0, U, U // 64)
    sub = taps[list(phis)]
    worst = 0.0
    f = np.linspace(0.0, 0.5 / os_, 300)
    t = np.arange(T)
    for row, phi in zip(sub, phis):
        d = (t - (T // 2 - 1)) - phi / U
        resp = (row[None, :].astype(np.float64) * np.exp(2j * np.pi * f[:, None] * d[None, :])).sum(axis=1)
        worst = max(worst, float(np.abs(resp - 1.0).max()))
    assert worst <= bound, worst


def test_interpolator_design_rejects_bad_arguments():
    lib = _lib.load()
    buf = (C.c_float * 64)()
    assert lib.gcwt_interp_taps(2, 7, 4.0, buf) == -1          # odd tap count
    assert lib.gcwt_interp_taps(2, 8, 0.5, buf) == -1          # under-sampled
    assert lib.gcwt_interp_taps(2, 8, 4.0, None) == -1
