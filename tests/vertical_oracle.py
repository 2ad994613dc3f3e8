"""ctypes binding of tests/vertical_oracle.c, the CPU restatement of vertical interpolation to pressure levels -- TEST
INFRASTRUCTURE ONLY (tests/ and profiles/tools/vertical_time.py).

The C file is compiled on first use with the oracle's flags (gcc -std=gnu99 -O2 -ffp-contract=off -fopenmp) into a temporary
directory keyed by the source's hash, so the repository tree is never written to.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.path.join(HERE, "vertical_oracle.c")

LIN, LOG, LOGLOG, NN = 0, 1, 2, 3  # MIFI_VINT_METHOD_*
VCOORD_PRESSURE, VCOORD_HYBRID, VCOORD_SIGMA = 0, 1, 2

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_lib = None


def _cc() -> str:
    return "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else (shutil.which("gcc") or "cc")


def library_path() -> str:
    """compile (once per source version) and return the shared library's path"""
    with open(SOURCE, "rb") as f:
        digest = hashlib.sha256(f.read()).hexdigest()[:16]
    path = os.path.join(tempfile.gettempdir(), f"fimex_b200_vertical_oracle_{os.getuid()}_{digest}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([_cc(), "-std=gnu99", "-O2", "-ffp-contract=off", "-fPIC", "-fopenmp", "-Wall", SOURCE, "-o", tmp, "-shared", "-lm"],
                       check=True, capture_output=True)
        os.replace(tmp, path)  # atomic: concurrent test processes see a whole library or none
    return path


def load():
    global _lib
    if _lib is None:
        lib = C.CDLL(library_path())
        lib.orc_vinterp_pressure.restype = C.c_int
        lib.orc_vinterp_pressure.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, _dp, C.c_int, C.c_int, _fp, _fp,
                                             C.c_long, C.c_long, _fp]
        lib.orc_vint_values.restype = None
        lib.orc_vint_values.argtypes = [C.c_int, _fp, _fp, _fp, C.c_size_t, C.c_double, C.c_double, C.c_double]
        lib.orc_vlog.restype = C.c_double
        lib.orc_vlog.argtypes = [C.c_double]
        _lib = lib
    return _lib


def vinterp(method, kind, ap, b, levels, field, ps=None, ptop=0.0, ps_scale=1.0, extrapolate=True):
    """orc_vinterp_pressure: field [nt][nk][...] -> float32 [nt][np][nxy]; ps [nt][...].
    kind: VCOORD_PRESSURE (ap = the levels), VCOORD_HYBRID (ap, b) or VCOORD_SIGMA (b = sigma, ptop)."""
    lev = np.ascontiguousarray(levels, dtype=np.float64)
    a = np.ascontiguousarray(ap if ap is not None else np.zeros(1), dtype=np.float64)
    bb = np.ascontiguousarray(b if b is not None else np.zeros(1), dtype=np.float64)
    nk = (bb if kind == VCOORD_SIGMA else a).size
    f32 = np.ascontiguousarray(field, dtype=np.float32)
    nt = f32.shape[0]
    nxy = f32.size // (nt * nk)
    p32 = np.ascontiguousarray(ps if ps is not None else np.zeros(nt * nxy), dtype=np.float32)
    out = np.empty((nt, lev.size, nxy), dtype=np.float32)
    rc = load().orc_vinterp_pressure(int(method), int(kind), a.ctypes.data_as(_dp), bb.ctypes.data_as(_dp), nk, float(ptop), float(ps_scale),
                                     lev.ctypes.data_as(_dp), lev.size, int(bool(extrapolate)), f32.ctypes.data_as(_fp), p32.ctypes.data_as(_fp),
                                     nxy, nt, out.ctypes.data_as(_fp))
    if rc != 1:
        raise RuntimeError("orc_vinterp_pressure failed")
    return out


def vint_values(method, A, B, a, b, x):
    """orc_vint_values: the two-level step with the argument list of mifi_get_values_linear_f (a, b, x: pressures)"""
    aa = np.ascontiguousarray(A, dtype=np.float32)
    bb = np.ascontiguousarray(B, dtype=np.float32)
    out = np.empty(aa.size, dtype=np.float32)
    load().orc_vint_values(int(method), aa.ctypes.data_as(_fp), bb.ctypes.data_as(_fp), out.ctypes.data_as(_fp), aa.size, float(a), float(b),
                           float(x))
    return out


def vlog(x) -> float:
    return load().orc_vlog(float(x))
