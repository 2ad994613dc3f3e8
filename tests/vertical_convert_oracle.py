"""ctypes binding of tests/vertical_convert_oracle.c, the CPU restatement of the vertical interpolator's data conversions (theta2T,
omega2vwind, add4Dpressure) -- TEST INFRASTRUCTURE ONLY (tests/ and profiles/tools/vertical_convert_time.py).

The C file includes tests/vertical_height_oracle.c and tests/vertical_oracle.c; all three are compiled on first use with the oracle's flags
(gcc -std=gnu99 -O2 -ffp-contract=off -fopenmp) into a temporary directory keyed by the sources' hash, so the repository tree is never
written to.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from vertical_oracle import HERE, VCOORD_HYBRID, VCOORD_PRESSURE, VCOORD_SIGMA, _cc  # noqa: F401

SOURCE = os.path.join(HERE, "vertical_convert_oracle.c")
INCLUDED = (os.path.join(HERE, "vertical_height_oracle.c"), os.path.join(HERE, "vertical_oracle.c"))

THETA2T, OMEGA2VWIND, PRESSURE = 0, 1, 2  # FB200_VCONV_*
OPS = {"theta2T": THETA2T, "omega2vwind": OMEGA2VWIND, "add4Dpressure": PRESSURE}

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_lib = None


def library_path() -> str:
    """compile (once per version of the three sources) and return the shared library's path"""
    digest = hashlib.sha256()
    for path in (SOURCE,) + INCLUDED:
        with open(path, "rb") as f:
            digest.update(f.read())
    path = os.path.join(tempfile.gettempdir(), f"fimex_b200_vertical_convert_oracle_{os.getuid()}_{digest.hexdigest()[:16]}.so")
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
        lib.orc_vconv_value.restype = C.c_double
        lib.orc_vconv_value.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double]
        lib.orc_vconvert.restype = C.c_int
        lib.orc_vconvert.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, _fp, _fp, _fp, C.c_long, C.c_long, _fp]
        lib.orc_vinterp_pressure.restype = C.c_int
        lib.orc_vinterp_pressure.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, _dp, C.c_int, C.c_int, _fp, _fp,
                                             C.c_long, C.c_long, _fp]
        _lib = lib
    return _lib


def value(op, x, T, p) -> float:
    """orc_vconv_value: one value in fp64, before the rounding to float"""
    return load().orc_vconv_value(int(op), float(x), float(T), float(p))


def _f32p(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32).ctypes.data_as(_fp)


def vconvert(op, kind, ap, b, nk, field=None, ps=None, t=None, ptop=0.0, ps_scale=1.0, nt=None, nxy=None):
    """orc_vconvert -> float32 [nt][nk][nxy].  kind: VCOORD_PRESSURE (ap = the levels), VCOORD_HYBRID (ap, b), VCOORD_SIGMA (b = sigma,
    ptop).  nt, nxy from the field, else from ps, else as given."""
    a = np.ascontiguousarray(ap if ap is not None else np.zeros(nk), dtype=np.float64)
    bb = np.ascontiguousarray(b if b is not None else np.zeros(nk), dtype=np.float64)
    f = None if field is None else np.ascontiguousarray(field, dtype=np.float32)
    p = None if ps is None else np.ascontiguousarray(ps, dtype=np.float32)
    tt = None if t is None else np.ascontiguousarray(t, dtype=np.float32)
    if f is not None:
        nt = f.shape[0]
        nxy = f.size // (nt * nk)
    elif p is not None:
        nt = p.shape[0]
        nxy = p.size // nt
    out = np.empty((nt, nk, nxy), dtype=np.float32)
    rc = load().orc_vconvert(int(op), int(kind), a.ctypes.data_as(_dp), bb.ctypes.data_as(_dp), nk, float(ptop), float(ps_scale), _f32p(f),
                             _f32p(p), _f32p(tt), nxy, nt, out.ctypes.data_as(_fp))
    if rc != 1:
        raise RuntimeError("orc_vconvert failed")
    return out


def vinterp_pressure(method, kind, ap, b, levels, field, ps=None, ptop=0.0, ps_scale=1.0, extrapolate=True):
    """orc_vinterp_pressure of the included pressure-branch restatement: field [nt][nk][...] -> float32 [nt][np][nxy]"""
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
