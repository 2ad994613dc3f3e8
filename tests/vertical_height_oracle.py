"""ctypes binding of tests/vertical_height_oracle.c, the CPU restatement of vertical interpolation to height and altitude levels --
TEST INFRASTRUCTURE ONLY (tests/ and profiles/tools/vertical_height_time.py).

The C file includes tests/vertical_oracle.c; both are compiled on first use with the oracle's flags (gcc -std=gnu99 -O2 -ffp-contract=off
-fopenmp) into a temporary directory keyed by the sources' hash, so the repository tree is never written to.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from vertical_oracle import HERE, LIN, NN, VCOORD_HYBRID, VCOORD_PRESSURE, VCOORD_SIGMA, _cc  # noqa: F401

SOURCE = os.path.join(HERE, "vertical_height_oracle.c")
INCLUDED = os.path.join(HERE, "vertical_oracle.c")

STANDARD, HYPSOMETRIC, FIELD = 0, 1, 2  # height converters
ALTITUDE, HEIGHT = 0, 1  # height targets

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_lib = None


def library_path() -> str:
    """compile (once per version of the two sources) and return the shared library's path"""
    digest = hashlib.sha256()
    for path in (SOURCE, INCLUDED):
        with open(path, "rb") as f:
            digest.update(f.read())
    path = os.path.join(tempfile.gettempdir(), f"fimex_b200_vertical_height_oracle_{os.getuid()}_{digest.hexdigest()[:16]}.so")
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
        lib.orc_vexp.restype = C.c_double
        lib.orc_vexp.argtypes = [C.c_double]
        lib.orc_zstd.restype = C.c_double
        lib.orc_zstd.argtypes = [C.c_double]
        lib.orc_height_column_z.restype = C.c_int
        lib.orc_height_column_z.argtypes = [C.c_int, C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, _fp,
                                            _fp, _fp, _fp, _fp, _dp]
        lib.orc_vinterp_height.restype = C.c_int
        lib.orc_vinterp_height.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                                           _dp, C.c_int, C.c_int, _fp, _fp, _fp, _fp, _fp, _fp, C.c_long, C.c_long, _fp]
        _lib = lib
    return _lib


def vexp(x) -> float:
    return load().orc_vexp(float(x))


def zstd(p) -> float:
    """standard-atmosphere altitude [m] of the pressure p [hPa]"""
    return load().orc_zstd(float(p))


def _f32_or_null(a):
    return (None, None) if a is None else (lambda x: (x, x.ctypes.data_as(_fp)))(np.ascontiguousarray(a, dtype=np.float32))


def _coefficients(kind, ap, b):
    a = np.ascontiguousarray(ap if ap is not None else np.zeros(1), dtype=np.float64)
    bb = np.ascontiguousarray(b if b is not None else np.zeros(1), dtype=np.float64)
    return a, bb, (bb if kind == VCOORD_SIGMA else a).size


def height_column(converter, target, kind, ap, b, ptop=0.0, ps=None, t=None, q=None, z=None, zs=None, ps_scale=1.0, z_scale=1.0, zs_scale=1.0,
                  nk=None):
    """orc_height_column_z for one column: (coordinate of every level k [m], direction: 1 surface at k = 0, 0 at k = nk - 1, -1 NaN column)"""
    a, bb, n = _coefficients(kind, ap, b)
    nk = n if nk is None else nk
    keep = [_f32_or_null(None if v is None else np.atleast_1d(v)) for v in (ps, t, q, z, zs)]
    zc = np.empty(nk, dtype=np.float64)
    d = load().orc_height_column_z(int(converter), int(target), int(kind), a.ctypes.data_as(_dp), bb.ctypes.data_as(_dp), nk, float(ptop),
                                   float(ps_scale), float(z_scale), float(zs_scale), *[k[1] for k in keep], zc.ctypes.data_as(_dp))
    return zc, d


def vinterp_height(method, converter, target, kind, ap, b, levels, field, ps=None, t=None, q=None, z=None, zs=None, ptop=0.0, ps_scale=1.0,
                   z_scale=1.0, zs_scale=1.0, extrapolate=True):
    """orc_vinterp_height: field, t, q, z [nt][nk][...] -> float32 [nt][np][nxy]; ps [nt][...]; zs [...].  Inputs the converter does not
    use may be None; for the field converter the coefficients are not used (nk is the field's second axis)."""
    lev = np.ascontiguousarray(levels, dtype=np.float64)
    f32 = np.ascontiguousarray(field, dtype=np.float32)
    nt, nk = f32.shape[0], f32.shape[1]
    nxy = f32.size // (nt * nk)
    a, bb, _ = _coefficients(kind, ap, b)
    keep = [_f32_or_null(v) for v in (ps, t, q, z, zs)]
    out = np.empty((nt, lev.size, nxy), dtype=np.float32)
    rc = load().orc_vinterp_height(int(method), int(converter), int(target), int(kind), a.ctypes.data_as(_dp), bb.ctypes.data_as(_dp), nk,
                                   float(ptop), float(ps_scale), float(z_scale), float(zs_scale), lev.ctypes.data_as(_dp), lev.size,
                                   int(bool(extrapolate)), f32.ctypes.data_as(_fp), *[k[1] for k in keep], nxy, nt, out.ctypes.data_as(_fp))
    if rc != 1:
        raise RuntimeError("orc_vinterp_height failed")
    return out
