"""ctypes binding of tests/vertical_depth_oracle.c, the CPU restatement of vertical interpolation to depth levels -- TEST INFRASTRUCTURE
ONLY (tests/ and profiles/tools/vertical_depth_time.py).

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

from vertical_oracle import HERE, LIN, NN, _cc  # noqa: F401

SOURCE = os.path.join(HERE, "vertical_depth_oracle.c")
INCLUDED = os.path.join(HERE, "vertical_oracle.c")

DEPTH, OCEAN_SIGMA, OCEAN_S_G1, OCEAN_S_G2 = 3, 4, 5, 6  # FB200_VCOORD_*

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_lib = None


def library_path() -> str:
    """compile (once per version of the two sources) and return the shared library's path"""
    digest = hashlib.sha256()
    for path in (SOURCE, INCLUDED):
        with open(path, "rb") as f:
            digest.update(f.read())
    path = os.path.join(tempfile.gettempdir(), f"fimex_b200_vertical_depth_oracle_{os.getuid()}_{digest.hexdigest()[:16]}.so")
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
        lib.orc_depth_column_z.restype = None
        lib.orc_depth_column_z.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp]
        lib.orc_vinterp_depth.restype = C.c_int
        lib.orc_vinterp_depth.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_double, _dp, C.c_int, C.c_int, _fp, _fp, _fp, C.c_long,
                                          C.c_long, _fp]
        _lib = lib
    return _lib


def _terms(s, Cs):
    ss = np.ascontiguousarray(s, dtype=np.float64).ravel()
    cc = np.ascontiguousarray(Cs if Cs is not None else np.zeros(ss.size), dtype=np.float64).ravel()
    return ss, cc


def column_z(vcoord, s, Cs=None, depth_c=0.0, h=0.0, eta=0.0):
    """orc_depth_column_z: z_k [m] of one column (float64 h and eta as given; no NaN-column rules)"""
    ss, cc = _terms(s, Cs)
    z = np.empty(ss.size, dtype=np.float64)
    load().orc_depth_column_z(int(vcoord), ss.ctypes.data_as(_dp), cc.ctypes.data_as(_dp), ss.size, float(depth_c), float(h), float(eta),
                              z.ctypes.data_as(_dp))
    return z


def vinterp_depth(method, vcoord, s, Cs, levels, field, eta=None, depth=None, depth_c=0.0, extrapolate=True):
    """orc_vinterp_depth: field [nt][nk][...] -> float32 [nt][np][nxy]; eta [nt][...] (None: 0); depth [...] (None for depth levels)"""
    lev = np.ascontiguousarray(levels, dtype=np.float64).ravel()
    ss, cc = _terms(s, Cs)
    f32 = np.ascontiguousarray(field, dtype=np.float32)
    nt, nk = f32.shape[0], f32.shape[1]
    assert nk == ss.size, (nk, ss.size)
    nxy = f32.size // (nt * nk)
    e32 = None if eta is None else np.ascontiguousarray(eta, dtype=np.float32)
    d32 = None if depth is None else np.ascontiguousarray(depth, dtype=np.float32)
    out = np.empty((nt, lev.size, nxy), dtype=np.float32)
    rc = load().orc_vinterp_depth(int(method), int(vcoord), ss.ctypes.data_as(_dp), cc.ctypes.data_as(_dp), nk, float(depth_c),
                                  lev.ctypes.data_as(_dp), lev.size, int(bool(extrapolate)), f32.ctypes.data_as(_fp),
                                  None if e32 is None else e32.ctypes.data_as(_fp), None if d32 is None else d32.ctypes.data_as(_fp), nxy, nt,
                                  out.ctypes.data_as(_fp))
    if rc != 1:
        raise RuntimeError("orc_vinterp_depth failed")
    return out


# ---------------------------------------------------------------------------------------------- a synthetic ROMS-like ocean
#: the z-levels ocean forecasts are commonly delivered on [m]
DEPTHS16 = np.array([0, 3, 10, 15, 25, 50, 75, 100, 150, 200, 250, 300, 500, 1000, 2000, 3000], dtype=np.float64)


def roms_stretching(n, theta_s=7.0, theta_b=2.0, w=False):
    """s and C(s) of ROMS's Vstretching = 4 (Shchepetkin 2010), k = 0 at the sea floor: s at the n rho points (k - n - 0.5) / n,
    k = 1 .. n, or at the n + 1 w points (k - n) / n, k = 0 .. n; C_sur = (1 - cosh(theta_s s)) / (cosh(theta_s) - 1), then
    C = (exp(theta_b C_sur) - 1) / (1 - exp(-theta_b))"""
    k = np.arange(0, n + 1) if w else np.arange(1, n + 1)
    s = (k - n) / n if w else (k - n - 0.5) / n
    csur = (1.0 - np.cosh(theta_s * s)) / (np.cosh(theta_s) - 1.0)
    return s, (np.exp(theta_b * csur) - 1.0) / (1.0 - np.exp(-theta_b))


def synthetic_ocean(nx, ny, rng, land=0.3):
    """(h, eta) [ny * nx] float32, seeded: a smooth random relief of which the lowest `land` share is land (h = 0, eta NaN as ROMS's
    zeta fill value), the sea floor from 5 m at the coast to 3000 m, and a sea surface height of up to about 1.5 m"""
    x, y = np.meshgrid(np.linspace(0, 1, nx), np.linspace(0, 1, ny))
    relief = np.zeros((ny, nx))
    for _ in range(6):
        kx, ky = rng.uniform(1, 6, 2)
        relief += rng.uniform(0.3, 1) * np.sin(2 * np.pi * kx * x + rng.uniform(0, 6.3)) * np.sin(2 * np.pi * ky * y + rng.uniform(0, 6.3))
    coast = np.quantile(relief, land)
    sea = relief > coast
    d = np.clip((relief - coast) / (relief.max() - coast), 0, 1)
    h = np.where(sea, 5 + 2995 * d ** 1.5, 0.0)
    eta = np.where(sea, 1.2 * np.sin(2 * np.pi * (x + 0.3 * y)) + rng.normal(0, 0.1, (ny, nx)), np.nan)
    return h.astype(np.float32).ravel(), eta.astype(np.float32).ravel()
