"""An independent CPU reference of forward interpolation (CachedForwardInterpolation, swath points to a grid) -- TEST
INFRASTRUCTURE ONLY.

Written from the reference's per-cell definitions, not from oracle/mifi_oracle.c:
  * bucket      RoundAndClamp (Utils.cc:42-58): round half away from zero, then -1 outside [0, max] or for NaN.  Written
                as trunc + an explicit test of the exact fractional part, because np.round rounds half to even and
                trunc(x + copysign(0.5, x)) rounds 0.49999999999999994 up.  A point belongs to a cell only when both of
                its indices are valid; each cell keeps its points in input (row-major) order.
  * values      forward_* drop NaN values, forward_undef_* keep them (CachedForwardInterpolation.cc:99-115).
  * sum / mean  std::accumulate(v, 0.f): a sequential float32 sum (np.add.accumulate is sequential), then / float(count).
  * max / min   std::max_element / std::min_element: the first extreme under operator<.
  * median      std::nth_element(v.begin(), v.begin() + n/2, v.end()); v[n/2] -- the C++ library's own nth_element,
                through tests/forward_reference_nth.cc, compiled on first use into a temporary directory.
An empty cell is NaN.  The module also holds the comparison rule and the seeded case generator of the forward tests.
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
SOURCE = os.path.join(HERE, "forward_reference_nth.cc")

(FORWARD_SUM, FORWARD_MEAN, FORWARD_MEDIAN, FORWARD_MAX, FORWARD_MIN, FORWARD_UNDEF_SUM, FORWARD_UNDEF_MEAN, FORWARD_UNDEF_MEDIAN,
 FORWARD_UNDEF_MAX, FORWARD_UNDEF_MIN) = range(5, 15)
METHODS = tuple(range(5, 15))
ARITHMETIC = (FORWARD_SUM, FORWARD_MEAN, FORWARD_UNDEF_SUM, FORWARD_UNDEF_MEAN)
MEDIANS = (FORWARD_MEDIAN, FORWARD_UNDEF_MEDIAN)
UNDEF_F = np.array([0x7FC00000], dtype=np.uint32).view(np.float32)[0]  # MIFI_UNDEFINED_F

_fp = C.POINTER(C.c_float)
_lib = None


def _cxx() -> str:
    return "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else (shutil.which("g++") or "c++")


def library_path() -> str:
    """compile (once per source version) and return the shared library's path"""
    with open(SOURCE, "rb") as f:
        digest = hashlib.sha256(f.read()).hexdigest()[:16]
    path = os.path.join(tempfile.gettempdir(), f"fimex_b200_forward_nth_{os.getuid()}_{digest}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([_cxx(), "-O2", "-fPIC", "-Wall", SOURCE, "-o", tmp, "-shared"], check=True, capture_output=True)
        os.replace(tmp, path)  # atomic: concurrent test processes see a whole library or none
    return path


def _load():
    global _lib
    if _lib is None:
        lib = C.CDLL(library_path())
        lib.ref_nth_element.restype = None
        lib.ref_nth_element.argtypes = [_fp, C.c_size_t, C.c_size_t]
        _lib = lib
    return _lib


def nth_element(values, nth):
    """std::nth_element(v, v + nth, v + n) on a float32 copy; returns the rearranged copy"""
    v = np.array(values, dtype=np.float32, copy=True)
    if v.size:
        _load().ref_nth_element(v.ctypes.data_as(_fp), int(nth), v.size)
    return v


def round_and_clamp(pos, maxi):
    """RoundAndClamp: index of the nearest cell, half away from zero; -1 outside [0, maxi] and for NaN / inf"""
    p = np.asarray(pos, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        t = np.trunc(p)
        r = t + np.where(np.abs(p - t) >= 0.5, np.copysign(1.0, p), 0.0)
        ok = np.isfinite(r) & (r >= 0) & (r <= maxi)
    return np.where(ok, r, -1).astype(np.int64)


def aggregate(method, v):
    """one cell's aggregate of its (already filtered) values in input order; v is a float32 array with at least one value"""
    if method in ARITHMETIC:
        with np.errstate(invalid="ignore"):  # inf + -inf
            s = np.add.accumulate(np.concatenate([np.zeros(1, np.float32), v]))[-1]
        if method in (FORWARD_MEAN, FORWARD_UNDEF_MEAN):
            s = np.float32(s / np.float32(v.size))
        return np.float32(s)
    if method in MEDIANS:
        return nth_element(v, v.size // 2)[v.size // 2]
    best = v[0]
    is_max = method in (FORWARD_MAX, FORWARD_UNDEF_MAX)
    for x in v[1:]:
        if (best < x) if is_max else (x < best):
            best = x
    return best


def forward(method, px, py, outX, outY, data):
    """CachedForwardInterpolation::interpolateValues: data [nz][inY][inX] (or [nz][n]) -> float32 [nz][outY][outX]"""
    xi = round_and_clamp(px, outX - 1)
    yi = round_and_clamp(py, outY - 1)
    n = xi.size
    d = np.ascontiguousarray(data, dtype=np.float32).reshape(-1, n)
    cell = np.where((xi >= 0) & (yi >= 0), yi * outX + xi, -1)
    mapped = np.flatnonzero(cell >= 0)
    order = mapped[np.argsort(cell[mapped], kind="stable")]  # stable: input order inside a cell
    sorted_cells = cell[order]
    bounds = np.searchsorted(sorted_cells, np.arange(outX * outY + 1))
    undef = method >= FORWARD_UNDEF_SUM
    out = np.full((d.shape[0], outX * outY), UNDEF_F, dtype=np.float32)
    for z in range(d.shape[0]):
        lv = d[z]
        for c in np.flatnonzero(np.diff(bounds)):
            v = lv[order[bounds[c]:bounds[c + 1]]]
            if not undef:
                v = v[~np.isnan(v)]
            if v.size:
                out[z, c] = aggregate(method, v)
    return out.reshape(d.shape[0], outY, outX)


def assert_forward_equal(got, want, method, what="", nan_payload=None):
    """Bit for bit, signed zeros included.  NaN bit patterns must match too, except where the aggregate is computed
    arithmetically (sum, mean: x86 keeps an operand's payload, NVIDIA GPUs return 0x7fffffff) -- or wherever nan_payload
    is False."""
    a = np.ascontiguousarray(got, dtype=np.float32).ravel()
    b = np.ascontiguousarray(want, dtype=np.float32).ravel()
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if nan_payload is None:
        nan_payload = method not in ARITHMETIC
    differ = a.view(np.uint32) != b.view(np.uint32)
    if not nan_payload:
        differ &= ~(np.isnan(a) & np.isnan(b))
    bad = np.flatnonzero(differ)
    assert bad.size == 0, (f"{what}: method {method}: {bad.size} of {a.size} values differ; first at {bad[:5]}: "
                           f"{a[bad[:5]].view(np.uint32)} vs {b[bad[:5]].view(np.uint32)}")


# ------------------------------------------------------------------------------------------------- the seeded case generator
_NANS = np.array([0x7FC00000, 0xFFC00000, 0x7FC00001, 0x7FA00000], dtype=np.uint32).view(np.float32)  # quiet NaNs, both signs


def _positions(rng, n, size, layout):
    if layout == "uniform":
        p = rng.uniform(-0.5, size - 0.5, n)
    elif layout == "clustered":  # a few cells receive everything
        centres = rng.integers(0, size, rng.integers(1, 4))
        p = centres[rng.integers(0, centres.size, n)] + rng.uniform(-0.45, 0.45, n)
    else:  # "overhang": over every edge
        p = rng.uniform(-3.0, size + 2.0, n)
    k = rng.random(n)
    p[k < 0.08] = np.round(p[k < 0.08] * 2) / 2  # x.5 ties: half away from zero
    p[(k >= 0.08) & (k < 0.10)] = np.nan
    p[(k >= 0.10) & (k < 0.11)] = rng.choice([1e12, -1e12, 3e9, -3e9, np.inf, -np.inf], ((k >= 0.10) & (k < 0.11)).sum())
    return p


def _values(rng, shape, nan_density):
    kind = rng.integers(0, 3)
    if kind == 0:
        v = rng.normal(10, 5, shape).astype(np.float32)
    elif kind == 1:  # repeats and both signs of zero
        v = rng.choice(np.array([-0.0, 0.0, 1.0, 2.0, -1.0], dtype=np.float32), shape)
    else:
        v = rng.normal(0, 1, shape).astype(np.float32)
        v[rng.random(shape) < 0.3] = rng.choice(np.array([-0.0, 0.0, 3.0], dtype=np.float32), 1)[0]
    nan = rng.random(shape) < nan_density
    v[nan] = rng.choice(_NANS, nan.sum())
    return v


def make_case(seed):
    """one forward case: dict(method, inX, inY, outX, outY, nz, px, py, data [nz][inY][inX] float32)"""
    rng = np.random.default_rng(seed)
    method = int(rng.choice(METHODS))
    inX, inY = int(rng.integers(1, 90)), int(rng.integers(1, 40))
    shape_kind = rng.integers(0, 4)
    if shape_kind == 0:  # fewer than four cells
        outX, outY = int(rng.integers(1, 4)), 1
    elif shape_kind == 1:  # a power-of-two cell count: the radix sort's end_bit
        e = int(rng.integers(1, 9))
        outX = 1 << int(rng.integers(0, e + 1))
        outY = (1 << e) // outX
    else:
        outX, outY = int(rng.integers(1, 70)), int(rng.integers(1, 40))
    nz = int(rng.choice([1, 2, 3, 4, 5, 7, 11]))
    layout = str(rng.choice(["uniform", "clustered", "overhang"]))
    n = inX * inY
    px = _positions(rng, n, outX, layout)
    py = _positions(rng, n, outY, layout)
    if rng.random() < 0.05:
        px[:] = -7.0  # nothing mapped
    data = _values(rng, (nz, inY, inX), float(rng.choice([0.0, 0.01, 0.3])))
    return dict(method=method, inX=inX, inY=inY, outX=outX, outY=outY, nz=nz, px=px, py=py, data=data)
