"""ctypes bindings for the CPU oracle -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this
module.  Nothing under fimex_b200/ does; the product path fails loudly without its CUDA library.

Two libraries:
  * ``Oracle``    = oracle/liboracle.so, the restatement (mifi_oracle.c + pj_oracle.c); always available
                    after ``make -C oracle``.
  * ``Reference`` = oracle/_ref/libmifi_ref.so, the reference's own src/interpolation.c compiled
                    unmodified (``make -C oracle ref``; needs /root/reference at build time only).
Both expose the same Python surface so a test can run one against the other.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libmifi_ref.so")

MIFI_OK, MIFI_ERROR = 1, -1
PROJ_AXIS, LONGITUDE, LATITUDE = 0, 1, 2
(NEAREST_NEIGHBOR, BILINEAR, BICUBIC, COORD_NN, COORD_NN_KD, FORWARD_SUM, FORWARD_MEAN, FORWARD_MEDIAN, FORWARD_MAX,
 FORWARD_MIN, FORWARD_UNDEF_SUM, FORWARD_UNDEF_MEAN, FORWARD_UNDEF_MEDIAN, FORWARD_UNDEF_MAX, FORWARD_UNDEF_MIN) = range(15)

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)


def build(ref: bool = True) -> None:
    """Compile the restatement and, when /root/reference is present, the reference itself."""
    subprocess.run(["make", "-C", HERE, "all"], check=True, capture_output=True)
    if ref and os.path.isdir("/root/reference"):
        subprocess.run(["make", "-C", HERE, "ref"], check=True, capture_output=True)


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(_fp)


class _Base:
    prefix = ""
    names: dict = {}

    def __init__(self, path):
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle` (and `make -C oracle ref` here)")
        self.lib = C.CDLL(path)

    def fn(self, key):
        return getattr(self.lib, self.names[key])

    # ---- scalar kernels ------------------------------------------------------------------------
    def points2position(self, points, axis, axis_type):
        pts, pp = _d(np.array(points, dtype=np.float64, copy=True))
        ax, ap = _d(axis)
        f = self.fn("points2position")
        f.restype = None if self.prefix == "orc_" else C.c_int
        if self.prefix == "orc_":
            f.argtypes = [_dp, C.c_long, _dp, C.c_int, C.c_int]
        else:
            f.argtypes = [_dp, C.c_int, _dp, C.c_int, C.c_int]
        f(pp, pts.size, ap, ax.size, axis_type)
        return pts

    def get_values(self, method, infield, x, y, ix, iy, iz):
        key = {NEAREST_NEIGHBOR: "get_values_nn", BILINEAR: "get_values_bilinear", BICUBIC: "get_values_bicubic"}[method]
        f = self.fn(key)
        f.argtypes = [_fp, _fp, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int]
        a, ap = _f(infield)
        out = np.empty(iz, dtype=np.float32)
        f(ap, out.ctypes.data_as(_fp), float(x), float(y), ix, iy, iz)
        return out

    def project_axes(self, proj_in, proj_out, xax, yax):
        xa, xp = _d(xax)
        ya, yp = _d(yax)
        n = xa.size * ya.size
        xo = np.empty(n)
        yo = np.empty(n)
        f = self.fn("project_axes")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p, C.c_char_p, _dp, _dp, C.c_int, C.c_int, _dp, _dp]
        rc = f(proj_in.encode(), proj_out.encode(), xp, yp, xa.size, ya.size, xo.ctypes.data_as(_dp), yo.ctypes.data_as(_dp))
        return rc, xo, yo

    def project_values(self, proj_in, proj_out, x, y):
        xa, xp = _d(np.array(x, dtype=np.float64, copy=True))
        ya, yp = _d(np.array(y, dtype=np.float64, copy=True))
        f = self.fn("project_values")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p, C.c_char_p, _dp, _dp, C.c_long if self.prefix == "orc_" else C.c_int]
        rc = f(proj_in.encode(), proj_out.encode(), xp, yp, xa.size)
        return rc, xa, ya

    def interpolate_f(self, method, proj_in, infield, in_x, in_y, in_xt, in_yt, iz, proj_out, out_x, out_y, out_xt, out_yt,
                      out_init=None):
        a, ap = _f(infield)
        ix, iy = len(in_x), len(in_y)
        ox, oy = len(out_x), len(out_y)
        out = np.full(ox * oy * iz, np.nan, dtype=np.float32) if out_init is None else np.array(out_init, dtype=np.float32, copy=True)
        ixa, ixp = _d(in_x)
        iya, iyp = _d(in_y)
        oxa, oxp = _d(out_x)
        oya, oyp = _d(out_y)
        f = self.fn("interpolate_f")
        f.restype = C.c_int
        f.argtypes = [C.c_int, C.c_char_p, _fp, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, _fp, _dp, _dp,
                      C.c_int, C.c_int, C.c_int, C.c_int]
        rc = f(method, proj_in.encode(), ap, ixp, iyp, in_xt, in_yt, ix, iy, iz, proj_out.encode(), out.ctypes.data_as(_fp), oxp,
               oyp, out_xt, out_yt, ox, oy)
        return rc, out.reshape(iz, oy, ox)

    def vector_matrix(self, proj_in, proj_out, out_x, out_y, xt, yt):
        oxa, oxp = _d(out_x)
        oya, oyp = _d(out_y)
        m = np.empty(4 * oxa.size * oya.size)
        f = self.fn("vector_matrix")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p, C.c_char_p, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, _dp]
        rc = f(proj_in.encode(), proj_out.encode(), oxp, oyp, xt, yt, oxa.size, oya.size, m.ctypes.data_as(_dp))
        return rc, m

    def vector_matrix_field(self, proj_in, proj_out, in_x_field, in_y_field, ox, oy):
        xa, xp = _d(in_x_field)
        ya, yp = _d(in_y_field)
        m = np.empty(4 * ox * oy)
        f = self.fn("vector_matrix_field")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p, C.c_char_p, _dp, _dp, C.c_int, C.c_int, _dp]
        rc = f(proj_in.encode(), proj_out.encode(), xp, yp, ox, oy, m.ctypes.data_as(_dp))
        return rc, m

    def vector_matrix_points(self, proj_in, proj_out, metric, x, y):
        xa, xp = _d(x)
        ya, yp = _d(y)
        m = np.empty(4 * xa.size)
        f = self.fn("vector_matrix_points")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p, C.c_char_p, C.c_int, _dp, _dp, C.c_int, _dp]
        rc = f(proj_in.encode(), proj_out.encode(), int(metric), xp, yp, xa.size, m.ctypes.data_as(_dp))
        return rc, m

    def vector_reproject_by_matrix(self, matrix, u, v, ox, oy, oz):
        m, mp = _d(matrix)
        uu, up = _f(np.array(u, dtype=np.float32, copy=True))
        vv, vp = _f(np.array(v, dtype=np.float32, copy=True))
        f = self.fn("vector_reproject_by_matrix")
        if self.prefix == "orc_":
            f.restype = None
            f.argtypes = [_dp, _fp, _fp, C.c_int, C.c_int, C.c_int]
            f(mp, up, vp, ox, oy, oz)
        else:
            f.restype = C.c_int
            f.argtypes = [C.c_int, _dp, _fp, _fp, C.c_int, C.c_int, C.c_int]
            f(0, mp, up, vp, ox, oy, oz)
        return uu, vv

    def vector_reproject_direction(self, matrix, angles, ox, oy, oz):
        m, mp = _d(matrix)
        aa, ap = _f(np.array(angles, dtype=np.float32, copy=True))
        f = self.fn("vector_reproject_direction")
        if self.prefix == "orc_":
            f.restype = None
            f.argtypes = [_dp, _fp, C.c_int, C.c_int, C.c_int]
            f(mp, ap, ox, oy, oz)
        else:
            f.restype = C.c_int
            f.argtypes = [C.c_int, _dp, _fp, C.c_int, C.c_int, C.c_int]
            f(0, mp, ap, ox, oy, oz)
        return aa

    def vector_reproject_values(self, proj_in, proj_out, u, v, out_x, out_y, xt, yt, oz):
        oxa, oxp = _d(out_x)
        oya, oyp = _d(out_y)
        uu, up = _f(np.array(u, dtype=np.float32, copy=True))
        vv, vp = _f(np.array(v, dtype=np.float32, copy=True))
        f = self.fn("vector_reproject_values")
        f.restype = C.c_int
        if self.prefix == "orc_":
            f.argtypes = [C.c_char_p, C.c_char_p, _fp, _fp, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
            rc = f(proj_in.encode(), proj_out.encode(), up, vp, oxp, oyp, xt, yt, oxa.size, oya.size, oz)
        else:
            f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, _fp, _fp, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
            rc = f(0, proj_in.encode(), proj_out.encode(), up, vp, oxp, oyp, xt, yt, oxa.size, oya.size, oz)
        return rc, uu, vv

    def string_to_method(self, s):
        f = self.fn("string_to_method")
        f.restype = C.c_int
        f.argtypes = [C.c_char_p]
        return f(s.encode())


class Oracle(_Base):
    """The restatement (oracle/mifi_oracle.c)."""
    prefix = "orc_"
    names = {k: "orc_" + k for k in (
        "points2position", "get_values_nn", "get_values_bilinear", "get_values_bicubic", "project_axes", "project_values",
        "interpolate_f", "vector_matrix", "vector_matrix_field", "vector_matrix_points", "vector_reproject_by_matrix",
        "vector_reproject_direction", "vector_reproject_values", "string_to_method")}

    def __init__(self, path=ORACLE_SO):
        super().__init__(path)

    # ---- restated C++ layers (no compiled reference exists for these) -------------------------
    def bilinear_is_ub(self, x, y, ix, iy):
        f = self.lib.orc_bilinear_is_ub
        f.restype = C.c_int
        f.argtypes = [C.c_double, C.c_double, C.c_int, C.c_int]
        return bool(f(float(x), float(y), ix, iy))

    def reduced_domain(self, px, py, inX, inY):
        """CachedInterpolation::createReducedDomain. Returns (reduced?, px, py, inX, inY, minX, minY)."""
        pxa, pxp = _d(np.array(px, dtype=np.float64, copy=True))
        pya, pyp = _d(np.array(py, dtype=np.float64, copy=True))
        ix, iy = C.c_size_t(inX), C.c_size_t(inY)
        mx, my = C.c_longlong(0), C.c_longlong(0)
        f = self.lib.orc_reduced_domain
        f.restype = C.c_int
        f.argtypes = [_dp, _dp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_longlong),
                      C.POINTER(C.c_longlong)]
        r = f(pxp, pyp, pxa.size, C.byref(ix), C.byref(iy), C.byref(mx), C.byref(my))
        return bool(r), pxa, pya, ix.value, iy.value, mx.value, my.value

    def cached_interpolate(self, method, px, py, inX, inY, outX, outY, indata, nthreads=0, out=None):
        """CachedInterpolation::interpolateValues: in [z][inY][inX] -> out [z][outY][outX]."""
        pxa, pxp = _d(px)
        pya, pyp = _d(py)
        a, ap = _f(indata)
        inZ = a.size // (inX * inY)
        if out is None:
            out = np.empty(inZ * outX * outY, dtype=np.float32)
        f = self.lib.orc_cached_interpolate
        f.restype = C.c_int
        f.argtypes = [C.c_int, _dp, _dp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, _fp, C.c_size_t, _fp, C.c_int]
        rc = f(method, pxp, pyp, inX, inY, outX, outY, ap, a.size, out.ctypes.data_as(_fp), nthreads)
        if rc != MIFI_OK:
            raise RuntimeError("orc_cached_interpolate failed")
        return out.reshape(inZ, outY, outX)

    def round_and_clamp(self, pos, maxi):
        p, pp = _d(pos)
        idx = np.empty(p.size, dtype=np.int32)
        f = self.lib.orc_round_and_clamp
        f.restype = None
        f.argtypes = [_dp, C.c_size_t, C.c_int, _ip]
        f(pp, p.size, int(maxi), idx.ctypes.data_as(_ip))
        return idx

    def forward_interpolate(self, method, px, py, inX, inY, outX, outY, indata):
        """CachedForwardInterpolation ctor (rounding) + interpolateValues."""
        xi = self.round_and_clamp(px, outX - 1)
        yi = self.round_and_clamp(py, outY - 1)
        a, ap = _f(indata)
        inZ = a.size // (inX * inY)
        out = np.empty(inZ * outX * outY, dtype=np.float32)
        f = self.lib.orc_forward_interpolate
        f.restype = C.c_int
        f.argtypes = [C.c_int, _ip, _ip, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, _fp, C.c_size_t, _fp]
        rc = f(method, xi.ctypes.data_as(_ip), yi.ctypes.data_as(_ip), inX, inY, outX, outY, ap, a.size, out.ctypes.data_as(_fp))
        if rc != MIFI_OK:
            raise RuntimeError("orc_forward_interpolate failed")
        return out.reshape(inZ, outY, outX)

    def nth_element(self, values, nth):
        """the restated std::nth_element(v, v + nth, v + n) of the forward median on a float32 copy; returns the copy"""
        a, ap = _f(np.array(values, dtype=np.float32, copy=True))
        f = self.lib.orc_nth_element
        f.restype = None
        f.argtypes = [_fp, C.c_size_t, C.c_size_t]
        if a.size:
            f(ap, int(nth), a.size)
        return a

    def bad2nan(self, data, bad):
        a, ap = _f(np.array(data, dtype=np.float32, copy=True))
        f = self.lib.orc_bad2nan
        f.restype = C.c_size_t
        f.argtypes = [_fp, C.c_size_t, C.c_float]
        f(ap, a.size, bad)
        return a

    _TAGS = {"int8": "i8", "int16": "i16", "int32": "i32", "float32": "f32", "float64": "f64", "uint8": "u8", "uint16": "u16",
             "uint32": "u32", "int64": "i64", "uint64": "u64"}

    def as_float(self, data, bad):
        """data2InterpolationArray (CDMInterpolator.cc:115-119): any CDM numeric type -> float32 with badValue -> NaN"""
        a = np.ascontiguousarray(data)
        out = np.empty(a.shape, dtype=np.float32)
        f = getattr(self.lib, "orc_as_float_" + self._TAGS[str(a.dtype)])
        f.restype = None
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_double, C.c_void_p]
        f(a.ctypes.data_as(C.c_void_p), a.size, float(bad), out.ctypes.data_as(C.c_void_p))
        return out

    def from_float(self, data, fill, dtype):
        """interpolationArray2Data (CDMInterpolator.cc:121-124): NaN -> fill, round + cast to `dtype`"""
        a = np.ascontiguousarray(data, dtype=np.float32)
        out = np.empty(a.shape, dtype=np.dtype(dtype))
        f = getattr(self.lib, "orc_from_float_" + self._TAGS[str(np.dtype(dtype))])
        f.restype = None
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_double, C.c_void_p]
        f(a.ctypes.data_as(C.c_void_p), a.size, float(fill), out.ctypes.data_as(C.c_void_p))
        return out

    def nan2fill(self, data, fill, dtype):
        return self.from_float(data, fill, dtype).ravel()

    def coordnn(self, tlon, tlat, lon2d, lat2d, nx, ny):
        """fastTranslatePointsToClosestInputCell. Returns (px, py, n_exact_ties)."""
        pxa, pxp = _d(np.array(tlon, dtype=np.float64, copy=True))
        pya, pyp = _d(np.array(tlat, dtype=np.float64, copy=True))
        lo, lop = _d(lon2d)
        la, lap = _d(lat2d)
        f = self.lib.orc_coordnn
        f.restype = C.c_long
        f.argtypes = [_dp, _dp, C.c_size_t, _dp, _dp, C.c_size_t, C.c_size_t]
        ties = f(pxp, pyp, pxa.size, lop, lap, nx, ny)
        return pxa, pya, ties

    def fill2d(self, field, relaxCrit, corrEff, maxLoop, lib=None, name="orc_fill2d"):
        """mifi_fill2d_f on every level of field[..., ny, nx]; returns (filled copy, NaN count per level)"""
        a = np.array(field, dtype=np.float32, copy=True, order="C")
        ny, nx = a.shape[-2:]
        f = getattr(lib or self.lib, name)
        f.restype = C.c_int
        f.argtypes = [C.c_size_t, C.c_size_t, _fp, C.c_float, C.c_float, C.c_size_t, C.POINTER(C.c_size_t)]
        counts = []
        flat = a.reshape(-1, ny, nx)
        for z in range(flat.shape[0]):
            n = C.c_size_t(0)
            f(nx, ny, flat[z].ctypes.data_as(_fp), relaxCrit, corrEff, maxLoop, C.byref(n))
            counts.append(n.value)
        return a, counts

    def creepfill2d(self, field, repeat, setWeight, defaultVal=None, lib=None, prefix="orc"):
        """mifi_creepfill2d_f (defaultVal None) / mifi_creepfillval2d_f on every level of field[..., ny, nx]"""
        a = np.array(field, dtype=np.float32, copy=True, order="C")
        ny, nx = a.shape[-2:]
        flat = a.reshape(-1, ny, nx)
        counts = []
        for z in range(flat.shape[0]):
            n = C.c_size_t(0)
            p = flat[z].ctypes.data_as(_fp)
            if prefix == "orc":
                f = self.lib.orc_creepfill2d
                f.restype = C.c_int
                f.argtypes = [C.c_size_t, C.c_size_t, _fp, C.c_int, C.c_float, C.c_ushort, C.c_char, C.POINTER(C.c_size_t)]
                f(nx, ny, p, int(defaultVal is None), 0.0 if defaultVal is None else defaultVal, repeat, bytes([setWeight & 0xff]), C.byref(n))
            elif defaultVal is None:
                f = lib.mifi_creepfill2d_f
                f.restype = C.c_int
                f.argtypes = [C.c_size_t, C.c_size_t, _fp, C.c_ushort, C.c_char, C.POINTER(C.c_size_t)]
                f(nx, ny, p, repeat, bytes([setWeight & 0xff]), C.byref(n))
            else:
                f = lib.mifi_creepfillval2d_f
                f.restype = C.c_int
                f.argtypes = [C.c_size_t, C.c_size_t, _fp, C.c_float, C.c_ushort, C.c_char, C.POINTER(C.c_size_t)]
                f(nx, ny, p, defaultVal, repeat, bytes([setWeight & 0xff]), C.byref(n))
            counts.append(n.value)
        return a, counts

    def coordkd(self, tlon, tlat, lon2d, lat2d, nx, ny, max_dist_m):
        """coord_kdtree search: target lon/lat (rad) -> source (ix, iy) as doubles, (-1000, -1000) if nothing is inside the radius"""
        px, pxp = _d(np.array(tlon, dtype=np.float64, copy=True))
        py, pyp = _d(np.array(tlat, dtype=np.float64, copy=True))
        lo, lop = _d(lon2d)
        la, lap = _d(lat2d)
        f = self.lib.orc_coordkd
        f.restype = C.c_long
        f.argtypes = [_dp, _dp, C.c_size_t, _dp, _dp, C.c_size_t, C.c_size_t, C.c_double]
        ties = f(pxp, pyp, px.size, lop, lap, nx, ny, float(max_dist_m))
        return px, py, int(ties)

    def max_distance_of_interest(self, xa, ya, is_metric):
        x, xp = _d(xa)
        y, yp = _d(ya)
        f = self.lib.orc_max_distance_of_interest
        f.restype = C.c_double
        f.argtypes = [_dp, C.c_size_t, _dp, C.c_size_t, C.c_int]
        return float(f(xp, x.size, yp, y.size, int(is_metric)))

    def grid_distance(self, lon2d, lat2d, nx, ny):
        lo, lop = _d(lon2d)
        la, lap = _d(lat2d)
        f = self.lib.orc_grid_distance
        f.restype = C.c_double
        f.argtypes = [_dp, _dp, C.c_size_t, C.c_size_t]
        return f(lop, lap, nx, ny)

    def lonlat_to_matrix(self, lonv, latv):
        lo, lop = _d(lonv)
        la, lap = _d(latv)
        n = lo.size * la.size
        lon2d = np.empty(n)
        lat2d = np.empty(n)
        f = self.lib.orc_lonlat_to_matrix
        f.restype = None
        f.argtypes = [_dp, _dp, C.c_size_t, C.c_size_t, _dp, _dp]
        f(lop, lap, lo.size, la.size, lon2d.ctypes.data_as(_dp), lat2d.ctypes.data_as(_dp))
        return lon2d, lat2d


class Reference(_Base):
    """The reference's src/interpolation.c, compiled unmodified (oracle/_ref/libmifi_ref.so)."""
    prefix = "mifi_"
    names = {
        "points2position": "mifi_points2position",
        "get_values_nn": "mifi_get_values_f",
        "get_values_bilinear": "mifi_get_values_bilinear_f",
        "get_values_bicubic": "mifi_get_values_bicubic_f",
        "project_axes": "mifi_project_axes",
        "project_values": "mifi_project_values",
        "interpolate_f": "mifi_interpolate_f",
        "vector_matrix": "mifi_get_vector_reproject_matrix",
        "vector_matrix_field": "mifi_get_vector_reproject_matrix_field",
        "vector_matrix_points": "mifi_get_vector_reproject_matrix_points",
        "vector_reproject_by_matrix": "mifi_vector_reproject_values_by_matrix_f",
        "vector_reproject_direction": "mifi_vector_reproject_direction_by_matrix_f",
        "vector_reproject_values": "mifi_vector_reproject_values_f",
        "string_to_method": "mifi_string_to_interpolation_method",
    }

    def __init__(self, path=REF_SO):
        super().__init__(path)

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def cached_interpolate(self, method, px, py, inX, inY, outX, outY, indata, nthreads=0, out=None):
        """The reference's own kernels (mifi_get_values_*_f) inside the restated CachedInterpolation.cc:118-147
        loop of oracle/ref_driver.c (OpenMP over target points, like the reference)."""
        pxa, pxp = _d(px)
        pya, pyp = _d(py)
        a, ap = _f(indata)
        inZ = a.size // (inX * inY)
        if out is None:
            out = np.empty(inZ * outX * outY, dtype=np.float32)
        f = self.lib.ref_cached_interpolate
        f.restype = C.c_int
        f.argtypes = [C.c_int, _dp, _dp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, _fp, C.c_size_t, _fp, C.c_int]
        rc = f(int(method), pxp, pyp, inX, inY, outX, outY, ap, a.size, out.ctypes.data_as(_fp), nthreads)
        if rc != MIFI_OK:
            raise RuntimeError("ref_cached_interpolate failed")
        return out.reshape(inZ, outY, outX)

    def max_threads(self):
        self.lib.ref_max_threads.restype = C.c_int
        return self.lib.ref_max_threads()
