"""ctypes binding of include/fimex_b200.h (the C ABI of libfimex_b200.so).

Everything here goes through the shared library; if it is missing the import of the first symbol raises
``FimexB200Error`` -- nothing falls back to numpy or to the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import enum
import os
import re

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("FIMEX_B200_LIB") or os.path.join(HERE, "lib", "libfimex_b200.so")  # override: A/B experiments only
HEADER = os.path.normpath(os.path.join(HERE, "..", "include", "fimex_b200.h"))

MIFI_OK, MIFI_ERROR = 1, -1
PROJ_AXIS, LONGITUDE, LATITUDE = 0, 1, 2
MIFI_VECTOR_KEEP_SIZE, MIFI_VECTOR_RESIZE = 0, 1


class Method(enum.IntEnum):
    """enum mifi_interpol_method (reference include/fimex/mifi_constants.h:52-147)"""
    UNKNOWN = -1
    NEAREST_NEIGHBOR = 0
    BILINEAR = 1
    BICUBIC = 2
    COORD_NN = 3
    COORD_NN_KD = 4
    FORWARD_SUM = 5
    FORWARD_MEAN = 6
    FORWARD_MEDIAN = 7
    FORWARD_MAX = 8
    FORWARD_MIN = 9
    FORWARD_UNDEF_SUM = 10
    FORWARD_UNDEF_MEAN = 11
    FORWARD_UNDEF_MEDIAN = 12
    FORWARD_UNDEF_MAX = 13
    FORWARD_UNDEF_MIN = 14


class DataType(enum.IntEnum):
    """enum CDMDataType (reference include/fimex/CDMDataType.h:35-49)"""
    NAT = 0
    CHAR = 1
    SHORT = 2
    INT = 3
    FLOAT = 4
    DOUBLE = 5
    STRING = 6
    UCHAR = 7
    USHORT = 8
    UINT = 9
    INT64 = 10
    UINT64 = 11


_NP2CDM = {"int8": DataType.CHAR, "int16": DataType.SHORT, "int32": DataType.INT, "float32": DataType.FLOAT, "float64": DataType.DOUBLE,
           "uint8": DataType.UCHAR, "uint16": DataType.USHORT, "uint32": DataType.UINT, "int64": DataType.INT64, "uint64": DataType.UINT64}


def cdm_type(dtype) -> DataType:
    """numpy / torch dtype -> CDMDataType"""
    try:
        if str(dtype).startswith("torch."):
            dtype = str(dtype)[len("torch."):]
        return _NP2CDM[str(np.dtype(dtype))]
    except (KeyError, TypeError):
        raise FimexB200Error(f"no CDM data type for {dtype}") from None


def default_fill_value(dtype) -> float:
    """defaultFillValue_ (reference src/CDM.cc:490-503, include/fimex/CDMconstants.h:149-158)"""
    return {DataType.DOUBLE: 9.9692099683868690e+36, DataType.FLOAT: float(np.float32(9.9692099683868690e+36)),
            DataType.INT64: -9223372036854775806.0, DataType.INT: -2147483647.0, DataType.SHORT: -32767.0, DataType.CHAR: -127.0,
            DataType.UINT64: 18446744073709551614.0, DataType.UINT: 4294967295.0, DataType.USHORT: 65535.0,
            DataType.UCHAR: 255.0}[cdm_type(dtype)]


class FimexB200Error(RuntimeError):
    """The counterpart of the reference's CDMException for this path."""


_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_vp = C.c_void_p
_lib = None


def lib_path() -> str:
    return _LIB_PATH


def declared_symbols() -> list:
    """Every function the public header declares (used by the CPU-side ABI test)."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:fb200|mifi)_[A-Za-z0-9_]+)\s*\(", text)))


def load(build_if_missing: bool = True):
    """Load libfimex_b200.so (building it with nvcc first if it is not there).  Raises when impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        if not build_if_missing:
            raise FimexB200Error(f"{_LIB_PATH} is missing; run `python -m fimex_b200.build`")
        from . import build as _build
        _build.build()
    try:
        lib = C.CDLL(_LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise FimexB200Error(f"cannot load {_LIB_PATH}: {e}") from e
    _declare(lib)
    _lib = lib
    return lib


def _declare(lib):
    sz, i, ll = C.c_size_t, C.c_int, C.c_longlong
    P = C.POINTER
    sig = {
        "fb200_version": (C.c_char_p, []),
        "fb200_last_error": (C.c_char_p, []),
        "fb200_set_device": (i, [i]),
        "fb200_get_device": (i, []),
        "fb200_kernel_launches": (C.c_ulonglong, []),
        "fb200_host_alloc": (_vp, [sz]),
        "fb200_host_free": (None, [_vp]),
        "fb200_host_trim": (None, []),
        "fb200_cached_interpolation_create": (i, [i, _vp, _vp, sz, sz, sz, sz, P(_vp)]),
        "fb200_cached_interpolation_create_device": (i, [i, _vp, _vp, sz, sz, sz, sz, P(_vp)]),
        "fb200_cached_interpolation_create_from_projection": (i, [i, C.c_char_p, _vp, _vp, sz, sz, i, i, C.c_char_p, _vp, _vp, sz, sz, i,
                                                                  P(_vp)]),
        "fb200_cached_interpolation_create_from_template": (i, [i, C.c_char_p, _vp, _vp, sz, sz, C.c_char_p, _vp, _vp, sz, sz, i, P(_vp)]),
        "fb200_vector_create_from_points": (i, [i, C.c_char_p, C.c_char_p, i, _vp, _vp, i, P(_vp)]),
        "fb200_cached_interpolation_create_from_coordinates": (i, [i, C.c_char_p, _vp, _vp, sz, sz, i, i, _vp, _vp, sz, sz, P(_vp)]),
        "fb200_cached_interpolation_create_from_coordinates_kd": (i, [i, C.c_char_p, _vp, _vp, sz, sz, i, i, _vp, _vp, sz, sz, C.c_double,
                                                                     P(_vp)]),
        "fb200_cached_forward_interpolation_create": (i, [i, _vp, _vp, sz, sz, sz, sz, P(_vp)]),
        "fb200_cached_forward_interpolation_create_from_coordinates": (i, [i, C.c_char_p, _vp, _vp, sz, sz, i, i, _vp, _vp, sz, sz, P(_vp)]),
        "fb200_interp_create_reduced_domain": (i, [_vp, P(i), P(ll), P(ll)]),
        "fb200_interp_in_x": (sz, [_vp]),
        "fb200_interp_in_y": (sz, [_vp]),
        "fb200_interp_out_x": (sz, [_vp]),
        "fb200_interp_out_y": (sz, [_vp]),
        "fb200_interp_method": (i, [_vp]),
        "fb200_interp_get_points": (i, [_vp, _vp, _vp]),
        "fb200_interp_device_points": (i, [_vp, P(_vp), P(_vp), P(sz)]),
        "fb200_interp_new_size": (sz, [_vp, sz]),
        "fb200_interp_interpolate_values": (i, [_vp, _vp, sz, _vp, P(sz)]),
        "fb200_interp_interpolate_values_device": (i, [_vp, _vp, sz, _vp, P(sz), _vp]),
        "fb200_interp_destroy": (None, [_vp]),
        "fb200_vector_create": (i, [i, _vp, i, i, P(_vp)]),
        "fb200_vector_create_from_projection": (i, [i, C.c_char_p, C.c_char_p, _vp, _vp, i, i, i, i, P(_vp)]),
        "fb200_vector_reproject_values": (i, [_vp, _vp, _vp, sz]),
        "fb200_vector_reproject_values_device": (i, [_vp, _vp, _vp, sz, _vp]),
        "fb200_vector_reproject_direction_values": (i, [_vp, _vp, sz]),
        "fb200_vector_get_matrix": (i, [_vp, _vp]),
        "fb200_vector_create_from_grid": (i, [i, C.c_char_p, _vp, _vp, i, i, i, i, P(_vp)]),
        "fb200_vector_get_slice": (i, [_vp, i, _vp, _vp, sz, C.c_double, C.c_double, i, _vp, _vp]),
        "fb200_vector_get_slice_device": (i, [_vp, i, _vp, _vp, sz, C.c_double, C.c_double, i, _vp, _vp, _vp]),
        "fb200_vector_destroy": (None, [_vp]),
        "fb200_interp_interpolate_vector": (i, [_vp, _vp, _vp, _vp, sz, _vp, _vp, P(sz)]),
        "fb200_interp_interpolate_vector_device": (i, [_vp, _vp, _vp, _vp, sz, _vp, _vp, P(sz), _vp]),
        "fb200_interp_add_preprocess": (i, [_vp, C.c_char_p]),
        "fb200_interp_add_postprocess": (i, [_vp, C.c_char_p]),
        "fb200_interp_get_data_slice": (i, [_vp, i, _vp, sz, C.c_double, i, _vp, P(sz)]),
        "fb200_interp_get_data_slice_device": (i, [_vp, i, _vp, sz, C.c_double, i, _vp, P(sz), _vp]),
        "fb200_interp_get_vector_slice": (i, [_vp, _vp, i, _vp, _vp, sz, C.c_double, C.c_double, i, _vp, _vp, P(sz)]),
        "fb200_interp_get_vector_slice_device": (i, [_vp, _vp, i, _vp, _vp, sz, C.c_double, C.c_double, i, _vp, _vp, P(sz), _vp]),
        "fb200_vinterp_create_hybrid": (i, [i, _vp, _vp, i, C.c_double, _vp, i, i, P(_vp)]),
        "fb200_vinterp_create_sigma": (i, [i, _vp, i, C.c_double, C.c_double, _vp, i, i, P(_vp)]),
        "fb200_vinterp_destroy": (None, [_vp]),
        "fb200_vinterp_interpolate_values": (i, [_vp, _vp, _vp, sz, sz, _vp]),
        "fb200_vinterp_interpolate_values_device": (i, [_vp, _vp, _vp, sz, sz, _vp, _vp]),
        "fb200_vinterp_get_data_slice": (i, [_vp, i, _vp, _vp, sz, sz, C.c_double, i, _vp]),
        "fb200_vinterp_get_data_slice_device": (i, [_vp, i, _vp, _vp, sz, sz, C.c_double, i, _vp, _vp]),
        "fb200_vinterp_create_height": (i, [i, i, i, i, _vp, _vp, i, C.c_double, C.c_double, C.c_double, C.c_double, _vp, i, i, P(_vp)]),
        "fb200_vinterp_interpolate_values_columns": (i, [_vp, _vp, _vp, sz, sz, _vp]),
        "fb200_vinterp_interpolate_values_columns_device": (i, [_vp, _vp, _vp, sz, sz, _vp, _vp]),
        "fb200_vinterp_get_data_slice_columns": (i, [_vp, i, _vp, _vp, sz, sz, C.c_double, i, _vp]),
        "fb200_vinterp_get_data_slice_columns_device": (i, [_vp, i, _vp, _vp, sz, sz, C.c_double, i, _vp, _vp]),
        "fb200_vinterp_create_depth": (i, [i, i, _vp, _vp, i, C.c_double, _vp, i, i, P(_vp)]),
        "fb200_vconvert_create": (i, [i, i, _vp, _vp, i, C.c_double, C.c_double, P(_vp)]),
        "fb200_vconvert_destroy": (None, [_vp]),
        "fb200_vconvert_values": (i, [_vp, _vp, _vp, sz, sz, _vp]),
        "fb200_vconvert_values_device": (i, [_vp, _vp, _vp, sz, sz, _vp, _vp]),
        "fb200_tinterp_create": (i, [_vp, i, _vp, i, i, P(_vp)]),
        "fb200_tinterp_destroy": (None, [_vp]),
        "fb200_tinterp_source_steps": (i, [_vp, i, P(i), P(i), P(C.c_double)]),
        "fb200_tinterp_get_step": (i, [_vp, i, i, _vp, _vp, sz, C.c_double, i, _vp]),
        "fb200_tinterp_get_step_device": (i, [_vp, i, i, _vp, _vp, sz, C.c_double, i, _vp, _vp]),
        "fb200_tinterp_get_data_slice_device": (i, [_vp, i, _vp, sz, C.c_double, i, _vp, _vp]),
        "fb200_merge_create": (i, [_vp, _vp, _vp, sz, sz, sz, sz, i, i, i, P(_vp)]),
        "fb200_merge_destroy": (None, [_vp]),
        "fb200_merge_get_data_slice": (i, [_vp, i, _vp, sz, C.c_double, _vp, sz, C.c_double, i, C.c_double, _vp, P(sz)]),
        "fb200_merge_get_data_slice_device": (i, [_vp, i, _vp, sz, C.c_double, _vp, sz, C.c_double, i, C.c_double, _vp, P(sz), _vp]),
        "mifi_string_to_interpolation_method": (i, [C.c_char_p]),
        "mifi_interpolate_f": (i, [i, C.c_char_p, _vp, _vp, _vp, i, i, i, i, i, C.c_char_p, _vp, _vp, _vp, i, i, i, i]),
        "mifi_vector_reproject_values_f": (i, [i, C.c_char_p, C.c_char_p, _vp, _vp, _vp, _vp, i, i, i, i, i]),
        "mifi_vector_reproject_values_by_matrix_f": (i, [i, _vp, _vp, _vp, i, i, i]),
        "mifi_vector_reproject_direction_by_matrix_f": (i, [i, _vp, _vp, i, i, i]),
        "mifi_get_vector_reproject_matrix": (i, [C.c_char_p, C.c_char_p, _vp, _vp, i, i, i, i, _vp]),
        "mifi_get_vector_reproject_matrix_field": (i, [C.c_char_p, C.c_char_p, _vp, _vp, i, i, _vp]),
        "mifi_get_vector_reproject_matrix_points": (i, [C.c_char_p, C.c_char_p, i, _vp, _vp, i, _vp]),
        "mifi_get_values_f": (i, [_vp, _vp, C.c_double, C.c_double, i, i, i]),
        "mifi_get_values_bilinear_f": (i, [_vp, _vp, C.c_double, C.c_double, i, i, i]),
        "mifi_get_values_bicubic_f": (i, [_vp, _vp, C.c_double, C.c_double, i, i, i]),
        "mifi_points2position": (i, [_vp, i, _vp, i, i]),
        "mifi_project_values": (i, [C.c_char_p, C.c_char_p, _vp, _vp, i]),
        "mifi_project_axes": (i, [C.c_char_p, C.c_char_p, _vp, _vp, i, i, _vp, _vp]),
        "mifi_bad2nanf": (sz, [_vp, _vp, C.c_float]),
        "mifi_nanf2bad": (sz, [_vp, _vp, C.c_float]),
        "mifi_fill2d_f": (i, [sz, sz, _vp, C.c_float, C.c_float, sz, P(sz)]),
        "mifi_creepfill2d_f": (i, [sz, sz, _vp, C.c_ushort, C.c_char, P(sz)]),
        "mifi_creepfillval2d_f": (i, [sz, sz, _vp, C.c_float, C.c_ushort, C.c_char, P(sz)]),
        "fb200_fill2d_device": (i, [_vp, sz, sz, sz, C.c_float, C.c_float, sz, _vp]),
        "fb200_creepfill2d_device": (i, [_vp, sz, sz, sz, i, C.c_float, C.c_ushort, C.c_char, _vp]),
        "mifi_setNumThreads": (i, [i]),
    }
    for name, (res, args) in sig.items():
        f = getattr(lib, name)  # AttributeError here == the library does not export what the header declares
        f.restype = res
        f.argtypes = args


# ------------------------------------------------------------------------------------------------ helpers
def last_error() -> str:
    return load().fb200_last_error().decode()


def check(rc: int, what: str = ""):
    if rc != MIFI_OK:
        raise FimexB200Error(f"{what}: {last_error()}" if what else last_error())


def version() -> str:
    return load().fb200_version().decode()


def set_device(dev: int):
    check(load().fb200_set_device(int(dev)), "fb200_set_device")


def kernel_launches() -> int:
    return int(load().fb200_kernel_launches())


def f64(a, copy=False):
    return np.array(a, dtype=np.float64, copy=True, order="C") if copy else np.ascontiguousarray(a, dtype=np.float64)


def f32(a, copy=False):
    return np.array(a, dtype=np.float32, copy=True, order="C") if copy else np.ascontiguousarray(a, dtype=np.float32)


def ptr(a):
    """address of a numpy array or a torch tensor (device or host) as c_void_p"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(a.data_ptr())  # torch.Tensor


# ------------------------------------------------------------------------------------------------ mifi_* (host arrays)
def mifi_string_to_interpolation_method(s: str) -> int:
    return load().mifi_string_to_interpolation_method(s.encode())


def mifi_points2position(points, axis, axis_type):
    """returns (rc, positions); the input array is not modified (the C function works in place on a copy)"""
    p = f64(points, copy=True)
    ax = f64(axis)
    rc = load().mifi_points2position(ptr(p), p.size, ptr(ax), ax.size, int(axis_type))
    return rc, p


def mifi_project_values(proj_in, proj_out, x, y):
    xa, ya = f64(x, copy=True), f64(y, copy=True)
    rc = load().mifi_project_values(proj_in.encode(), proj_out.encode(), ptr(xa), ptr(ya), xa.size)
    return rc, xa, ya


def mifi_project_axes(proj_in, proj_out, xaxis, yaxis):
    xa, ya = f64(xaxis), f64(yaxis)
    xo = np.empty(xa.size * ya.size)
    yo = np.empty(xa.size * ya.size)
    rc = load().mifi_project_axes(proj_in.encode(), proj_out.encode(), ptr(xa), ptr(ya), xa.size, ya.size, ptr(xo), ptr(yo))
    return rc, xo, yo


def mifi_interpolate_f(method, proj_in, infield, in_x, in_y, in_xt, in_yt, iz, proj_out, out_x, out_y, out_xt, out_yt, out_init=None):
    a = f32(infield)
    ixa, iya, oxa, oya = f64(in_x), f64(in_y), f64(out_x), f64(out_y)
    out = np.full(iz * oya.size * oxa.size, np.nan, dtype=np.float32) if out_init is None else f32(out_init, copy=True)
    rc = load().mifi_interpolate_f(int(method), proj_in.encode(), ptr(a), ptr(ixa), ptr(iya), in_xt, in_yt, ixa.size, iya.size, iz,
                                   proj_out.encode(), ptr(out), ptr(oxa), ptr(oya), out_xt, out_yt, oxa.size, oya.size)
    return rc, out.reshape(iz, oya.size, oxa.size)


def mifi_get_vector_reproject_matrix(proj_in, proj_out, out_x, out_y, xt, yt):
    oxa, oya = f64(out_x), f64(out_y)
    m = np.empty(4 * oxa.size * oya.size)
    rc = load().mifi_get_vector_reproject_matrix(proj_in.encode(), proj_out.encode(), ptr(oxa), ptr(oya), xt, yt, oxa.size, oya.size, ptr(m))
    return rc, m


def mifi_get_vector_reproject_matrix_field(proj_in, proj_out, in_x_field, in_y_field, ox, oy):
    xa, ya = f64(in_x_field), f64(in_y_field)
    m = np.empty(4 * ox * oy)
    rc = load().mifi_get_vector_reproject_matrix_field(proj_in.encode(), proj_out.encode(), ptr(xa), ptr(ya), ox, oy, ptr(m))
    return rc, m


def mifi_get_vector_reproject_matrix_points(proj_in, proj_out, metric, x, y):
    xa, ya = f64(x), f64(y)
    m = np.empty(4 * xa.size)
    rc = load().mifi_get_vector_reproject_matrix_points(proj_in.encode(), proj_out.encode(), int(metric), ptr(xa), ptr(ya), xa.size, ptr(m))
    return rc, m


def mifi_vector_reproject_values_by_matrix_f(method, matrix, u, v, ox, oy, oz):
    m = f64(matrix)
    uu, vv = f32(u, copy=True), f32(v, copy=True)
    rc = load().mifi_vector_reproject_values_by_matrix_f(method, ptr(m), ptr(uu), ptr(vv), ox, oy, oz)
    return rc, uu, vv


def mifi_vector_reproject_direction_by_matrix_f(method, matrix, angles, ox, oy, oz):
    m = f64(matrix)
    a = f32(angles, copy=True)
    rc = load().mifi_vector_reproject_direction_by_matrix_f(method, ptr(m), ptr(a), ox, oy, oz)
    return rc, a


def mifi_vector_reproject_values_f(method, proj_in, proj_out, u, v, out_x, out_y, xt, yt, oz):
    oxa, oya = f64(out_x), f64(out_y)
    uu, vv = f32(u, copy=True), f32(v, copy=True)
    rc = load().mifi_vector_reproject_values_f(method, proj_in.encode(), proj_out.encode(), ptr(uu), ptr(vv), ptr(oxa), ptr(oya), xt, yt,
                                               oxa.size, oya.size, oz)
    return rc, uu, vv


def _one_point(fn, infield, x, y, ix, iy, iz):
    a = f32(infield)
    out = np.empty(iz, dtype=np.float32)
    rc = fn(ptr(a), ptr(out), float(x), float(y), ix, iy, iz)
    return rc, out


def mifi_get_values_f(infield, x, y, ix, iy, iz):
    return _one_point(load().mifi_get_values_f, infield, x, y, ix, iy, iz)


def mifi_get_values_bilinear_f(infield, x, y, ix, iy, iz):
    return _one_point(load().mifi_get_values_bilinear_f, infield, x, y, ix, iy, iz)


def mifi_get_values_bicubic_f(infield, x, y, ix, iy, iz):
    return _one_point(load().mifi_get_values_bicubic_f, infield, x, y, ix, iy, iz)


def mifi_bad2nanf(data, bad):
    a = f32(data, copy=True)
    load().mifi_bad2nanf(C.c_void_p(a.ctypes.data), C.c_void_p(a.ctypes.data + a.nbytes), C.c_float(bad))
    return a


def mifi_nanf2bad(data, bad):
    a = f32(data, copy=True)
    load().mifi_nanf2bad(C.c_void_p(a.ctypes.data), C.c_void_p(a.ctypes.data + a.nbytes), C.c_float(bad))
    return a


# ------------------------------------------------------------------------------------------------ 2-D pre/post-processes
def mifi_fill2d_f(field, relaxCrit, corrEff, maxLoop):
    """one level [ny][nx] of host data; returns (rc, filled copy, nChanged)"""
    a = f32(field, copy=True)
    ny, nx = a.shape[-2:]
    n = C.c_size_t(0)
    rc = load().mifi_fill2d_f(nx, ny, ptr(a), relaxCrit, corrEff, int(maxLoop), C.byref(n))
    return rc, a, n.value


def mifi_creepfill2d_f(field, repeat, setWeight, defaultVal=None):
    """mifi_creepfill2d_f, or mifi_creepfillval2d_f when defaultVal is given; one level [ny][nx] of host data"""
    a = f32(field, copy=True)
    ny, nx = a.shape[-2:]
    n = C.c_size_t(0)
    w = bytes([int(setWeight) & 0xff])
    if defaultVal is None:
        rc = load().mifi_creepfill2d_f(nx, ny, ptr(a), int(repeat), w, C.byref(n))
    else:
        rc = load().mifi_creepfillval2d_f(nx, ny, ptr(a), float(defaultVal), int(repeat), w, C.byref(n))
    return rc, a, n.value


def fill2d_device(field, relaxCrit, corrEff, maxLoop, stream=None):
    """all levels of a CUDA tensor [..., ny, nx] in place (processArray_, CDMInterpolator.cc:136-159)"""
    ny, nx = field.shape[-2:]
    nz = field.numel() // max(1, nx * ny)
    check(load().fb200_fill2d_device(ptr(field), nx, ny, nz, relaxCrit, corrEff, int(maxLoop), stream), "fill2d")
    return field


def creepfill2d_device(field, repeat, setWeight, defaultVal=None, stream=None):
    ny, nx = field.shape[-2:]
    nz = field.numel() // max(1, nx * ny)
    check(load().fb200_creepfill2d_device(ptr(field), nx, ny, nz, int(defaultVal is not None), 0.0 if defaultVal is None else float(defaultVal),
                                          int(repeat), bytes([int(setWeight) & 0xff]), stream), "creepfill2d")
    return field
