"""Host-side mirror of the pressure, height and depth branches of the reference's CDMVerticalInterpolator
(``--verticalInterpolate.type=pressure|height|altitude|depth --verticalInterpolate.method=... --verticalInterpolate.level1=...``).

The source vertical coordinate is given by its CF standard name and formula terms, as the reference reads them from the CDM:

* ``air_pressure``: pressure levels, terms ``{"p": levels}``;
* ``atmosphere_hybrid_sigma_pressure_coordinate``: terms ``{"ap": ap, "b": b}`` or ``{"a": a, "p0": p0, "b": b}``;
* ``atmosphere_sigma_coordinate``: terms ``{"sigma": sigma, "ptop": ptop}``.

The surface pressure ``ps`` is not a term here: it is a field, passed with every slice.  All pressures are in the unit of the
target levels (hPa, as the reference's level1 option); ``ps_scale`` converts the ``ps`` field to it (0.01 for Pa).  Height and
altitude levels are in metres (:class:`HeightInterpolator`), as are depth levels below the sea surface (:class:`DepthInterpolator`, from
depth levels or the CF ocean sigma and s-coordinates).  :class:`PressureConversion` runs the data conversions on the model
levels (theta2T, omega2vwind, add4Dpressure) on the same column pressures.  The arithmetic runs in libfimex_b200.so on the GPU (DESIGN.md
section 2 states it).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .cached import _is_torch, _stream_ptr
from .capi import FimexB200Error, check, f64, load, ptr

#: --verticalInterpolate.method values -> MIFI_VINT_METHOD_* (include/fimex/mifi_constants.h)
METHODS = {"linear": 0, "log": 1, "loglog": 2, "nearestneighbor": 3}

PRESSURE = "air_pressure"
HYBRID = "atmosphere_hybrid_sigma_pressure_coordinate"
SIGMA = "atmosphere_sigma_coordinate"
VCOORD_PRESSURE, VCOORD_HYBRID, VCOORD_SIGMA = 0, 1, 2  # FB200_VCOORD_*

#: --verticalInterpolate.type values of the height branch -> FB200_VZ_ALTITUDE / _HEIGHT
TARGETS = {"altitude": 0, "height": 1}
#: the ways to the altitude of every source level -> FB200_VZ_*
CONVERTERS = {"standard": 0, "hypsometric": 1, "field": 2}

DEPTH = "depth"
OCEAN_SIGMA = "ocean_sigma_coordinate"
OCEAN_S_G1 = "ocean_s_coordinate_g1"
OCEAN_S_G2 = "ocean_s_coordinate_g2"
VCOORD_DEPTH, VCOORD_OCEAN_SIGMA, VCOORD_OCEAN_S_G1, VCOORD_OCEAN_S_G2 = 3, 4, 5, 6  # FB200_VCOORD_*


def vertical_method(name: str) -> int:
    """--verticalInterpolate.method string -> MIFI_VINT_METHOD_*; an unknown name raises"""
    try:
        return METHODS[name]
    except KeyError:
        raise FimexB200Error(f"unknown vertical interpolation method: '{name}' (one of {', '.join(METHODS)})") from None


def _source_levels(standard_name: str, terms: dict):
    """(vcoord, a, b, ptop, nk) of the source vertical coordinate: pressure levels a = p; hybrid a = ap, b; sigma b = sigma, ptop"""
    t = {k: v for k, v in terms.items() if k != "ps"}
    if standard_name == PRESSURE:
        p = f64(t["p"]).ravel()
        return VCOORD_PRESSURE, p, None, 0.0, p.size
    if standard_name == HYBRID:
        if "ap" in t:
            ap = f64(t["ap"]).ravel()
        elif "a" in t and "p0" in t:
            ap = f64(t["a"]).ravel() * float(np.asarray(t["p0"], dtype=np.float64).reshape(-1)[0])  # ap_k = a_k * p0, fp64
        else:
            raise FimexB200Error(f"{HYBRID} needs the terms ap, b or a, p0, b; got {sorted(terms)}")
        b = f64(t["b"]).ravel()
        if b.size != ap.size:
            raise FimexB200Error(f"{HYBRID}: {ap.size} values of ap but {b.size} of b")
        return VCOORD_HYBRID, ap, b, 0.0, ap.size
    if standard_name == SIGMA:
        sigma = f64(t["sigma"]).ravel()
        return VCOORD_SIGMA, None, sigma, float(np.asarray(t["ptop"], dtype=np.float64).reshape(-1)[0]), sigma.size
    raise FimexB200Error(f"vertical coordinate '{standard_name}' is not supported (one of {PRESSURE}, {HYBRID}, {SIGMA})")


class _VerticalHandle:
    """Lifetime of an fb200_vinterp (or fb200_vconvert) handle and the shape checks of its calls."""

    nk = 0
    needs_ps = False
    _destroy = "fb200_vinterp_destroy"

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            getattr(load(), self._destroy)(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _shape(self, field, ps):
        if field.ndim < 2 or field.shape[1] != self.nk:
            raise FimexB200Error(f"field must be [nt][{self.nk}][...], got shape {tuple(field.shape)}")
        nt = int(field.shape[0])
        nxy = int(np.prod(field.shape[2:], dtype=np.int64))
        if self.needs_ps and (ps is None or int(np.prod(ps.shape, dtype=np.int64)) != nt * nxy):
            raise FimexB200Error(f"ps must hold nt * nxy = {nt * nxy} values")
        return nt, nxy, (nt, self.levels.size) + tuple(field.shape[2:])

    def _values_columns(self, field, ps, columns, stream):
        """interpolateValues through the _columns calls; columns(nt, nxy, device) -> (fb200_vcolumns, arrays to keep alive)"""
        lib = load()
        if _is_torch(field):
            import torch
            if not field.is_cuda or field.dtype != torch.float32 or not field.is_contiguous():
                raise FimexB200Error("device path needs a contiguous float32 CUDA tensor")
            nt, nxy, shape = self._shape(field, ps)
            cols, keep = columns(nt, nxy, True)
            out = torch.empty(shape, dtype=torch.float32, device=field.device)
            check(lib.fb200_vinterp_interpolate_values_columns_device(self._h, ptr(field), C.byref(cols), nxy, nt, ptr(out), _stream_ptr(stream)),
                  "interpolateValues")
            return out
        a = capi.f32(field)
        nt, nxy, shape = self._shape(a, ps)
        cols, keep = columns(nt, nxy, False)
        out = np.empty(shape, dtype=np.float32)
        check(lib.fb200_vinterp_interpolate_values_columns(self._h, ptr(a), C.byref(cols), nxy, nt, ptr(out)), "interpolateValues")
        return out

    def _slice_columns(self, field, ps, columns, bad_value, out_dtype, stream):
        """getDataSlice through the _columns calls, as _values_columns"""
        lib = load()
        if _is_torch(field):
            import torch
            if not field.is_cuda or not field.is_contiguous():
                raise FimexB200Error("device path needs a contiguous CUDA tensor")
            odt = out_dtype if out_dtype is not None else field.dtype
            bad = capi.default_fill_value(field.dtype) if bad_value is None else float(bad_value)
            nt, nxy, shape = self._shape(field, ps)
            cols, keep = columns(nt, nxy, True)
            out = torch.empty(shape, dtype=odt, device=field.device)
            check(lib.fb200_vinterp_get_data_slice_columns_device(self._h, int(capi.cdm_type(field.dtype)), ptr(field), C.byref(cols), nxy, nt,
                                                                  bad, int(capi.cdm_type(odt)), ptr(out), _stream_ptr(stream)), "getDataSlice")
            return out
        a = np.ascontiguousarray(field)
        odt = np.dtype(out_dtype) if out_dtype is not None else a.dtype
        bad = capi.default_fill_value(a.dtype) if bad_value is None else float(bad_value)
        nt, nxy, shape = self._shape(a, ps)
        cols, keep = columns(nt, nxy, False)
        out = np.empty(shape, dtype=odt)
        check(lib.fb200_vinterp_get_data_slice_columns(self._h, int(capi.cdm_type(a.dtype)), ptr(a), C.byref(cols), nxy, nt, bad,
                                                       int(capi.cdm_type(odt)), ptr(out)), "getDataSlice")
        return out


def _device_ps(ps):
    """ps of a device-path call, as the C ABI reads it: float32 on the device (the shape is checked by _shape); anything else raises"""
    import torch
    if not _is_torch(ps) or not ps.is_cuda or ps.dtype != torch.float32:
        raise FimexB200Error("ps must be a float32 CUDA tensor on the device path")
    return ps.contiguous()


class VerticalInterpolator(_VerticalHandle):
    """Interpolates [nt][nk][...] fields on the source vertical coordinate to [nt][np][...] on the target pressure levels."""

    def __init__(self, standard_name: str, terms: dict, method: str, levels, ps_scale: float = 1.0, extrapolate: bool = True):
        self.method = vertical_method(method)
        self.levels = f64(levels).ravel()
        self._h = C.c_void_p()
        lib = load()
        vcoord, a, b, ptop, self.nk = _source_levels(standard_name, terms)
        self.needs_ps = vcoord != VCOORD_PRESSURE
        if vcoord == VCOORD_SIGMA:
            rc = lib.fb200_vinterp_create_sigma(self.method, ptr(b), self.nk, ptop, float(ps_scale), ptr(self.levels), self.levels.size,
                                                int(bool(extrapolate)), C.byref(self._h))
        else:
            rc = lib.fb200_vinterp_create_hybrid(self.method, ptr(a), ptr(b), self.nk, float(ps_scale), ptr(self.levels), self.levels.size,
                                                 int(bool(extrapolate)), C.byref(self._h))
        check(rc, "VerticalInterpolator")

    def interpolateValues(self, field, ps=None, stream=None):
        """float32 [nt][nk][...] with NaN for undefined values -> float32 [nt][np][...] (numpy or CUDA tensors)"""
        lib = load()
        if _is_torch(field):
            import torch
            if not field.is_cuda or field.dtype != torch.float32 or not field.is_contiguous():
                raise FimexB200Error("device path needs a contiguous float32 CUDA tensor")
            nt, nxy, shape = self._shape(field, ps)
            psd = _device_ps(ps) if self.needs_ps else None
            out = torch.empty(shape, dtype=torch.float32, device=field.device)
            check(lib.fb200_vinterp_interpolate_values_device(self._h, ptr(field), ptr(psd), nxy, nt, ptr(out), _stream_ptr(stream)),
                  "interpolateValues")
            return out
        a = capi.f32(field)
        nt, nxy, shape = self._shape(a, ps)
        p = capi.f32(ps) if ps is not None and self.needs_ps else None
        out = np.empty(shape, dtype=np.float32)
        check(lib.fb200_vinterp_interpolate_values(self._h, ptr(a), ptr(p), nxy, nt, ptr(out)), "interpolateValues")
        return out

    def getDataSlice(self, field, ps=None, bad_value=None, out_dtype=None, stream=None):
        """The per-slice body of the vertical getDataSlice: `field` [nt][nk][...] of any CDM numeric type (numpy array, or CUDA tensor
        for the device-resident path), fill -> NaN, interpolate, NaN -> fill and cast to `out_dtype` (default: the input's type).
        `bad_value` = CDM::getFillValue of the variable (default: the type's default fill value); `ps` [nt][...] float32."""
        lib = load()
        if _is_torch(field):
            import torch
            if not field.is_cuda or not field.is_contiguous():
                raise FimexB200Error("device path needs a contiguous CUDA tensor")
            odt = out_dtype if out_dtype is not None else field.dtype
            bad = capi.default_fill_value(field.dtype) if bad_value is None else float(bad_value)
            nt, nxy, shape = self._shape(field, ps)
            psd = _device_ps(ps) if self.needs_ps else None
            out = torch.empty(shape, dtype=odt, device=field.device)
            check(lib.fb200_vinterp_get_data_slice_device(self._h, int(capi.cdm_type(field.dtype)), ptr(field), ptr(psd), nxy, nt, bad,
                                                          int(capi.cdm_type(odt)), ptr(out), _stream_ptr(stream)), "getDataSlice")
            return out
        a = np.ascontiguousarray(field)
        odt = np.dtype(out_dtype) if out_dtype is not None else a.dtype
        bad = capi.default_fill_value(a.dtype) if bad_value is None else float(bad_value)
        nt, nxy, shape = self._shape(a, ps)
        p = capi.f32(ps) if ps is not None and self.needs_ps else None
        out = np.empty(shape, dtype=odt)
        check(lib.fb200_vinterp_get_data_slice(self._h, int(capi.cdm_type(a.dtype)), ptr(a), ptr(p), nxy, nt, bad, int(capi.cdm_type(odt)),
                                               ptr(out)), "getDataSlice")
        return out


class _Columns(C.Structure):
    """fb200_vcolumns"""
    _fields_ = [("ps", C.c_void_p), ("t", C.c_void_p), ("q", C.c_void_p), ("z", C.c_void_p), ("zs", C.c_void_p)]


def _fill_columns(slots, device):
    """{slot of fb200_vcolumns: (argument name, array, number of values)} -> (the fb200_vcolumns, the arrays it points into, kept alive
    by the caller): float32, CUDA tensors on the device path"""
    cols, keep = _Columns(), []
    for slot, (name, a, n) in slots.items():
        if device:
            import torch
            if not _is_torch(a) or not a.is_cuda or a.dtype != torch.float32:
                raise FimexB200Error(f"{name} must be a float32 CUDA tensor on the device path")
            a = a.contiguous()
        else:
            a = capi.f32(a)
        if int(np.prod(a.shape, dtype=np.int64)) != n:
            raise FimexB200Error(f"{name} must hold {n} values, got shape {tuple(a.shape)}")
        keep.append(a)
        setattr(cols, slot, ptr(a).value)
    return cols, keep


class HeightInterpolator(_VerticalHandle):
    """Interpolates [nt][nk][...] fields on the source vertical coordinate to [nt][np][...] on target levels in metres: above the
    ground (``type="height"``) or above sea level (``type="altitude"``).  The altitude of every source level comes from
    ``converter``:

    * ``"hypsometric"``: integrated upward from the surface over the air temperature ``t`` [K] and, when given, the specific
      humidity ``q`` [kg/kg]; hybrid or sigma source levels only;
    * ``"standard"``: the standard-atmosphere altitude of each level's pressure [hPa after ``ps_scale``];
    * ``"field"``: ``z_scale * z`` for a per-level field ``z`` (geopotential: ``z_scale = 1 / 9.80665``); the terms only give nk.

    ``zs`` [...] is the surface altitude (times ``zs_scale``; surface geopotential: ``1 / 9.80665``): height targets of the standard
    and field converters and altitude targets of the hypsometric one need it.  ``ps`` [nt][...], ``t``, ``q``, ``z`` [nt][nk][...]
    are float32.  Methods: ``linear`` and ``nearestneighbor`` (``log`` and ``loglog`` are defined on ln p)."""

    def __init__(self, standard_name: str, terms: dict, method: str, levels, type: str = "height", converter: str = "hypsometric",
                 ps_scale: float = 1.0, z_scale: float = 1.0, zs_scale: float = 1.0, extrapolate: bool = True):
        self.method = vertical_method(method)
        if self.method not in (METHODS["linear"], METHODS["nearestneighbor"]):
            raise FimexB200Error(f"height levels take the methods linear and nearestneighbor only (log and loglog are defined on ln p), "
                                 f"got '{method}'")
        if type not in TARGETS:
            raise FimexB200Error(f"unknown height target type: '{type}' (one of {', '.join(TARGETS)})")
        if converter not in CONVERTERS:
            raise FimexB200Error(f"unknown height converter: '{converter}' (one of {', '.join(CONVERTERS)})")
        self.levels = f64(levels).ravel()
        self._h = C.c_void_p()
        vcoord, a, b, ptop, self.nk = _source_levels(standard_name, terms)
        if converter == "hypsometric" and vcoord == VCOORD_PRESSURE:
            raise FimexB200Error("the hypsometric converter needs a surface pressure: hybrid or sigma source levels, not pressure levels")
        self.needs_ps = converter == "hypsometric" or (converter == "standard" and vcoord != VCOORD_PRESSURE)
        self.needs_t = converter == "hypsometric"
        self.needs_z = converter == "field"
        self.needs_zs = (type == "height") != (converter == "hypsometric")
        lib = load()
        rc = lib.fb200_vinterp_create_height(self.method, CONVERTERS[converter], TARGETS[type], vcoord, ptr(a), ptr(b), self.nk, ptop,
                                             float(ps_scale), float(z_scale), float(zs_scale), ptr(self.levels), self.levels.size,
                                             int(bool(extrapolate)), C.byref(self._h))
        check(rc, "HeightInterpolator")

    def _columns(self, nt, nxy, device, ps, t, q, z, zs):
        """the fb200_vcolumns of a call, and the arrays it points into (kept alive by the caller)"""
        level, column = nt * nxy, nt * self.nk * nxy
        given = {"ps": (ps, self.needs_ps, level, "the surface pressure ps"),
                 "t": (t, self.needs_t, column, "the air temperature t"),
                 "q": (q, self.needs_t, column, "the specific humidity q"),
                 "z": (z, self.needs_z, column, "the altitude field z"),
                 "zs": (zs, self.needs_zs, nxy, "the surface altitude zs")}
        slots = {}
        for name, (a, used, n, what) in given.items():
            if a is None or not used:
                if used and name != "q":
                    raise FimexB200Error(f"this converter and target need {what}")
                continue
            slots[name] = (name, a, n)
        return _fill_columns(slots, device)

    def interpolateValues(self, field, ps=None, t=None, q=None, z=None, zs=None, stream=None):
        """float32 [nt][nk][...] with NaN for undefined values -> float32 [nt][np][...] (numpy or CUDA tensors)"""
        return self._values_columns(field, ps, lambda nt, nxy, device: self._columns(nt, nxy, device, ps, t, q, z, zs), stream)

    def getDataSlice(self, field, ps=None, t=None, q=None, z=None, zs=None, bad_value=None, out_dtype=None, stream=None):
        """The per-slice body of the vertical getDataSlice: `field` [nt][nk][...] of any CDM numeric type (numpy array, or CUDA tensor
        for the device-resident path), fill -> NaN, interpolate, NaN -> fill and cast to `out_dtype` (default: the input's type).
        `bad_value` = CDM::getFillValue of the variable (default: the type's default fill value)."""
        return self._slice_columns(field, ps, lambda nt, nxy, device: self._columns(nt, nxy, device, ps, t, q, z, zs), bad_value, out_dtype,
                                   stream)


def _depth_source(standard_name: str, terms: dict):
    """(vcoord, s, C, depth_c) of the source vertical coordinate of a depth handle: depth levels s = the levels; ocean sigma s = sigma;
    g1, g2 s, C, depth_c.  The fields eta and depth of the ocean coordinates are not terms here."""
    def need(t, *names):
        missing = [n for n in names if n not in t]
        if missing:
            raise FimexB200Error(f"{standard_name} needs the terms {', '.join(names)}; got {sorted(terms)}")
    if standard_name == DEPTH:
        need(terms, "depth")
        return VCOORD_DEPTH, f64(terms["depth"]).ravel(), None, 0.0
    t = {k: v for k, v in terms.items() if k not in ("eta", "depth")}
    if standard_name == OCEAN_SIGMA:
        need(t, "sigma")
        return VCOORD_OCEAN_SIGMA, f64(t["sigma"]).ravel(), None, 0.0
    if standard_name in (OCEAN_S_G1, OCEAN_S_G2):
        need(t, "s", "C", "depth_c")
        s, Ck = f64(t["s"]).ravel(), f64(t["C"]).ravel()
        if s.size != Ck.size:
            raise FimexB200Error(f"{standard_name}: {s.size} values of s but {Ck.size} of C")
        vcoord = VCOORD_OCEAN_S_G1 if standard_name == OCEAN_S_G1 else VCOORD_OCEAN_S_G2
        return vcoord, s, Ck, float(np.asarray(t["depth_c"], dtype=np.float64).reshape(-1)[0])
    raise FimexB200Error(f"vertical coordinate '{standard_name}' is not supported for depth levels "
                         f"(one of {DEPTH}, {OCEAN_SIGMA}, {OCEAN_S_G1}, {OCEAN_S_G2})")


class DepthInterpolator(_VerticalHandle):
    """Interpolates [nt][nk][...] fields on the source vertical coordinate to [nt][np][...] on target depths in metres below the sea
    surface datum, positive down (``--verticalInterpolate.type=depth``).  Source coordinates and their terms:

    * ``depth``: depth levels, positive down, ``{"depth": levels}``;
    * ``ocean_sigma_coordinate``: ``{"sigma": sigma}``;
    * ``ocean_s_coordinate_g1`` and ``_g2``: ``{"s": s, "C": C, "depth_c": depth_c}``.

    The ocean coordinates read two fields with every slice: ``depth`` [...], the sea-floor depth h [m, positive down], which they
    need, and ``eta`` [nt][...], the sea surface height [m] (None: 0), both float32.  A column with h NaN or <= 0 (land) or a NaN eta
    gives NaN.  Methods: ``linear`` and ``nearestneighbor``."""

    def __init__(self, standard_name: str, terms: dict, method: str, levels, extrapolate: bool = True):
        self.method = vertical_method(method)
        if self.method not in (METHODS["linear"], METHODS["nearestneighbor"]):
            raise FimexB200Error(f"depth levels take the methods linear and nearestneighbor only (log and loglog are defined on ln p), "
                                 f"got '{method}'")
        self.levels = f64(levels).ravel()
        self._h = C.c_void_p()
        vcoord, s, Ck, depth_c = _depth_source(standard_name, terms)
        self.nk = s.size
        self.needs_depth = vcoord != VCOORD_DEPTH
        rc = load().fb200_vinterp_create_depth(self.method, vcoord, ptr(s), ptr(Ck), self.nk, depth_c, ptr(self.levels), self.levels.size,
                                               int(bool(extrapolate)), C.byref(self._h))
        check(rc, "DepthInterpolator")

    def _columns(self, nt, nxy, device, eta, depth):
        """the fb200_vcolumns of a call (eta in the ps slot, the sea-floor depth in the zs slot), and the arrays it points into"""
        slots = {}
        if self.needs_depth:
            if depth is None:
                raise FimexB200Error("ocean s- and sigma coordinates need the sea-floor depth")
            slots["zs"] = ("depth", depth, nxy)
            if eta is not None:
                slots["ps"] = ("eta", eta, nt * nxy)
        return _fill_columns(slots, device)

    def interpolateValues(self, field, eta=None, depth=None, stream=None):
        """float32 [nt][nk][...] with NaN for undefined values -> float32 [nt][np][...] (numpy or CUDA tensors)"""
        return self._values_columns(field, None, lambda nt, nxy, device: self._columns(nt, nxy, device, eta, depth), stream)

    def getDataSlice(self, field, eta=None, depth=None, bad_value=None, out_dtype=None, stream=None):
        """The per-slice body of the vertical getDataSlice: `field` [nt][nk][...] of any CDM numeric type (numpy array, or CUDA tensor
        for the device-resident path), fill -> NaN, interpolate, NaN -> fill and cast to `out_dtype` (default: the input's type).
        `bad_value` = CDM::getFillValue of the variable (default: the type's default fill value)."""
        return self._slice_columns(field, None, lambda nt, nxy, device: self._columns(nt, nxy, device, eta, depth), bad_value, out_dtype,
                                   stream)


#: --verticalInterpolate.dataConversion values -> FB200_VCONV_*
CONVERSIONS = {"theta2T": 0, "omega2vwind": 1, "add4Dpressure": 2}


class PressureConversion(_VerticalHandle):
    """The data conversions of the vertical interpolator on the model levels (``--verticalInterpolate.dataConversion``, the
    reference's CDMPressureConversions), each on the column pressure p_k [hPa] of the source vertical coordinate (terms as for
    :class:`VerticalInterpolator`; ``ps_scale`` converts ``ps`` to hPa):

    * ``"theta2T"``: air potential temperature -> air temperature, ``T = theta (p_k / 1000)^(2/7)`` [K];
    * ``"omega2vwind"``: omega [Pa/s] and the air temperature ``t`` [K] -> upward air velocity ``w = -omega R_d T / (g0 p_k)`` [m/s];
    * ``"add4Dpressure"``: the pressure field p_k itself [hPa], [nt][nk][...]; there is no input field.

    Float32 in, float32 out; numpy arrays (host buffers) or CUDA tensors (device-resident, on ``stream``)."""

    _destroy = "fb200_vconvert_destroy"

    def __init__(self, standard_name: str, terms: dict, operation: str, ps_scale: float = 1.0):
        if operation not in CONVERSIONS:
            raise FimexB200Error(f"unknown data conversion: '{operation}' (one of {', '.join(CONVERSIONS)})")
        self.operation = operation
        self._h = C.c_void_p()
        vcoord, a, b, ptop, self.nk = _source_levels(standard_name, terms)
        self.needs_ps = vcoord != VCOORD_PRESSURE
        self.needs_t = operation == "omega2vwind"
        check(load().fb200_vconvert_create(CONVERSIONS[operation], vcoord, ptr(a), ptr(b), self.nk, ptop, float(ps_scale), C.byref(self._h)),
              "PressureConversion")

    def convert(self, field=None, ps=None, t=None, nt=None, stream=None):
        """``field`` [nt][nk][...] (theta or omega; None for add4Dpressure), ``ps`` [nt][...] (hybrid and sigma levels), ``t``
        [nt][nk][...] (omega2vwind) -> float32 [nt][nk][...].  add4Dpressure takes its shape from ``ps``, or on pressure levels from
        ``nt``: [nt][nk]."""
        pressure = self.operation == "add4Dpressure"
        if pressure:
            if ps is not None:
                nt_, nxy, rest = int(ps.shape[0]), int(np.prod(ps.shape[1:], dtype=np.int64)), tuple(ps.shape[1:])
            elif self.needs_ps:
                raise FimexB200Error("this vertical coordinate needs the surface pressure ps")
            elif nt is None:
                raise FimexB200Error("add4Dpressure on pressure levels needs nt")
            else:
                nt_, nxy, rest = int(nt), 1, ()
            device = _is_torch(ps)
        else:
            if field is None:
                raise FimexB200Error(f"{self.operation} needs the field")
            device = _is_torch(field)
            if field.ndim < 2 or field.shape[1] != self.nk:
                raise FimexB200Error(f"field must be [nt][{self.nk}][...], got shape {tuple(field.shape)}")
            nt_, nxy, rest = int(field.shape[0]), int(np.prod(field.shape[2:], dtype=np.int64)), tuple(field.shape[2:])
        slots = {}
        if self.needs_ps:
            if ps is None:
                raise FimexB200Error("this vertical coordinate needs the surface pressure ps")
            slots["ps"] = ("ps", ps, nt_ * nxy)
        if self.needs_t:
            if t is None:
                raise FimexB200Error("omega2vwind needs the air temperature t")
            slots["t"] = ("t", t, nt_ * self.nk * nxy)
        cols, keep = _fill_columns(slots, device)
        shape = (nt_, self.nk) + rest
        lib = load()
        if device:
            import torch
            d_in = None
            if not pressure:
                if not field.is_cuda or field.dtype != torch.float32 or not field.is_contiguous():
                    raise FimexB200Error("device path needs a contiguous float32 CUDA tensor")
                d_in = field
            out = torch.empty(shape, dtype=torch.float32, device=ps.device if pressure else field.device)
            check(lib.fb200_vconvert_values_device(self._h, ptr(d_in), C.byref(cols), nxy, nt_, ptr(out), _stream_ptr(stream)), "convert")
            return out
        a = None if pressure else capi.f32(field)
        out = np.empty(shape, dtype=np.float32)
        check(lib.fb200_vconvert_values(self._h, ptr(a), C.byref(cols), nxy, nt_, ptr(out)), "convert")
        return out
