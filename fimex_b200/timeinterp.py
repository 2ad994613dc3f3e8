"""Host-side mirror of the reference's CDMTimeInterpolator (``--timeInterpolate.timeSpec``): the linear change of the time axis,
with the blend on the GPU (libfimex_b200.so, include/fimex_b200.h section (1h); DESIGN.md section 2 states the arithmetic).

A :class:`TimeInterpolator` is built from the data's time values and their CF unit, ``"<seconds|minutes|hours|days> since
YYYY-MM-DD[ HH:MM[:SS]]"`` in the standard (Gregorian) or proleptic Gregorian calendar, and from either explicit target times in
that unit or a time specification.  The subset of the reference's TimeSpec implemented here, with numpy ``datetime64`` arithmetic:

* absolute times: a comma list of ``YYYY-MM-DD HH:MM:SS``, e.g. ``2000-01-01 00:00:00,2000-01-01 06:00:00``;
* sequences: ``a,b,...,c`` is ``a + i (b - a)`` for i = 0, 1, ... up to and including ``c`` (b > a); values listed before
  ``a`` are kept as they are.  ``x`` stands for the last source time;
* the relative form ``v1,v2,...;relativeStart=R;unit=U`` (U one of seconds, minutes, hours, days; relativeStart defaults to 0):
  target = base + (R + v) U, where base is the first source time rounded down to a whole U; ``x`` is the last source time as
  such an offset.

Anything else raises :class:`~fimex_b200.capi.FimexB200Error`.  The standard calendar is read as proleptic Gregorian, which it
equals from 1582-10-15 on; earlier times are refused in it.
"""
from __future__ import annotations

import ctypes as C
import re

import numpy as np

from . import capi
from .cached import _is_torch, _stream_ptr
from .capi import FimexB200Error, check, f64, load, ptr

_UNIT_SECONDS = {"second": 1, "seconds": 1, "minute": 60, "minutes": 60, "hour": 3600, "hours": 3600, "day": 86400, "days": 86400}
_CALENDARS = ("standard", "gregorian", "proleptic_gregorian")
_GREGORIAN_START = np.datetime64("1582-10-15T00:00:00", "s")
_CF_UNIT = re.compile(r"^\s*([A-Za-z]+)\s+since\s+(\d{1,4})-(\d{1,2})-(\d{1,2})(?:[ T](\d{1,2}):(\d{1,2})(?::(\d{1,2}))?)?\s*(?:Z|UTC)?\s*$")
_ABS_TIME = re.compile(r"^(\d{4})-(\d{2})-(\d{2}) (\d{2}):(\d{2}):(\d{2})$")
_EPOCH = np.datetime64("1970-01-01T00:00:00", "s")


def _datetime(y, mo, d, h=0, mi=0, s=0, what="time"):
    try:
        return np.datetime64(f"{int(y):04d}-{int(mo):02d}-{int(d):02d}T{int(h):02d}:{int(mi):02d}:{int(s):02d}", "s")
    except ValueError:
        raise FimexB200Error(f"invalid {what}") from None


def parse_time_unit(unit: str, calendar: str = "standard"):
    """CF time unit -> (seconds of one unit, the epoch as datetime64[s]); other units and calendars raise"""
    if calendar not in _CALENDARS:
        raise FimexB200Error(f"calendar '{calendar}' is not supported (one of {', '.join(_CALENDARS)})")
    m = _CF_UNIT.match(unit or "")
    if not m or m.group(1).lower() not in _UNIT_SECONDS:
        raise FimexB200Error(f"time unit '{unit}' is not '<seconds|minutes|hours|days> since YYYY-MM-DD[ HH:MM[:SS]]'")
    epoch = _datetime(*(g or 0 for g in m.groups()[1:]), what=f"date in the time unit '{unit}'")
    return _UNIT_SECONDS[m.group(1).lower()], epoch


#: the most target times one handle takes (fb200_tinterp_create)
MAX_TARGETS = 1 << 20


def expand_sequence(tokens, last):
    """TimeSpec values -> floats: 'x' is `last`, 'a,b,...,c' is a + i (b - a) for i = 0 ... n, b > a.  The tokens are already
    numbers (or 'x' / '...').  n = floor((c - a) / (b - a) + 1e-9): c is included when it lies within 1e-9 of a step of the last
    value, so that a decimal step such as 0.1, which does not divide c - a exactly in binary, still reaches c.  More than
    MAX_TARGETS values raise before any is formed."""
    tokens = [last if t == "x" else t for t in tokens]
    if "..." not in tokens:
        if len(tokens) > MAX_TARGETS:
            raise FimexB200Error(f"more than {MAX_TARGETS} target times")
        return [float(t) for t in tokens]
    i = tokens.index("...")
    if i < 2 or i != len(tokens) - 2 or tokens.count("...") != 1:
        raise FimexB200Error("'...' needs two values before it and one after it: a,b,...,c")
    head = [float(t) for t in tokens[:i]]
    a, b, c = head[-2], head[-1], float(tokens[-1])
    if not b > a:
        raise FimexB200Error(f"the step of a,b,...,c must be positive, got {a},{b}")
    span = (c - a) / (b - a) + 1e-9
    if not span < MAX_TARGETS:  # also refuses an infinite or NaN span
        raise FimexB200Error(f"'{a},{b},...,{c}' gives more than {MAX_TARGETS} target times")
    n = int(np.floor(span))
    if len(head) - 2 + n + 1 > MAX_TARGETS:
        raise FimexB200Error(f"more than {MAX_TARGETS} target times")
    return head[:-2] + [a + k * (b - a) for k in range(n + 1)]


def expand_time_spec(spec: str, times, unit: str, calendar: str = "standard") -> np.ndarray:
    """the target times of a time specification (the subset in this module's docstring), in the data's unit"""
    unit_s, epoch = parse_time_unit(unit, calendar)
    src = f64(times).ravel()
    if src.size == 0:
        raise FimexB200Error("no source times")
    offset = float((epoch - _EPOCH) / np.timedelta64(1, "s"))  # the epoch in seconds since 1970-01-01
    first_s, last_s = offset + src[0] * unit_s, offset + src[-1] * unit_s  # source times in seconds since 1970-01-01
    parts = [p.strip() for p in (spec or "").split(";")]
    tokens = [t.strip() for t in parts[0].split(",")]
    if not parts[0] or any(not t for t in tokens):
        raise FimexB200Error(f"empty value in the time specification '{spec}'")
    if len(parts) == 1:  # absolute times, in seconds since 1970-01-01
        vals = []
        for t in tokens:
            m = _ABS_TIME.match(t)
            if t in ("x", "..."):
                vals.append(t)
            elif m:
                vals.append(float((_datetime(*m.groups(), what=f"time '{t}'") - _EPOCH) / np.timedelta64(1, "s")))
            else:
                raise FimexB200Error(f"'{t}' is not a time 'YYYY-MM-DD HH:MM:SS' (a relative specification needs ';unit=')")
        abs_s = np.asarray(expand_sequence(vals, last_s), dtype=np.float64)
    else:
        opts = {}
        for p in parts[1:]:
            key, eq, value = p.partition("=")
            if not eq or key.strip() not in ("relativeStart", "unit") or key.strip() in opts:
                raise FimexB200Error(f"'{p}' in the time specification: expected relativeStart=R or unit=U once each")
            opts[key.strip()] = value.strip()
        u = opts.get("unit", "")
        if u not in _UNIT_SECONDS:
            raise FimexB200Error(f"the relative time specification needs unit=<seconds|minutes|hours|days>, got '{u}'")
        try:
            start = float(opts.get("relativeStart", "0"))
            rel = [t if t in ("x", "...") else float(t) for t in tokens]
        except ValueError:
            raise FimexB200Error(f"'{spec}': the values of a relative time specification are numbers, 'x' or '...'") from None
        us = _UNIT_SECONDS[u]
        base = np.floor(first_s / us) * us
        last_rel = (last_s - base) / us - start
        abs_s = base + (start + np.asarray(expand_sequence(rel, last_rel), dtype=np.float64)) * us
    if calendar != "proleptic_gregorian":
        gs = float((_GREGORIAN_START - _EPOCH) / np.timedelta64(1, "s"))
        if min(first_s, float(abs_s.min())) < gs:
            raise FimexB200Error("times before 1582-10-15 in the standard calendar are not supported (use proleptic_gregorian)")
    return (abs_s - offset) / unit_s


class TimeInterpolator:
    """The hot-path half of CDMTimeInterpolator: [nt][...] source steps at ``times`` (CF ``unit``) -> [nt_new][...] at the new axis
    ``self.times`` (same unit), from ``new_times`` (in that unit) or a ``time_spec`` string.  ``extrapolate``: targets outside the
    source range use the end pair on that side (default); off, they give NaN, stored as the fill value."""

    def __init__(self, times, unit: str, new_times=None, time_spec: str = None, extrapolate: bool = True, calendar: str = "standard"):
        if (new_times is None) == (time_spec is None):
            raise FimexB200Error("give either new_times or time_spec")
        self._h = C.c_void_p()
        self.source_times = f64(times).ravel()
        self.unit = unit
        self.extrapolate = bool(extrapolate)
        parse_time_unit(unit, calendar)
        self.times = f64(new_times).ravel() if time_spec is None else expand_time_spec(time_spec, self.source_times, unit, calendar)
        check(load().fb200_tinterp_create(ptr(self.source_times), self.source_times.size, ptr(self.times), self.times.size,
                                          int(bool(extrapolate)), C.byref(self._h)), "TimeInterpolator")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            load().fb200_tinterp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def source_steps(self, j: int):
        """(ia, ib, w) of target step j: output = step ia + w (step ib - step ia); ia = ib = -1 where no bracket applies"""
        ia, ib, w = C.c_int(), C.c_int(), C.c_double()
        check(load().fb200_tinterp_source_steps(self._h, int(j), C.byref(ia), C.byref(ib), C.byref(w)), "source_steps")
        return ia.value, ib.value, w.value

    @staticmethod
    def _types(x, bad_value, out_dtype):
        odt = out_dtype if out_dtype is not None else x.dtype
        bad = capi.default_fill_value(x.dtype) if bad_value is None else float(bad_value)
        return odt, bad

    def get_data_slice_step(self, j: int, a, b, bad_value=None, out_dtype=None, stream=None):
        """Target step j from the source steps the map names (``source_steps(j)``), as the reference's getDataSlice(var, j):
        ``a``, ``b`` of one shape and any CDM numeric type, numpy arrays or CUDA tensors (not read where no bracket applies);
        fill -> NaN, blend, NaN -> fill and cast to ``out_dtype`` (default: the input's type).  ``bad_value`` = the variable's fill
        value (default: the type's default fill value)."""
        lib = load()
        if _is_torch(a):
            import torch
            if not (_is_torch(b) and a.is_cuda and b.is_cuda and a.is_contiguous() and b.is_contiguous()):
                raise FimexB200Error("device path needs two contiguous CUDA tensors")
            if a.dtype != b.dtype or a.shape != b.shape or a.device != b.device:
                raise FimexB200Error("a and b must have one dtype, shape and device")
            odt, bad = self._types(a, bad_value, out_dtype)
            out = torch.empty(a.shape, dtype=odt, device=a.device)
            check(lib.fb200_tinterp_get_step_device(self._h, int(j), int(capi.cdm_type(a.dtype)), ptr(a), ptr(b), a.numel(), bad,
                                                    int(capi.cdm_type(odt)), ptr(out), _stream_ptr(stream)), "get_data_slice_step")
            return out
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        if a.dtype != b.dtype or a.shape != b.shape:
            raise FimexB200Error("a and b must have one dtype and shape")
        odt, bad = self._types(a, bad_value, out_dtype)
        out = np.empty(a.shape, dtype=np.dtype(odt))
        check(lib.fb200_tinterp_get_step(self._h, int(j), int(capi.cdm_type(a.dtype)), ptr(a), ptr(b), a.size, bad, int(capi.cdm_type(odt)),
                                         ptr(out)), "get_data_slice_step")
        return out

    def get_data_slice(self, stack, bad_value=None, out_dtype=None, stream=None):
        """The whole time axis on the device: a contiguous CUDA tensor [nt][...] of any CDM numeric type -> [nt_new][...], every
        source step read once; fill values and types as :meth:`get_data_slice_step`."""
        if not _is_torch(stack) or not stack.is_cuda or not stack.is_contiguous():
            raise FimexB200Error("get_data_slice needs a contiguous CUDA tensor; host arrays go step by step (get_data_slice_step)")
        if stack.ndim < 1 or stack.shape[0] != self.source_times.size:
            raise FimexB200Error(f"stack must be [{self.source_times.size}][...], got shape {tuple(stack.shape)}")
        import torch
        odt, bad = self._types(stack, bad_value, out_dtype)
        n = int(np.prod(stack.shape[1:], dtype=np.int64))
        out = torch.empty((self.times.size,) + tuple(stack.shape[1:]), dtype=odt, device=stack.device)
        check(load().fb200_tinterp_get_data_slice_device(self._h, int(capi.cdm_type(stack.dtype)), ptr(stack), n, bad, int(capi.cdm_type(odt)),
                                                         ptr(out), _stream_ptr(stream)), "get_data_slice")
        return out
