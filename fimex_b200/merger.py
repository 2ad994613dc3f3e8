"""Host-side mirror of CDMMerger -- a "free beneficiary" of the regridding path (SURVEY.md 8f rank 4): every horizontal
interpolation it does goes through the same tables and gather kernels.

Reference (arebru/fimex 0.67.2):
  CDMMerger::setTargetGridFromInner / setTargetGrid / getDataSlice     src/CDMMerger.cc:153-207
  CDMMergerPrivate::makeCDM (smooth -> interpolate -> overlay)          src/CDMMerger.cc:211-229
  CDMMergerPrivate::extendInnerAxis                                     src/CDMMerger.cc:233-274
  CDMBorderSmoothing::getDataSlice (inner/outer blend on the inner grid) src/CDMBorderSmoothing.cc:97-158
  CDMBorderSmoothing_Linear::operator()                                 src/CDMBorderSmoothing_Linear.cc:43-84
  CDMOverlay::getDataSlice (top where defined, else base)               src/CDMOverlay.cc:63-92
  makeMergedCDM (outer interpolated to the inner grid)                  src/CDMMergeUtils.cc:214-246

One merged slice is one call of fb200_merge_get_data_slice[_device] (include/fimex_b200.h, section 1i): the outer -> inner
gather, the linear border blend on the inner grid, the blended inner -> target gather, the outer -> target gather and the overlay
all run on the GPU, on the three `Interpolator` handles built by setTargetGrid.  `linear_border_smoothing` below restates the
blend in numpy; it is the reference the tests hold the kernel to, not part of the slice path.  As in interpolator.py the CDM
side (which variables, coordinate systems, units) stays with the host application: grids are described by proj4 string and
axes.
"""
from __future__ import annotations

import ctypes as C
import re

import numpy as np

from . import capi
from .cached import _is_torch, _stream_ptr
from .capi import FimexB200Error, Method, check, load, ptr
from .interpolator import Interpolator

_LINEAR = re.compile(r"\s*LINEAR\s*\(\s*(\d+)\s*,\s*(\d+)\s*\)\s*")


def parse_smoothing(spec):
    """--merge.smoothing (CDMBorderSmoothing_LinearFactory): "LINEAR(transitionWidth,borderWidth)" -> (t, b), integers with t >= 1
    (the blend divides by it) and b >= 0; anything else raises"""
    m = _LINEAR.fullmatch(spec) if isinstance(spec, str) else None
    if m is None:
        raise FimexB200Error(f"cannot parse smoothing '{spec}': expected LINEAR(transitionWidth,borderWidth)")
    t, b = int(m.group(1)), int(m.group(2))
    if t < 1:
        raise FimexB200Error(f"smoothing '{spec}': the transition width must be at least 1")
    return t, b


def extend_inner_axis(inner, outer):
    """CDMMergerPrivate::extendInnerAxis (:233-274): the inner axis continued with its own step over the outer axis' range"""
    vi, vo = np.asarray(inner, dtype=np.float64), np.asarray(outer, dtype=np.float64)
    if vi.size < 2:
        raise FimexB200Error("no data for axis in inner")
    if vo.size < 2:
        raise FimexB200Error("no data for axis in outer")
    step_i, step_o = vi[1] - vi[0], vo[1] - vo[0]
    close = lambda a, b: abs(a - b) <= 1e-5 * max(abs(a), abs(b), 1e-30)  # `equal()` of the reference: relative comparison
    if not all(close(d, step_i) for d in np.diff(vi)):
        raise FimexB200Error("axis in inner does not have constant step size, cannot merge")
    if not all(close(d, step_o) for d in np.diff(vo)):
        raise FimexB200Error("axis in outer does not have constant step size, cannot merge")
    min_i, max_i = (vi[0], vi[-1]) if step_i > 0 else (vi[-1], vi[0])
    min_o, max_o = (vo[0], vo[-1]) if step_o > 0 else (vo[-1], vo[0])
    if min_i < min_o or max_i > max_o:
        raise FimexB200Error("top not inside  bottom")
    before = []
    n = vi[0] - step_i
    while min_o <= n <= max_o:
        before.append(n)
        n -= step_i
    after = []
    n = vi[-1] + step_i
    while min_o <= n <= max_o:
        after.append(n)
        n += step_i
    return np.concatenate([np.array(before[::-1], dtype=np.float64), vi, np.array(after, dtype=np.float64)])


def linear_border_smoothing(inner, outer, transition_width=5, border_width=2, use_outer_if_inner_undefined=True):
    """CDMBorderSmoothing::getDataSlice + CDMBorderSmoothing_Linear (defaults :55 of the header): `inner` and `outer` are
    [.., ny, nx] float64 arrays ON THE INNER GRID (NaN = undefined); outside the border the outer value, in the interior the inner
    one, a linear ramp over `transition_width` cells in between (corner distances are Euclidean)"""
    vi, vo = np.asarray(inner, dtype=np.float64), np.asarray(outer, dtype=np.float64)
    ny, nx = vi.shape[-2:]
    x = np.arange(nx)[None, :] + np.zeros((ny, 1), dtype=np.int64)
    y = np.arange(ny)[:, None] + np.zeros((1, nx), dtype=np.int64)
    xmin1, ymin1 = border_width, border_width
    xmax1, ymax1 = xmin1 + transition_width, ymin1 + transition_width
    xmax2, ymax2 = nx - border_width, ny - border_width
    xmin2, ymin2 = xmax2 - transition_width, ymax2 - transition_width
    dx = np.where(x < xmax1, xmax1 - x, np.where(x >= xmin2, x - xmin2, 0)).astype(np.float64)
    dy = np.where(y < ymax1, ymax1 - y, np.where(y >= ymin2, y - ymin2, 0)).astype(np.float64)
    alpha = np.clip(np.sqrt(dx * dx + dy * dy) / transition_width, 0.0, 1.0)  # one of dx, dy is 0 along the edges: dist == the other
    outside = (x < xmin1) | (x >= xmax2) | (y < ymin1) | (y >= ymax2)
    inside = (x >= xmax1) & (x < xmin2) & (y >= ymax1) & (y < ymin2)
    blended = vi + alpha * (vo - vi)
    blended = np.where(vo - vi == 0, vo, blended)
    merged = np.where(outside, vo, np.where(inside, vi, blended))
    merged = np.where(np.isnan(vo), vi, merged)  # outer undefined (or no smoothing): the inner value
    return np.where(np.isnan(vi), vo if use_outer_if_inner_undefined else np.nan, merged)


class _MergeHandle:
    """fb200_merge: borrows the three interpolation handles, so it keeps their owners alive"""

    def __init__(self, o2i, i2t, o2t, inner_shape, outer_shape, t, b, use_outer):
        self.keep = (o2i, i2t, o2t)
        self.key = (t, b, bool(use_outer))
        self._h = C.c_void_p()
        (nyi, nxi), (nyo, nxo) = inner_shape, outer_shape
        check(load().fb200_merge_create(o2i._h, i2t._h, o2t._h, nxi, nyi, nxo, nyo, int(t), int(b), int(bool(use_outer)), C.byref(self._h)),
              "CDMMerger")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            load().fb200_merge_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _fill_for(dtype, value):
    """the bad / fill value of a slice: as given, else NaN for floating types and defaultFillValue_ for integer types"""
    if value is not None:
        return float(value)
    return float("nan") if np.dtype(str(dtype).replace("torch.", "")).kind == "f" else capi.default_fill_value(dtype)


class Merger:
    """CDMMerger for one variable's horizontal coordinate systems: an inner (fine, small) grid merged into an outer (coarse,
    large) one on a target grid.

    proj_inner / proj_outer : proj4 strings; x/y axes in the projection's unit, degrees when `is_degree` (the inner grid's, and the
    outer grid's too unless `outer_is_degree` says otherwise: a projected inner grid inside a lat/lon outer one)
    """

    def __init__(self, proj_inner, x_inner, y_inner, proj_outer, x_outer, y_outer, is_degree, outer_is_degree=None):
        self.proj_inner, self.proj_outer = proj_inner, proj_outer
        self.x_inner, self.y_inner = np.asarray(x_inner, dtype=np.float64), np.asarray(y_inner, dtype=np.float64)
        self.x_outer, self.y_outer = np.asarray(x_outer, dtype=np.float64), np.asarray(y_outer, dtype=np.float64)
        self.is_degree = bool(is_degree)
        self.outer_is_degree = self.is_degree if outer_is_degree is None else bool(outer_is_degree)
        self.gridInterpolationMethod = Method.BILINEAR  # src/CDMMerger.cc:84
        self.transitionWidth, self.borderWidth = 5, 2   # CDMBorderSmoothing_LinearFactory defaults
        self.useOuterIfInnerUndefined = True
        self._outer_to_inner = None
        self._inner_to_target = None
        self._outer_to_target = None
        self._merge = None

    def setGridInterpolationMethod(self, method):
        """takes effect with the next setTargetGrid / setTargetGridFromInner, as in the reference"""
        self.gridInterpolationMethod = Method(int(method))

    def setSmoothing(self, spec):
        """CDMMerger::setSmoothing with the --merge.smoothing option string, e.g. "LINEAR(5,2)" """
        self.transitionWidth, self.borderWidth = parse_smoothing(spec)
        if self._outer_to_target is not None:
            self._merge_handle()
        return self

    def setUseOuterIfInnerUndefined(self, flag):
        """CDMBorderSmoothing::setUseOuterIfInnerUndefined"""
        self.useOuterIfInnerUndefined = bool(flag)
        return self

    def _merge_handle(self):
        """the fb200_merge handle of the current target grid and smoothing, rebuilt whenever one of them has changed"""
        key = (self.transitionWidth, self.borderWidth, bool(self.useOuterIfInnerUndefined))
        if self._merge is None or self._merge.key != key:
            if not (int(self.transitionWidth) >= 1 and int(self.borderWidth) >= 0):
                raise FimexB200Error(f"smoothing LINEAR({self.transitionWidth},{self.borderWidth}): the transition width must be at least 1 "
                                     "and the border width at least 0")
            self._merge = None
            self._merge = _MergeHandle(self._outer_to_inner.cachedInterpolation, self._inner_to_target.cachedInterpolation,
                                       self._outer_to_target.cachedInterpolation, (self.y_inner.size, self.x_inner.size),
                                       (self.y_outer.size, self.x_outer.size), self.transitionWidth, self.borderWidth, self.useOuterIfInnerUndefined)
        return self._merge

    def setTargetGrid(self, proj, tx, ty, tx_unit="m", ty_unit="m"):
        """CDMMerger::setTargetGrid -> makeCDM (:211-229)"""
        unit = "degree" if self.is_degree else "m"
        m = self.gridInterpolationMethod
        self._merge = None
        # readerSmooth: outer interpolated onto the INNER grid (makeMergedCDM, CDMMergeUtils.cc:234-243)
        self._outer_to_inner = Interpolator(self.proj_outer, self.x_outer, self.y_outer, self.outer_is_degree)
        self._outer_to_inner.changeProjection(m, self.proj_inner, self.x_inner, self.y_inner, unit, unit)
        # interpolatedST: the smoothed inner field onto the target grid
        self._inner_to_target = Interpolator(self.proj_inner, self.x_inner, self.y_inner, self.is_degree)
        self._inner_to_target.changeProjection(m, proj, tx, ty, tx_unit, ty_unit)
        # readerOverlay: the outer field onto the target grid, underneath
        self._outer_to_target = Interpolator(self.proj_outer, self.x_outer, self.y_outer, self.outer_is_degree)
        self._outer_to_target.changeProjection(m, proj, tx, ty, tx_unit, ty_unit)
        self.target_shape = (len(np.atleast_1d(ty)) if not isinstance(ty, str) else None, len(np.atleast_1d(tx)) if not isinstance(tx, str) else None)
        self._merge_handle()
        return self

    def setTargetGridFromInner(self):
        """CDMMerger::setTargetGridFromInner (:153-196): the inner grid extended over the outer grid's range, inner projection"""
        if self.proj_inner is None or self.proj_outer is None:
            raise FimexB200Error("extending grid failed, no inner variable with CS found")
        unit = "degree" if self.is_degree else "m"
        vx = extend_inner_axis(self.x_inner, self.x_outer)
        vy = extend_inner_axis(self.y_inner, self.y_outer)
        self.target_x, self.target_y = vx, vy
        return self.setTargetGrid(self.proj_inner, vx, vy, unit, unit)

    def getDataSlice(self, inner, outer, inner_bad_value=None, outer_bad_value=None, out_dtype=None, out_fill=None, stream=None):
        """One merged slice in one call (CDMMerger::getDataSlice): `inner` [.., nyI, nxI] and `outer` [.., nyO, nxO] with the same
        leading dimensions, of one CDM type -- numpy arrays (host buffers) or contiguous CUDA tensors (the result is a CUDA tensor;
        enqueued on `stream`, default the current torch stream, without synchronising).  Values equal to the bad values are
        undefined (default: NaN for floating types, defaultFillValue_ for integer ones); the result [.., nyT, nxT] is of `out_dtype`
        (default: the inner's type) with undefined cells set to `out_fill` (default: NaN for floating types, defaultFillValue_ for
        integer ones)."""
        if self._outer_to_target is None:
            raise FimexB200Error("must call setTargetGrid or setTargetGridFromInner before getDataSlice")
        mh = self._merge_handle()
        lib = load()
        ci = self._inner_to_target.cachedInterpolation
        ny_t, nx_t = ci.getOutY(), ci.getOutX()
        on_device = _is_torch(inner)
        if on_device:
            import torch
            if not _is_torch(outer) or not (inner.is_cuda and outer.is_cuda) or inner.device != outer.device:
                raise FimexB200Error("inner and outer must both be CUDA tensors on one device")
            if inner.dtype != outer.dtype:
                raise FimexB200Error(f"inner and outer differ in type: {inner.dtype} and {outer.dtype}")
            if not (inner.is_contiguous() and outer.is_contiguous()):
                raise FimexB200Error("device path needs contiguous CUDA tensors")
            dtype = inner.dtype
            odt = out_dtype if out_dtype is not None else dtype
        else:
            vi, vo = np.asarray(inner), np.asarray(outer)
            if vi.dtype != vo.dtype:  # one CDM type for both: the common type both convert to without loss where there is one
                common = np.result_type(vi.dtype, vo.dtype)
                vi, vo = vi.astype(common), vo.astype(common)
            inner, outer = np.ascontiguousarray(vi), np.ascontiguousarray(vo)
            dtype = inner.dtype
            odt = np.dtype(out_dtype) if out_dtype is not None else dtype
        if inner.ndim < 2 or outer.ndim < 2 or tuple(inner.shape[-2:]) != (self.y_inner.size, self.x_inner.size) or \
                tuple(outer.shape[-2:]) != (self.y_outer.size, self.x_outer.size):
            raise FimexB200Error(f"inner {tuple(inner.shape)} and outer {tuple(outer.shape)} do not end in the inner "
                                 f"({self.y_inner.size}, {self.x_inner.size}) and outer ({self.y_outer.size}, {self.x_outer.size}) grids")
        lead = tuple(inner.shape[:-2])
        if tuple(outer.shape[:-2]) != lead:
            raise FimexB200Error(f"inner and outer differ in their leading dimensions: {lead} and {tuple(outer.shape[:-2])}")
        bad_i, bad_o, fill = _fill_for(dtype, inner_bad_value), _fill_for(dtype, outer_bad_value), _fill_for(odt, out_fill)
        in_code, out_code = int(capi.cdm_type(dtype)), int(capi.cdm_type(odt))
        nz = int(np.prod(lead, dtype=np.int64)) if lead else 1
        new_size = C.c_size_t()
        if on_device:
            out = torch.empty(lead + (ny_t, nx_t), dtype=odt, device=inner.device)
            check(lib.fb200_merge_get_data_slice_device(mh._h, in_code, ptr(inner), inner.numel(), bad_i, ptr(outer), outer.numel(), bad_o, out_code,
                                                        fill, ptr(out), C.byref(new_size), _stream_ptr(stream)), "CDMMerger getDataSlice")
        else:
            out = np.empty(lead + (ny_t, nx_t), dtype=odt)
            check(lib.fb200_merge_get_data_slice(mh._h, in_code, ptr(inner), inner.size, bad_i, ptr(outer), outer.size, bad_o, out_code, fill,
                                                 ptr(out), C.byref(new_size)), "CDMMerger getDataSlice")
        assert new_size.value == nz * ny_t * nx_t
        return out
