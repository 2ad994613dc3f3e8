"""The merger on the GPU (fb200_merge_*, fimex_b200.Merger.getDataSlice): one merged slice -- outer -> inner gather, linear border
smoothing, inner -> target gather, outer -> target gather, overlay -- against a reference chain built only from pieces pinned
elsewhere: the oracle's cached_interpolate gathers on each handle's own position table and reduced domain, the numpy restatement
linear_border_smoothing (held to the rule in tests/test_merge_host.py), np.where, and the oracle's as_float / from_float adapters.
The bar is bit-identical values and identical NaN / fill masks, for the host-buffer and the device form.

FIMEX_B200_MERGEFUZZ_SEEDS sets the number of fuzz seeds (default 36)."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import Method  # noqa: E402
from fimex_b200.capi import MIFI_ERROR, MIFI_OK, FimexB200Error  # noqa: E402

SEEDS = int(os.environ.get("FIMEX_B200_MERGEFUZZ_SEEDS", "36"))
LATLON = "+proj=latlong +a=6371000 +e=0 +no_defs"
STERE = "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0 +no_defs"
LCC = "+proj=lcc +lat_0=63 +lon_0=15 +lat_1=63 +lat_2=63 +a=6371000 +e=0 +no_defs"
METHODS = [Method.NEAREST_NEIGHBOR, Method.BILINEAR, Method.BICUBIC]
# (in type, out type, badInner, badOuter, outFill): the three values distinct wherever the types allow
TYPES = [
    (np.int16, np.int16, -999.0, -32767.0, -12345.0),
    (np.int16, np.float32, -32767.0, -999.0, np.nan),
    (np.uint8, np.uint8, 254.0, 253.0, 0.0),
    (np.float32, np.float32, -999.0, np.nan, -1.0e30),
    (np.float32, np.int16, np.nan, -888.0, -32767.0),
    (np.float64, np.float64, np.nan, -888.0, 1.0e36),
    (np.float64, np.float64, -777.0, np.nan, np.nan),
    (np.float64, np.int16, -777.0, -888.0, -32000.0),
]


@pytest.fixture(autouse=True)
def _device():
    fb.set_device(0)


def _same(got, want, what=""):
    """identical bytes; for floating types every non-NaN value bit-identical (signed zeros included) and identical NaN masks"""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.dtype == want.dtype and got.shape == want.shape, f"{what}: {got.dtype}{got.shape} vs {want.dtype}{want.shape}"
    if got.dtype.kind == "f":
        u = {4: np.uint32, 8: np.uint64}[got.dtype.itemsize]
        differ = (got.view(u) != want.view(u)) & ~(np.isnan(got) & np.isnan(want))
    else:
        differ = got != want
    bad = np.flatnonzero(differ)
    assert bad.size == 0, f"{what}: {bad.size} of {got.size} differ, first at {bad[0]}: {got.ravel()[bad[0]]} vs {want.ravel()[bad[0]]}"


def _gather(oracle, interp, field):
    """cached_interpolate on the handle's own (cropped) position table, from the handle's reduced domain of the full source field"""
    ci = interp.cachedInterpolation
    red = ci.reducedDomain()
    x0, y0 = (red[2], red[3]) if red else (0, 0)
    src = np.ascontiguousarray(field[..., y0:y0 + ci.getInY(), x0:x0 + ci.getInX()], dtype=np.float32)
    px, py = ci.points()
    out = oracle.cached_interpolate(int(interp.method), px, py, ci.getInX(), ci.getInY(), ci.getOutX(), ci.getOutY(), src.reshape(-1))
    return out + np.float32(0)  # interpolationArray2Data to float: -0 -> +0 (CDMInterpolator.cc:121-124)


def _reference(oracle, merger, inner, outer, bad_i, bad_o, out_dtype, fill):
    lead = inner.shape[:-2]
    inner3 = inner.reshape((-1,) + inner.shape[-2:])
    outer3 = outer.reshape((-1,) + outer.shape[-2:])
    fo = oracle.as_float(outer3, bad_o)
    on_inner = _gather(oracle, merger._outer_to_inner, fo)
    vi = inner3.astype(np.float64)
    if not np.isnan(bad_i):
        vi[inner3 == np.array(bad_i).astype(inner3.dtype)] = np.nan
    smooth = fb.linear_border_smoothing(vi, on_inner.astype(np.float64), merger.transitionWidth, merger.borderWidth,
                                        merger.useOuterIfInnerUndefined).astype(np.float32)
    top = _gather(oracle, merger._inner_to_target, smooth)
    base = _gather(oracle, merger._outer_to_target, fo)
    merged = np.where(np.isnan(top), base, top)
    return oracle.from_float(merged, fill, out_dtype).reshape(lead + merged.shape[-2:])


def _field(rng, shape, dtype, bad, smooth_base):
    dt = np.dtype(dtype)
    if dt.kind == "f":
        v = smooth_base + rng.normal(0.0, 3.0, shape)  # fp64 values that are not float-representable
        v = v.astype(dt)
    elif dt == np.uint8:
        v = np.clip(np.round(smooth_base / 3.0 + rng.normal(0.0, 5.0, shape)), 0, 240).astype(dt)
    else:
        v = np.round((smooth_base - 273.15) * 50 + rng.normal(0.0, 40.0, shape)).astype(dt)
    hole = rng.random(shape) < 0.05
    if np.isnan(bad):
        if dt.kind == "f":
            v[hole] = np.nan
    else:
        v[hole] = dt.type(bad)
    return v


def _axis(start, step, n):
    return start + step * np.arange(n, dtype=np.float64)


def _geometry(rng, seed):
    """a Merger with its target grid set, and the inner / outer grid shapes; lat/lon pairs, or a projected inner grid in a lat/lon
    outer one; targets from the inner grid extended over the outer one, or a box that reduces all three domains"""
    kind = seed % 4
    t, b = [(5, 2), (1, 0), (10, 3), (3, 1)][seed % 4 if seed % 5 else 2]
    if kind in (0, 1, 2):  # lat/lon pair, inner at a finer step inside the outer grid
        so = float(rng.choice([0.5, 1.0]))
        k = int(rng.choice([2, 4, 5]))
        si = so / k
        nxo, nyo = int(rng.integers(14, 36)), int(rng.integers(12, 30))
        lon0, lat0 = float(rng.uniform(-30, 10)), float(rng.uniform(35, 50))
        xo, yo = _axis(lon0, so, nxo), _axis(lat0 + so * (nyo - 1), -so, nyo)  # descending latitudes, as the reference's files
        # inner: small (below 2 (b + t) where the draw wants it) or up to most of the outer grid
        max_nxi, max_nyi = int((nxo - 5) * so / si), int((nyo - 5) * so / si)
        small = seed % 3 == 0
        nxi = int(rng.integers(2, 2 * (b + t) + 1)) if small else int(rng.integers(min(2 * (b + t), max_nxi - 1), max_nxi))
        nyi = int(rng.integers(2, 2 * (b + t) + 1)) if small else int(rng.integers(min(2 * (b + t), max_nyi - 1), max_nyi))
        nxi, nyi = max(2, min(nxi, max_nxi)), max(2, min(nyi, max_nyi))
        xi = _axis(lon0 + 2 * so + si * int(rng.integers(0, k)), si, nxi)
        yi = _axis(yo[0] - 2 * so - si * int(rng.integers(0, k)), -si, nyi)
        m = fb.Merger(LATLON, xi, yi, LATLON, xo, yo, True)
        m.setGridInterpolationMethod(METHODS[seed % 3])
        m.setSmoothing(f"LINEAR({t},{b})")
        if kind == 0:
            m.setTargetGridFromInner()
        else:  # a box around part of the inner grid: every handle reads a reduced domain
            tx = _axis(xi[0] - 1.3 * so, si * 1.5, int(rng.integers(5, max(6, nxi + 3))))
            ty = _axis(yi[0] + 1.1 * so, -si * 1.5, int(rng.integers(5, max(6, nyi + 3))))
            m.setTargetGrid(LATLON, tx, ty, "degree", "degree")
        return m, (nyi, nxi), (nyo, nxo)
    # a projected inner grid (metres) inside a lat/lon outer one
    proj = STERE if seed % 8 == 3 else LCC
    xo, yo = _axis(-60.0, 2.0, 61), _axis(86.0, -2.0, 27)
    step = float(rng.choice([25000.0, 50000.0]))
    nxi, nyi = int(rng.integers(4, 40)), int(rng.integers(4, 40))
    if proj == STERE:
        x0, y0 = -step * nxi / 2, -2.6e6
    else:
        x0, y0 = -step * nxi / 2, -step * nyi / 2
    xi, yi = _axis(x0, step, nxi), _axis(y0, step, nyi)
    m = fb.Merger(proj, xi, yi, LATLON, xo, yo, False, outer_is_degree=True)
    m.setGridInterpolationMethod(METHODS[seed % 3])
    m.setSmoothing(f"LINEAR({t},{b})")
    tx = _axis(x0 - 3 * step, step * 0.7, nxi + 8)
    ty = _axis(y0 - 3 * step, step * 0.7, nyi + 8)
    m.setTargetGrid(proj, tx, ty, "m", "m")
    return m, (nyi, nxi), (yo.size, xo.size)


def _check(oracle, m, inner, outer, bad_i, bad_o, out_dtype, fill, what, device=True):
    want = _reference(oracle, m, inner, outer, bad_i, bad_o, out_dtype, fill)
    got = m.getDataSlice(inner, outer, bad_i, bad_o, out_dtype, fill)
    _same(got, want, what + " host")
    if device:
        import torch
        gd = m.getDataSlice(torch.from_numpy(inner).cuda(), torch.from_numpy(outer).cuda(), bad_i, bad_o, getattr(torch, np.dtype(out_dtype).name), fill)
        torch.cuda.synchronize()
        _same(gd.cpu().numpy(), want, what + " device")
    return got


@pytest.mark.parametrize("seed", range(SEEDS))
def test_merge_fuzz(oracle, seed):
    rng = np.random.default_rng(4200 + seed)
    m, ishape, oshape = _geometry(rng, seed)
    in_t, out_t, bad_i, bad_o, fill = TYPES[seed % len(TYPES)]
    if seed % 7 == 5:
        m.setUseOuterIfInnerUndefined(False)
    nz = [1, 3, 2, 1, 5][seed % 5]
    lead = (nz,) if seed % 2 else ((1, nz) if nz > 1 else ())
    inner = _field(rng, lead + ishape, in_t, bad_i, 285.0)
    outer = _field(rng, lead + oshape, in_t, bad_o, 280.0)
    _check(oracle, m, inner, outer, bad_i, bad_o, out_t, fill,
           f"seed {seed} {m.gridInterpolationMethod.name} LINEAR({m.transitionWidth},{m.borderWidth}) inner {ishape} outer {oshape} "
           f"{np.dtype(in_t).name}->{np.dtype(out_t).name} nz {nz}")


def _reference_files(fx):
    proj = str(fx["merge_inner_proj4"])
    xi, yi = fx["merge_inner_longitude"].astype(np.float64), fx["merge_inner_latitude"].astype(np.float64)
    xo, yo = fx["merge_outer_longitude"].astype(np.float64), fx["merge_outer_latitude"].astype(np.float64)
    m = fb.Merger(proj, xi, yi, proj, xo, yo, True)
    m.setTargetGridFromInner()
    return m, fx["merge_inner_ga_2t_1"][0, 0], fx["merge_outer_ga_2t_1"][0, 0]


@pytest.fixture(scope="module")
def fx():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "interpolator_fixtures.npz"))


def test_reference_files_host_device_typed(fx, oracle):
    """test/testMerger.cc:44-77 on the reference's files: the three known answers through both forms, and typed slices (int16 with
    fill values, as the files would hold packed temperatures) against the reference chain"""
    import torch
    m, vi, vo = _reference_files(fx)
    known = ((28, 56, 288.104), (24, 56, 288.467), (8, 56, 289.937))
    nan = float("nan")
    for got in (m.getDataSlice(vi, vo), m.getDataSlice(torch.from_numpy(vi).cuda(), torch.from_numpy(vo).cuda()).cpu().numpy()):
        assert got.shape == (113, 61) and got.dtype == np.float64
        for ilon, ilat, expected in known:
            assert abs(got[ilat, ilon] - expected) < 0.001, (ilon, ilat, got[ilat, ilon])
        _same(got, _reference(oracle, m, vi, vo, nan, nan, np.float64, nan), "reference files, float64")
    # packed: 0.01 K above 273.15, two holes in each field with distinct fill values, int16 and float32 out
    pi = np.round((vi - 273.15) * 100).astype(np.int16)
    po = np.round((vo - 273.15) * 100).astype(np.int16)
    pi[20, 10], pi[3, 4] = -999, -999
    po[7, 8], po[0, 0] = -32767, -32767
    for out_t, fill in ((np.int16, -12345.0), (np.float32, nan)):
        got = _check(oracle, m, pi, po, -999.0, -32767.0, out_t, fill, f"reference files int16 -> {np.dtype(out_t).name}")
        if out_t == np.int16:
            for ilon, ilat, expected in known:
                assert abs(got[ilat, ilon] / 100 + 273.15 - expected) < 0.02


def test_large_stack_pageable_staging(oracle):
    """a stack of more than 8 MB of host buffers (the pageable staging path, several pipeline chunks) with a reduced domain on every
    handle: host form and device form against the reference chain"""
    xo, yo = _axis(-20.0, 0.5, 60), _axis(70.0, -0.5, 50)
    xi, yi = _axis(-17.0, 0.1, 220), _axis(67.0, -0.1, 160)
    m = fb.Merger(LATLON, xi, yi, LATLON, xo, yo, True)
    m.setTargetGrid(LATLON, _axis(-18.0, 0.08, 300), _axis(68.0, -0.08, 220), "degree", "degree")
    for h in (m._outer_to_inner, m._inner_to_target, m._outer_to_target):
        assert h.cachedInterpolation.reducedDomain() is not None
    rng = np.random.default_rng(77)
    nz = 24
    inner = _field(rng, (nz,) + (yi.size, xi.size), np.float32, -999.0, 285.0)
    outer = _field(rng, (nz,) + (yo.size, xo.size), np.float32, np.nan, 280.0)
    assert inner.nbytes + outer.nbytes + nz * 300 * 220 * 4 > 8 << 20
    _check(oracle, m, inner, outer, -999.0, np.nan, np.float32, np.nan, "large stack")


def test_device_on_a_side_stream_equals_host(fx):
    import torch
    m, vi, vo = _reference_files(fx)
    rng = np.random.default_rng(5)
    inner = np.stack([vi + rng.normal(0, 1, vi.shape) for _ in range(6)]).astype(np.float32)
    outer = np.stack([vo + rng.normal(0, 1, vo.shape) for _ in range(6)]).astype(np.float32)
    host = m.getDataSlice(inner, outer, out_dtype=np.int16, out_fill=-32767.0)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        di, do = torch.from_numpy(inner).cuda(), torch.from_numpy(outer).cuda()
        got = m.getDataSlice(di, do, out_dtype=torch.int16, out_fill=-32767.0, stream=s)
    s.synchronize()
    _same(got.cpu().numpy(), host, "side stream")


def test_concurrent_calls_on_one_handle(fx):
    m, vi, vo = _reference_files(fx)
    rng = np.random.default_rng(9)
    inner = np.stack([vi + rng.normal(0, 1, vi.shape) for _ in range(40)])
    outer = np.stack([vo + rng.normal(0, 1, vo.shape) for _ in range(40)])
    want = m.getDataSlice(inner, outer)
    errors, results = [], [None, None]

    def run(k):
        try:
            for _ in range(5):
                results[k] = m.getDataSlice(inner, outer)
                _same(results[k], want, f"thread {k}")
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


def _create(lib, o2i, i2t, o2t, inner, outer, t=5, b=2):
    h = C.c_void_p()
    rc = lib.fb200_merge_create(o2i, i2t, o2t, inner[1], inner[0], outer[1], outer[0], t, b, 1, C.byref(h))
    return rc, h


def test_errors(fx):
    lib = fb.load()
    m, vi, vo = _reference_files(fx)
    o2i, i2t, o2t = (x.cachedInterpolation._h for x in (m._outer_to_inner, m._inner_to_target, m._outer_to_target))
    ishape, oshape = vi.shape, vo.shape

    def refused(rc, words):
        assert rc == MIFI_ERROR
        msg = fb.last_error()
        assert words in msg, msg

    rc, h = _create(lib, o2i, i2t, o2t, ishape, oshape)
    assert rc == MIFI_OK
    lib.fb200_merge_destroy(h)
    # grids that do not chain
    refused(_create(lib, o2i, i2t, o2t, (ishape[0], ishape[1] + 1), oshape)[0], "inner grid is")
    refused(_create(lib, o2i, i2t, o2t, ishape, (oshape[0] + 1, oshape[1]))[0], "outer grid is")
    refused(_create(lib, i2t, o2i, o2t, ishape, oshape)[0], "grid")
    refused(_create(lib, o2i, o2t, i2t, ishape, oshape)[0], "grid")
    other = fb.Interpolator(str(fx["merge_inner_proj4"]), m.x_inner, m.y_inner, True)
    other.changeProjection(Method.BILINEAR, str(fx["merge_inner_proj4"]), m.target_x[:-1], m.target_y, "degree", "degree")
    refused(_create(lib, o2i, other.cachedInterpolation._h, o2t, ishape, oshape)[0], "target")
    # a forward-method handle
    fwd = fb.CachedForwardInterpolation("x", "y", Method.FORWARD_MEAN, np.zeros(ishape[0] * ishape[1]), np.zeros(ishape[0] * ishape[1]),
                                        ishape[1], ishape[0], 61, 113)
    refused(_create(lib, o2i, fwd._h, o2t, ishape, oshape)[0], "nearest neighbour, bilinear or bicubic")
    # bad widths
    refused(_create(lib, o2i, i2t, o2t, ishape, oshape, t=0)[0], "transition width")
    refused(_create(lib, o2i, i2t, o2t, ishape, oshape, b=-1)[0], "border width")
    with pytest.raises(FimexB200Error):
        m.setSmoothing("LINEAR(0,2)")
    # null pointers
    refused(_create(lib, None, i2t, o2t, ishape, oshape)[0], "null")
    refused(lib.fb200_merge_create(o2i, i2t, o2t, ishape[1], ishape[0], oshape[1], oshape[0], 5, 2, 1, None), "null")
    mh = m._merge_handle()._h
    a, o = np.ascontiguousarray(vi), np.ascontiguousarray(vo)
    out = np.empty(61 * 113)
    n = C.c_size_t()
    D = int(fb.DataType.DOUBLE)
    ptr = fb.capi.ptr
    nan = float("nan")
    refused(lib.fb200_merge_get_data_slice(None, D, ptr(a), a.size, nan, ptr(o), o.size, nan, D, nan, ptr(out), C.byref(n)), "null merge handle")
    refused(lib.fb200_merge_get_data_slice(mh, D, None, a.size, nan, ptr(o), o.size, nan, D, nan, ptr(out), C.byref(n)), "null data pointer")
    refused(lib.fb200_merge_get_data_slice(mh, D, ptr(a), a.size, nan, ptr(o), o.size, nan, D, nan, None, C.byref(n)), "null data pointer")
    # wrong sizes
    refused(lib.fb200_merge_get_data_slice(mh, D, ptr(a), a.size - 1, nan, ptr(o), o.size, nan, D, nan, ptr(out), C.byref(n)), "whole number")
    refused(lib.fb200_merge_get_data_slice(mh, D, ptr(a), a.size, nan, ptr(o), o.size + 1, nan, D, nan, ptr(out), C.byref(n)), "whole number")
    two = np.concatenate([o, o])
    refused(lib.fb200_merge_get_data_slice(mh, D, ptr(a), a.size, nan, ptr(two), two.size, nan, D, nan, ptr(out), C.byref(n)), "levels")
    refused(lib.fb200_merge_get_data_slice(mh, 99, ptr(a), a.size, nan, ptr(o), o.size, nan, D, nan, ptr(out), C.byref(n)), "data type")
    with pytest.raises(FimexB200Error):
        m.getDataSlice(vi[:-1], vo)
    with pytest.raises(FimexB200Error):
        m.getDataSlice(np.stack([vi, vi]), vo)
    # nothing to do: zero levels
    assert lib.fb200_merge_get_data_slice(mh, D, None, 0, nan, None, 0, nan, D, nan, None, C.byref(n)) == MIFI_OK and n.value == 0
