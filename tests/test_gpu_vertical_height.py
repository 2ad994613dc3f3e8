"""Vertical interpolation to height and altitude levels on the GPU against the oracle (orc_vinterp_height, tests/vertical_height_oracle.c), bit for
bit: every converter x target x method x extrapolation mode x column direction x source coordinate at odd sizes, the host and device
entry points, NaN in t, ps and zs, typed slices, concurrent calls on one handle, a whole ERA5-size step, the device-resident chain
horizontal getDataSlice -> height getDataSlice, and height handles on the calls that pass ps alone."""
import ctypes as C
import threading
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal
import vertical_height_oracle as vo

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import capi  # noqa: E402
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, HeightInterpolator  # noqa: E402

G0 = 9.80665
METHODS = {"linear": 0, "nearestneighbor": 3}
CONVERTERS = {"standard": 0, "hypsometric": 1, "field": 2}
TARGETS = {"altitude": 0, "height": 1}
KINDS = {"pressure": 0, "hybrid": 1, "sigma": 2}
HEIGHTS = np.array([10, 20, 50, 100, 150, 200, 250, 300, 500, 750, 1000, 1500, 2000, 3000, 5000], dtype=np.float64)


def hybrid_table(nk, rng):
    """the seeded L137-like table of test_gpu_vertical.py (hPa)"""
    u = np.cumsum(rng.uniform(0.6, 1.4, nk))
    u = (u - u[0]) / (u[-1] - u[0])
    eta = np.exp(np.log(2e-5) * (1 - u) ** 1.6)
    b = np.clip((eta - 0.2) / 0.8, 0, None)
    return 1013.25 * (eta - b), b


def _source(kind, nk, down, rng):
    """(standard_name, terms, oracle kind, ap, b, ptop, p(ps)) with the surface at k = nk - 1, or at k = 0 when `down`"""
    ap, b = hybrid_table(nk, rng)
    ptop = 0.0
    if kind == "pressure":
        oap, ob = ap + b * 1013.25, None
        terms = {"p": oap}
    elif kind == "hybrid":
        oap, ob = ap, b
        terms = {"ap": ap, "b": b}
    else:
        ptop = 5.0
        oap, ob = None, np.linspace(0.0, 1.0, nk) ** 1.3
        terms = {"sigma": ob, "ptop": ptop}
    if down:
        oap = None if oap is None else oap[::-1].copy()
        ob = None if ob is None else ob[::-1].copy()
        terms = {k: (v[::-1].copy() if isinstance(v, np.ndarray) else v) for k, v in terms.items()}
    name = {"pressure": PRESSURE, "hybrid": HYBRID, "sigma": SIGMA}[kind]

    def pres(ps):  # [nt][nxy] -> [nt][nk][nxy]
        psd = ps.astype(np.float64)[:, None, :]
        if kind == "pressure":
            return np.broadcast_to(oap[None, :, None], (ps.shape[0], nk, ps.shape[1]))
        if kind == "hybrid":
            return oap[None, :, None] + ob[None, :, None] * psd
        return ptop + ob[None, :, None] * (psd - ptop)
    return name, terms, KINDS[kind], oap, ob, ptop, pres


def _inputs(nt, nk, nxy, pres, rng, nan_share=0.01):
    """field, ps [hPa], t [K], q [kg/kg], z [geopotential, m2/s2], zs [surface geopotential]: seeded, plausible and monotone in k"""
    field = rng.normal(250, 30, (nt, nk, nxy)).astype(np.float32)
    field[rng.random(field.shape) < nan_share] = np.nan
    ps = rng.uniform(480, 1040, (nt, nxy)).astype(np.float32)
    p = pres(ps)
    zstd = 44330.8 * (1 - (p / 1013.25) ** 0.190263)  # the troposphere's formula, continued: a smooth monotone altitude
    t = np.maximum(288.15 - 6.5e-3 * zstd, 210.0) + rng.normal(0, 1.5, p.shape)
    q = rng.uniform(0, 0.02, p.shape) * np.exp(-np.maximum(zstd, 0) / 2500)
    z = (zstd * G0).astype(np.float32)
    zs = rng.uniform(-50, 2500, nxy).astype(np.float32) * np.float32(G0)
    return field, ps, t.astype(np.float32), q.astype(np.float32), z, zs


def _oracle(method, converter, target, okind, oap, ob, ptop, levels, field, ps, t, q, z, zs, extrapolate=True):
    hyps, fld = converter == "hypsometric", converter == "field"
    needs_zs = (target == "height") != hyps
    return vo.vinterp_height(METHODS[method], CONVERTERS[converter], TARGETS[target], okind, oap, ob, levels, field,
                             ps=ps if (hyps or (converter == "standard" and okind != 0)) else None, t=t if hyps else None, q=q if hyps else None,
                             z=z if fld else None, zs=zs if needs_zs else None, ptop=ptop, z_scale=1 / G0, zs_scale=1 / G0,
                             extrapolate=extrapolate)


def _levels(target, np_, rng):
    lev = rng.uniform(-200, 16000, np_) if target == "altitude" else rng.uniform(-50, 12000, np_)
    if np_ > 2:
        lev[:2] = [10.0, 100.0]
    return lev


def _cuda(*arrays):
    import torch
    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


@pytest.mark.parametrize("size", [(3, 17, 517, 9), (1, 2, 33, 1)], ids=["nt3_k17_nxy517_p9", "nt1_k2_nxy33_p1"])
@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("direction", ["up", "down"])
@pytest.mark.parametrize("extrapolate", [True, False])
@pytest.mark.parametrize("method", list(METHODS))
@pytest.mark.parametrize("target", list(TARGETS))
@pytest.mark.parametrize("converter", list(CONVERTERS))
def test_bit_identical_to_oracle(oracle, converter, target, method, extrapolate, direction, kind, size):
    if converter == "hypsometric" and kind == "pressure":
        pytest.skip("the hypsometric converter needs a surface pressure (refused, test_vertical_height_host.py)")
    nt, nk, nxy, np_ = size
    rng = np.random.default_rng(zlib.crc32(repr((converter, target, method, extrapolate, direction, kind, size)).encode()))
    name, terms, okind, oap, ob, ptop, pres = _source(kind, nk, direction == "down", rng)
    levels = _levels(target, np_, rng)
    field, ps, t, q, z, zs = _inputs(nt, nk, nxy, pres, rng)
    want = _oracle(method, converter, target, okind, oap, ob, ptop, levels, field, ps, t, q, z, zs, extrapolate)
    hi = HeightInterpolator(name, terms, method, levels, type=target, converter=converter, z_scale=1 / G0, zs_scale=1 / G0,
                            extrapolate=extrapolate)
    host = hi.interpolateValues(field, ps=ps, t=t, q=q, z=z, zs=zs)
    dev = hi.interpolateValues(*_cuda(field), **dict(zip(["ps", "t", "q", "z", "zs"], _cuda(ps, t, q, z, zs)))).cpu().numpy()
    what = f"{converter} {target} {method} extrapolate={extrapolate} {direction} {kind} {size}"
    nn = method == "nearestneighbor"
    assert_bit_equal(host, want, what + " host", nan_payload=nn)
    assert_bit_equal(dev, want, what + " device", nan_payload=nn)
    assert np.isfinite(want).mean() > 0.1, what  # the case exercises values, not only NaN


def test_hypsometric_without_q_and_in_pa(oracle):
    rng = np.random.default_rng(3)
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", 40, False, rng)
    field, ps, t, q, z, zs = _inputs(2, 40, 999, pres, rng)
    ps_pa = (ps.astype(np.float64) * 100).astype(np.float32)
    want = vo.vinterp_height(0, 1, 0, okind, oap, ob, HEIGHTS + 1000.0, field, ps=ps_pa, t=t, zs=zs, ps_scale=0.01, zs_scale=1 / G0)
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS + 1000.0, type="altitude", converter="hypsometric", ps_scale=0.01, zs_scale=1 / G0)
    assert_bit_equal(hi.interpolateValues(field, ps=ps_pa, t=t, zs=zs), want, "no q, Pa")


@pytest.mark.parametrize("converter, target", [("hypsometric", "altitude"), ("hypsometric", "height"), ("standard", "height"),
                                               ("field", "height")])
def test_nan_in_t_ps_and_zs(oracle, converter, target):
    rng = np.random.default_rng(zlib.crc32(f"{converter}{target}".encode()))
    nt, nk, nxy = 2, 30, 1003
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", nk, False, rng)
    field, ps, t, q, z, zs = _inputs(nt, nk, nxy, pres, rng, nan_share=0.0)
    t[rng.random(t.shape) < 0.01] = np.nan
    q[rng.random(q.shape) < 0.01] = np.nan
    z[rng.random(z.shape) < 0.01] = np.nan
    ps[rng.random(ps.shape) < 0.05] = np.nan
    zs[rng.random(zs.shape) < 0.05] = np.nan
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS * 3, type=target, converter=converter, z_scale=1 / G0, zs_scale=1 / G0)
    want = _oracle("linear", converter, target, okind, oap, ob, ptop, HEIGHTS * 3, field, ps, t, q, z, zs)
    got = hi.interpolateValues(*_cuda(field), **dict(zip(["ps", "t", "q", "z", "zs"], _cuda(ps, t, q, z, zs)))).cpu().numpy()
    assert_bit_equal(got, want, f"NaN {converter} {target}")
    assert np.isnan(want).mean() > 0.05 and np.isfinite(want).mean() > 0.3


@pytest.mark.parametrize("method", list(METHODS))
def test_typed_slices_int16(oracle, method):
    rng = np.random.default_rng(13)
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", 60, True, rng)
    field, ps, t, q, z, zs = _inputs(2, 60, 1201, pres, rng, nan_share=0.02)
    packed = np.clip(np.round((np.nan_to_num(field, nan=250.0) - 250.0) * 100), -32000, 32000).astype(np.int16)
    packed[np.isnan(field)] = -32767
    hi = HeightInterpolator(name, terms, method, HEIGHTS, converter="hypsometric")
    want = oracle.from_float(_oracle(method, "hypsometric", "height", okind, oap, ob, ptop, HEIGHTS, oracle.as_float(packed, -32767.0), ps, t, q, z,
                                     zs), -32767.0, np.int16)
    host = hi.getDataSlice(packed, ps=ps, t=t, q=q, bad_value=-32767.0)
    assert host.dtype == np.int16 and host.shape == (2, HEIGHTS.size, 1201) and np.array_equal(host.ravel(), want.ravel())
    dev = hi.getDataSlice(*_cuda(packed), **dict(zip(["ps", "t", "q"], _cuda(ps, t, q))), bad_value=-32767.0).cpu().numpy()
    assert np.array_equal(dev.ravel(), want.ravel())


def test_concurrent_calls_on_one_handle(oracle):
    rng = np.random.default_rng(21)
    name, terms, okind, oap, ob, ptop, pres = _source("sigma", 50, False, rng)
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS, type="altitude", converter="hypsometric", zs_scale=1 / G0)
    cases = [_inputs(3, 50, 2053 + 7 * i, pres, np.random.default_rng(100 + i)) for i in range(6)]
    results = [None] * len(cases)

    def work(i):
        field, ps, t, q, z, zs = cases[i]
        for _ in range(3):
            results[i] = hi.interpolateValues(field, ps=ps, t=t, q=q, zs=zs)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for i, (field, ps, t, q, z, zs) in enumerate(cases):
        want = _oracle("linear", "hypsometric", "altitude", okind, oap, ob, ptop, HEIGHTS, field, ps, t, q, z, zs)
        assert_bit_equal(results[i], want, f"thread {i}")


def test_era5_step_memcmp_equal(oracle):
    """one whole ERA5-size time step: 1440 x 721 columns, 137 levels with t and q -> 15 heights, host buffers"""
    rng = np.random.default_rng(137)
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", 137, False, rng)
    nxy = 1440 * 721
    field, ps, t, q, z, zs = _inputs(1, 137, nxy, pres, rng, nan_share=0.0)
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS, converter="hypsometric")
    got = hi.interpolateValues(field.reshape(1, 137, 721, 1440), ps=ps, t=t, q=q)
    want = _oracle("linear", "hypsometric", "height", okind, oap, ob, ptop, HEIGHTS, field, ps, t, q, z, zs)
    assert got.shape == (1, HEIGHTS.size, 721, 1440)
    assert got.tobytes() == want.tobytes()


def test_chain_horizontal_then_height_on_the_device(oracle):
    """field, t and ps of the horizontally interpolated CDM: horizontal get_data_slice_device, then the height call on the device"""
    import torch
    rng = np.random.default_rng(34)
    inX, inY, outX, outY, nt, nk = 97, 61, 83, 45, 2, 30
    px = rng.uniform(-0.5, inX - 0.5, outX * outY)
    py = rng.uniform(-0.5, inY - 0.5, outX * outY)
    ci = fb.CachedInterpolation("x", "y", fb.Method.BILINEAR, px, py, inX, inY, outX, outY)
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", nk, False, rng)
    field, ps, t, q, z, zs = _inputs(nt, nk, inX * inY, pres, rng)
    nan = float("nan")
    h_field = ci.getDataSlice(torch.from_numpy(field.reshape(nt * nk, inY, inX)).cuda(), nan)
    h_t = ci.getDataSlice(torch.from_numpy(t.reshape(nt * nk, inY, inX)).cuda(), nan)
    h_ps = ci.getDataSlice(torch.from_numpy(ps.reshape(nt, inY, inX)).cuda(), nan)
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS, converter="hypsometric")
    got = hi.getDataSlice(h_field.reshape(nt, nk, outY, outX), ps=h_ps, t=h_t, bad_value=nan).cpu().numpy()
    o = {k: oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, v.reshape(-1, inY, inX)) for k, v in (("f", field), ("t", t), ("ps", ps))}
    want = vo.vinterp_height(0, 1, 1, okind, oap, ob, HEIGHTS, o["f"].reshape(nt, nk, -1), ps=o["ps"].reshape(nt, -1), t=o["t"].reshape(nt, nk, -1))
    assert_bit_equal(got.reshape(want.shape), want, "chain")


def test_height_handles_on_the_calls_that_pass_ps_alone(oracle):
    lib = fb.load()
    rng = np.random.default_rng(55)
    name, terms, okind, oap, ob, ptop, pres = _source("hybrid", 20, False, rng)
    field, ps, t, q, z, zs = _inputs(2, 20, 300, pres, rng)
    out = np.empty((2, HEIGHTS.size, 300), np.float32)
    # t is needed: MIFI_ERROR, and the message names it
    hi = HeightInterpolator(name, terms, "linear", HEIGHTS, converter="hypsometric")
    assert lib.fb200_vinterp_interpolate_values(hi._h, capi.ptr(field), capi.ptr(ps), 300, 2, capi.ptr(out)) == fb.MIFI_ERROR
    assert "air temperature t" in fb.last_error()
    assert lib.fb200_vinterp_get_data_slice(hi._h, int(fb.DataType.FLOAT), capi.ptr(field), capi.ptr(ps), 300, 2, float("nan"),
                                            int(fb.DataType.FLOAT), capi.ptr(out)) == fb.MIFI_ERROR
    # zs is needed
    hs = HeightInterpolator(name, terms, "linear", HEIGHTS, type="height", converter="standard")
    assert lib.fb200_vinterp_interpolate_values(hs._h, capi.ptr(field), capi.ptr(ps), 300, 2, capi.ptr(out)) == fb.MIFI_ERROR
    assert "surface altitude zs" in fb.last_error()
    # ps alone is enough for standard altitudes: the old call computes what the new one does
    ha = HeightInterpolator(name, terms, "nearestneighbor", HEIGHTS * 10, type="altitude", converter="standard")
    assert lib.fb200_vinterp_interpolate_values(ha._h, capi.ptr(field), capi.ptr(ps), 300, 2, capi.ptr(out)) == fb.MIFI_OK
    want = _oracle("nearestneighbor", "standard", "altitude", okind, oap, ob, ptop, HEIGHTS * 10, field, ps, t, q, z, zs)
    assert_bit_equal(out, want, "standard altitudes on the ps-only call", nan_payload=True)
    # the Python layer and the columns call refuse missing inputs too
    with pytest.raises(fb.FimexB200Error, match="air temperature t"):
        hi.interpolateValues(field, ps=ps)
    with pytest.raises(fb.FimexB200Error, match="surface altitude zs"):
        hs.interpolateValues(field, ps=ps)
    cols = type("Cols", (C.Structure,), {"_fields_": [(n, C.c_void_p) for n in ("ps", "t", "q", "z", "zs")]})()
    cols.ps = capi.ptr(ps).value
    assert lib.fb200_vinterp_interpolate_values_columns(hs._h, capi.ptr(field), C.byref(cols), 300, 2, capi.ptr(out)) == fb.MIFI_ERROR
    assert "surface altitude zs" in fb.last_error()
