"""Vertical interpolation to pressure levels on the GPU against the oracle (orc_vinterp_pressure, tests/vertical_oracle.c), bit for bit: every method x
source coordinate x extrapolation mode x column direction at odd sizes, the host and device entry points, typed slices, concurrent
calls on one handle, a whole ERA5-size step, and the device-resident chain horizontal getDataSlice -> vertical getDataSlice."""
import threading
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal
import vertical_oracle as vo

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, VerticalInterpolator  # noqa: E402

METHODS = {"linear": 0, "log": 1, "loglog": 2, "nearestneighbor": 3}
ERA5_LEVELS = np.array([1, 2, 3, 5, 7, 10, 20, 30, 50, 70, 100, 125, 150, 175, 200, 225, 250, 300, 350, 400, 450, 500, 550, 600, 650, 700,
                        750, 775, 800, 825, 850, 875, 900, 925, 950, 975, 1000], dtype=np.float64)


def hybrid_table(nk, rng):
    """a seeded, monotone, synthetic hybrid table (hPa) shaped like ECMWF's: near-geometric spacing aloft, dense near the ground,
    b = 0 above eta = 0.2; p_k(ps) stays monotone for ps in [400, 1100] hPa"""
    u = np.cumsum(rng.uniform(0.6, 1.4, nk))
    u = (u - u[0]) / (u[-1] - u[0])
    eta = np.exp(np.log(2e-5) * (1 - u) ** 1.6)
    b = np.clip((eta - 0.2) / 0.8, 0, None)
    ap = 1013.25 * (eta - b)
    return ap, b


def _setup(kind, nk, direction, rng):
    ap, b = hybrid_table(nk, rng)
    if kind == "pressure":
        p = ap + b * 1013.25
        terms, okind, oap, ob, ptop = {"p": p}, 0, p, None, 0.0
    elif kind == "hybrid":
        terms, okind, oap, ob, ptop = {"ap": ap, "b": b}, 1, ap, b, 0.0
    else:
        sigma = np.linspace(0.0, 1.0, nk) ** 1.3
        ptop = 5.0
        terms, okind, oap, ob, ptop = {"sigma": sigma, "ptop": ptop}, 2, None, sigma, ptop
    if direction == "down":  # surface first: pressure decreasing with k
        terms = {k: (v[::-1].copy() if isinstance(v, np.ndarray) else v) for k, v in terms.items()}
        oap = None if oap is None else oap[::-1].copy()
        ob = None if ob is None else ob[::-1].copy()
    name = {"pressure": PRESSURE, "hybrid": HYBRID, "sigma": SIGMA}[kind]
    return name, terms, okind, oap, ob, ptop


def _fields(nt, nk, nxy, rng, nan_share=0.01):
    field = rng.normal(250, 30, (nt, nk, nxy)).astype(np.float32)
    field[rng.random(field.shape) < nan_share] = np.nan
    ps = rng.uniform(480, 1040, (nt, nxy)).astype(np.float32)
    return field, ps


@pytest.mark.parametrize("size", [(3, 17, 517, 9), (1, 2, 33, 1)], ids=["nt3_k17_nxy517_p9", "nt1_k2_nxy33_p1"])
@pytest.mark.parametrize("direction", ["up", "down"])
@pytest.mark.parametrize("extrapolate", [True, False])
@pytest.mark.parametrize("kind", ["pressure", "hybrid", "sigma"])
@pytest.mark.parametrize("method", list(METHODS))
def test_bit_identical_to_oracle(oracle, method, kind, extrapolate, direction, size):
    import torch
    nt, nk, nxy, np_ = size
    rng = np.random.default_rng(zlib.crc32(repr((method, kind, extrapolate, direction, size)).encode()))
    name, terms, okind, oap, ob, ptop = _setup(kind, nk, direction, rng)
    levels = rng.uniform(0.5, 1100, np_)
    if np_ > 2:
        levels[:2] = [850.0, 500.0]
    field, ps = _fields(nt, nk, nxy, rng)
    want = vo.vinterp(METHODS[method], okind, oap, ob, levels, field, ps=ps, ptop=ptop, extrapolate=extrapolate)
    vi = VerticalInterpolator(name, terms, method, levels, extrapolate=extrapolate)
    host = vi.interpolateValues(field, ps)
    dev = vi.interpolateValues(torch.from_numpy(field).cuda(), torch.from_numpy(ps).cuda()).cpu().numpy()
    what = f"{method} {kind} extrapolate={extrapolate} {direction} {size}"
    nn = method == "nearestneighbor"
    assert_bit_equal(host, want, what + " host", nan_payload=nn)
    assert_bit_equal(dev, want, what + " device", nan_payload=nn)
    np.testing.assert_array_equal(host.view(np.uint32), dev.view(np.uint32))


def test_pressure_levels_ignore_ps(oracle):
    import torch
    rng = np.random.default_rng(5)
    p = np.array([1000.0, 850.0, 700.0, 500.0, 300.0, 100.0])
    field, _ = _fields(2, p.size, 301, rng)
    vi = VerticalInterpolator(PRESSURE, {"p": p}, "log", ERA5_LEVELS)
    want = vo.vinterp(1, 0, p, None, ERA5_LEVELS, field)
    assert_bit_equal(vi.interpolateValues(field), want, "no ps")
    assert_bit_equal(vi.interpolateValues(torch.from_numpy(field).cuda()).cpu().numpy(), want, "no ps, device")


def test_a_p0_form_and_ps_scale(oracle):
    rng = np.random.default_rng(8)
    ap, b = hybrid_table(40, rng)
    a, p0 = ap / 1000.0, 1000.0
    field, ps = _fields(2, 40, 999, rng)
    ps_pa = (ps.astype(np.float64) * 100).astype(np.float32)
    vi = VerticalInterpolator(HYBRID, {"a": a, "p0": p0, "b": b}, "loglog", ERA5_LEVELS, ps_scale=0.01)
    want = vo.vinterp(2, 1, a * p0, b, ERA5_LEVELS, field, ps=ps_pa, ps_scale=0.01)
    assert_bit_equal(vi.interpolateValues(field, ps_pa), want, "a, p0 and Pa")


@pytest.mark.parametrize("method", ["log", "nearestneighbor"])
def test_typed_slices_int16(oracle, method):
    import torch
    rng = np.random.default_rng(13)
    ap, b = hybrid_table(60, rng)
    field, ps = _fields(2, 60, 1201, rng, nan_share=0.02)
    packed = np.clip(np.round((np.nan_to_num(field, nan=250.0) - 250.0) * 100), -32000, 32000).astype(np.int16)
    packed[np.isnan(field)] = -32767
    vi = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, method, ERA5_LEVELS)
    # int16 in and out: the variable's fill value -> NaN on the way in, NaN -> fill on the way out
    want = oracle.from_float(vo.vinterp(METHODS[method], 1, ap, b, ERA5_LEVELS, oracle.as_float(packed, -32767.0), ps=ps), -32767.0, np.int16)
    host = vi.getDataSlice(packed, ps, bad_value=-32767.0)
    assert host.dtype == np.int16 and host.shape == (2, ERA5_LEVELS.size, 1201) and np.array_equal(host.ravel(), want.ravel())
    dev = vi.getDataSlice(torch.from_numpy(packed).cuda(), torch.from_numpy(ps).cuda(), bad_value=-32767.0).cpu().numpy()
    assert np.array_equal(dev.ravel(), want.ravel())
    # float in, int16 out
    want_f = oracle.from_float(vo.vinterp(METHODS[method], 1, ap, b, ERA5_LEVELS, field, ps=ps), -32000.0, np.int16)
    got_f = vi.getDataSlice(field, ps, bad_value=-32000.0, out_dtype=np.int16)
    assert got_f.dtype == np.int16 and np.array_equal(got_f.ravel(), want_f.ravel())


def test_concurrent_calls_on_one_handle(oracle):
    rng = np.random.default_rng(21)
    ap, b = hybrid_table(50, rng)
    vi = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, "log", ERA5_LEVELS)
    cases = [_fields(3, 50, 2053 + 7 * i, np.random.default_rng(100 + i)) for i in range(6)]
    results = [None] * len(cases)

    def work(i):
        for _ in range(3):
            results[i] = vi.interpolateValues(*cases[i])

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for i, (field, ps) in enumerate(cases):
        assert_bit_equal(results[i], vo.vinterp(1, 1, ap, b, ERA5_LEVELS, field, ps=ps), f"thread {i}")


@pytest.mark.parametrize("method", ["log", "linear"])
def test_era5_step_memcmp_equal(oracle, method):
    """one whole ERA5-size time step: 1440 x 721 columns, 137 levels -> the 37 ERA5 pressure levels"""
    rng = np.random.default_rng(137)
    ap, b = hybrid_table(137, rng)
    nxy = 1440 * 721
    field = rng.normal(250, 30, (1, 137, nxy)).astype(np.float32)
    ps = rng.uniform(500, 1040, (1, nxy)).astype(np.float32)
    vi = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, method, ERA5_LEVELS)
    got = vi.interpolateValues(field.reshape(1, 137, 721, 1440), ps.reshape(1, 721, 1440))
    want = vo.vinterp(METHODS[method], 1, ap, b, ERA5_LEVELS, field, ps=ps)
    assert got.shape == (1, 37, 721, 1440)
    assert got.tobytes() == want.tobytes()


def test_chain_horizontal_then_vertical_on_the_device(oracle):
    """field and ps of the horizontally interpolated CDM: horizontal get_data_slice_device, then vertical on the device"""
    import torch
    rng = np.random.default_rng(34)
    inX, inY, outX, outY, nt, nk = 97, 61, 83, 45, 2, 30
    px = rng.uniform(-0.5, inX - 0.5, outX * outY)
    py = rng.uniform(-0.5, inY - 0.5, outX * outY)
    ci = fb.CachedInterpolation("x", "y", fb.Method.BILINEAR, px, py, inX, inY, outX, outY)
    ap, b = hybrid_table(nk, rng)
    field, ps = _fields(nt, nk, inX * inY, rng)
    nan = float("nan")
    h_field = ci.getDataSlice(torch.from_numpy(field.reshape(nt * nk, inY, inX)).cuda(), nan)
    h_ps = ci.getDataSlice(torch.from_numpy(ps.reshape(nt, inY, inX)).cuda(), nan)
    vi = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, "log", ERA5_LEVELS)
    got = vi.getDataSlice(h_field.reshape(nt, nk, outY, outX), h_ps.reshape(nt, outY, outX), bad_value=nan).cpu().numpy()
    o_field = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, field.reshape(nt * nk, inY, inX))
    o_ps = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, ps.reshape(nt, inY, inX))
    want = vo.vinterp(1, 1, ap, b, ERA5_LEVELS, o_field.reshape(nt, nk, -1), ps=o_ps.reshape(nt, -1))
    assert_bit_equal(got.reshape(want.shape), want, "chain")
