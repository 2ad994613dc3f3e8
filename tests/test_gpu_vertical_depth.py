"""Vertical interpolation to depth levels on the GPU against the oracle (orc_vinterp_depth, tests/vertical_depth_oracle.c), bit for bit,
NaN masks included: every source coordinate x method x extrapolation mode x column direction, with and without eta, on the host and
device entry points; land and NaN eta; typed slices; concurrent calls on one handle; a whole step of the timing workload; the
device-resident chain horizontal getDataSlice -> depth getDataSlice; ocean handles refused on the calls that cannot pass the sea-floor
depth, and depth-level handles on them."""
import threading
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal
import vertical_depth_oracle as vo

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import capi  # noqa: E402
from fimex_b200.vertical import DEPTH, OCEAN_S_G1, OCEAN_S_G2, OCEAN_SIGMA, DepthInterpolator  # noqa: E402

METHODS = {"linear": 0, "nearestneighbor": 3}
VCOORDS = {DEPTH: vo.DEPTH, OCEAN_SIGMA: vo.OCEAN_SIGMA, OCEAN_S_G1: vo.OCEAN_S_G1, OCEAN_S_G2: vo.OCEAN_S_G2}


def _source(name, nk, down, rng):
    """(terms, s, C, depth_c) with the sea floor at k = 0 (ROMS's order), or the surface at k = 0 when `down`"""
    if name == DEPTH:
        s = np.concatenate([[0.0], np.cumsum(rng.uniform(0.5, 1.5, nk - 1))])
        s = s / s[-1] * rng.uniform(2000, 3500)
        s, Cs, dc = s[::-1].copy(), None, 0.0  # deepest first, as the others
    elif name == OCEAN_SIGMA:
        s = np.linspace(-1, 0, nk + 1)[:-1] + 0.5 / nk
        Cs, dc = None, 0.0
    else:
        s, Cs = vo.roms_stretching(nk, theta_s=rng.uniform(3, 8), theta_b=rng.uniform(0.1, 3))
        dc = float(rng.uniform(5, 300))
    if down:
        s = s[::-1].copy()
        Cs = None if Cs is None else Cs[::-1].copy()
    if name == DEPTH:
        terms = {"depth": s}
    elif name == OCEAN_SIGMA:
        terms = {"sigma": s, "eta": None, "depth": None}
    else:
        terms = {"s": s, "C": Cs, "depth_c": dc, "eta": None, "depth": None}
    return terms, s, Cs, dc


def _inputs(nt, nk, nxy, rng, land=0.3, nan_share=0.01, eta_nan=0.02):
    """field [nt][nk][nxy], eta [nt][nxy] [m], h [nxy] [m]: seeded; land as h = 0, NaN or < 0; a few NaN eta over sea"""
    field = rng.normal(10, 5, (nt, nk, nxy)).astype(np.float32)
    field[rng.random(field.shape) < nan_share] = np.nan
    h = rng.uniform(5, 3000, nxy)
    is_land = rng.random(nxy) < land
    h[is_land] = rng.choice([0.0, np.nan, -3.0], int(is_land.sum()))
    eta = rng.uniform(-1.5, 1.5, (nt, nxy))
    eta[rng.random(eta.shape) < eta_nan] = np.nan
    return field, eta.astype(np.float32), h.astype(np.float32)


def _levels(np_, rng):
    if np_ >= vo.DEPTHS16.size:
        return np.concatenate([vo.DEPTHS16, rng.uniform(-5, 3600, np_ - vo.DEPTHS16.size)])
    return rng.uniform(1, 400, np_)


def _oracle(method, name, s, Cs, dc, levels, field, eta, h, extrapolate=True):
    ocean = name != DEPTH
    return vo.vinterp_depth(METHODS[method], VCOORDS[name], s, Cs, levels, field, eta=eta if ocean else None, depth=h if ocean else None,
                            depth_c=dc, extrapolate=extrapolate)


def _cuda(*arrays):
    import torch
    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


@pytest.mark.parametrize("size", [(3, 35, 517, 19), (1, 2, 33, 1)], ids=["nt3_k35_nxy517_p19", "nt1_k2_nxy33_p1"])
@pytest.mark.parametrize("eta_given", [True, False], ids=["eta", "no_eta"])
@pytest.mark.parametrize("direction", ["up", "down"])
@pytest.mark.parametrize("extrapolate", [True, False])
@pytest.mark.parametrize("method", list(METHODS))
@pytest.mark.parametrize("name", list(VCOORDS))
def test_bit_identical_to_oracle(oracle, name, method, extrapolate, direction, eta_given, size):
    nt, nk, nxy, np_ = size
    rng = np.random.default_rng(zlib.crc32(repr((name, method, extrapolate, direction, eta_given, size)).encode()))
    terms, s, Cs, dc = _source(name, nk, direction == "down", rng)
    levels = _levels(np_, rng)
    field, eta, h = _inputs(nt, nk, nxy, rng)
    if np_ == 1:  # one target half way down the median sea column: inside many columns even of two levels without extrapolation
        x = -vo.column_z(VCOORDS[name], s, Cs, dc, float(np.median(h[h > 0])), 0.0)
        levels = np.array([0.5 * (x[0] + x[-1])])
    if not eta_given:
        eta = None
    want = _oracle(method, name, s, Cs, dc, levels, field, eta, h, extrapolate)
    di = DepthInterpolator(name, terms, method, levels, extrapolate=extrapolate)
    host = di.interpolateValues(field, eta=eta, depth=h)
    d_field, d_eta, d_h = _cuda(field, eta, h)
    dev = di.interpolateValues(d_field, eta=d_eta, depth=d_h).cpu().numpy()
    what = f"{name} {method} extrapolate={extrapolate} {direction} eta={eta_given} {size}"
    nn = method == "nearestneighbor"
    assert_bit_equal(host, want, what + " host", nan_payload=nn)
    assert_bit_equal(dev, want, what + " device", nan_payload=nn)
    assert np.isfinite(want).mean() > 0.1, what  # the case exercises values, not only NaN


@pytest.mark.parametrize("name", [OCEAN_SIGMA, OCEAN_S_G1, OCEAN_S_G2])
def test_land_and_nan_eta(oracle, name):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    nt, nk, nxy = 2, 30, 1003
    terms, s, Cs, dc = _source(name, nk, False, rng)
    field, eta, h = _inputs(nt, nk, nxy, rng, land=0.4, nan_share=0.0, eta_nan=0.1)
    di = DepthInterpolator(name, terms, "linear", vo.DEPTHS16)
    want = _oracle("linear", name, s, Cs, dc, vo.DEPTHS16, field, eta, h)
    got = di.interpolateValues(*_cuda(field), **dict(zip(["eta", "depth"], _cuda(eta, h)))).cpu().numpy()
    assert_bit_equal(got, want, f"land {name}")
    dead = ~(h > 0)[None, :] | np.isnan(eta)  # [nt][nxy]
    assert np.isnan(want.transpose(0, 2, 1)[dead]).all() and np.isfinite(want.transpose(0, 2, 1)[~dead]).mean() > 0.9


@pytest.mark.parametrize("method", list(METHODS))
def test_typed_slices_int16(oracle, method):
    rng = np.random.default_rng(13)
    terms, s, Cs, dc = _source(OCEAN_S_G2, 35, True, rng)
    field, eta, h = _inputs(2, 35, 1201, rng, nan_share=0.02)
    packed = np.clip(np.round((np.nan_to_num(field, nan=10.0) - 10.0) * 1000), -32000, 32000).astype(np.int16)
    packed[np.isnan(field)] = -32767
    di = DepthInterpolator(OCEAN_S_G2, terms, method, vo.DEPTHS16)
    want = oracle.from_float(_oracle(method, OCEAN_S_G2, s, Cs, dc, vo.DEPTHS16, oracle.as_float(packed, -32767.0), eta, h), -32767.0, np.int16)
    host = di.getDataSlice(packed, eta=eta, depth=h, bad_value=-32767.0)
    assert host.dtype == np.int16 and host.shape == (2, vo.DEPTHS16.size, 1201) and np.array_equal(host.ravel(), want.ravel())
    dev = di.getDataSlice(*_cuda(packed), **dict(zip(["eta", "depth"], _cuda(eta, h))), bad_value=-32767.0).cpu().numpy()
    assert np.array_equal(dev.ravel(), want.ravel())


def test_concurrent_calls_on_one_handle(oracle):
    rng = np.random.default_rng(21)
    terms, s, Cs, dc = _source(OCEAN_S_G1, 40, False, rng)
    di = DepthInterpolator(OCEAN_S_G1, terms, "linear", vo.DEPTHS16)
    cases = [_inputs(3, 40, 2053 + 7 * i, np.random.default_rng(100 + i)) for i in range(6)]
    results = [None] * len(cases)

    def work(i):
        field, eta, h = cases[i]
        for _ in range(3):
            results[i] = di.interpolateValues(field, eta=eta, depth=h)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for i, (field, eta, h) in enumerate(cases):
        assert_bit_equal(results[i], _oracle("linear", OCEAN_S_G1, s, Cs, dc, vo.DEPTHS16, field, eta, h), f"thread {i}")


def test_timing_workload_step_memcmp_equal(oracle):
    """one whole step of profiles/tools/vertical_depth_time.py's workload: 2600 x 900 columns, 30 % land, 35 g2 levels -> 16 depths,
    host buffers"""
    rng = np.random.default_rng(20261020)
    s, Cs = vo.roms_stretching(35)
    h, eta = vo.synthetic_ocean(2600, 900, rng)
    field = np.random.default_rng(5).normal(10, 5, (1, 35, h.size)).astype(np.float32)
    terms = {"s": s, "C": Cs, "depth_c": 250.0}
    di = DepthInterpolator(OCEAN_S_G2, terms, "linear", vo.DEPTHS16)
    got = di.interpolateValues(field.reshape(1, 35, 900, 2600), eta=eta[None], depth=h)
    want = vo.vinterp_depth(0, vo.OCEAN_S_G2, s, Cs, vo.DEPTHS16, field, eta=eta[None], depth=h, depth_c=250.0)
    assert got.shape == (1, vo.DEPTHS16.size, 900, 2600)
    assert got.tobytes() == want.tobytes()
    assert 0.25 < np.isnan(want).mean() < 0.4


def test_chain_horizontal_then_depth_on_the_device(oracle):
    """field, eta and the sea-floor depth through the horizontal get_data_slice_device, then the depth call on the device"""
    import torch
    rng = np.random.default_rng(34)
    inX, inY, outX, outY, nt, nk = 97, 61, 83, 45, 2, 30
    px = rng.uniform(-0.5, inX - 0.5, outX * outY)
    py = rng.uniform(-0.5, inY - 0.5, outX * outY)
    ci = fb.CachedInterpolation("x", "y", fb.Method.BILINEAR, px, py, inX, inY, outX, outY)
    terms, s, Cs, dc = _source(OCEAN_S_G2, nk, False, rng)
    field, eta, h = _inputs(nt, nk, inX * inY, rng)
    nan = float("nan")
    h_field = ci.getDataSlice(torch.from_numpy(field.reshape(nt * nk, inY, inX)).cuda(), nan)
    h_eta = ci.getDataSlice(torch.from_numpy(eta.reshape(nt, inY, inX)).cuda(), nan)
    h_h = ci.getDataSlice(torch.from_numpy(h.reshape(1, inY, inX)).cuda(), nan)
    di = DepthInterpolator(OCEAN_S_G2, terms, "linear", vo.DEPTHS16)
    got = di.getDataSlice(h_field.reshape(nt, nk, outY, outX), eta=h_eta, depth=h_h, bad_value=nan).cpu().numpy()
    o = {k: oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, v.reshape(-1, inY, inX)) for k, v in (("f", field), ("eta", eta), ("h", h))}
    want = vo.vinterp_depth(0, vo.OCEAN_S_G2, s, Cs, vo.DEPTHS16, o["f"].reshape(nt, nk, -1), eta=o["eta"].reshape(nt, -1), depth=o["h"].reshape(-1),
                            depth_c=dc)
    assert_bit_equal(got.reshape(want.shape), want, "chain")
    assert np.isfinite(want).mean() > 0.2


def test_ocean_handles_on_the_calls_without_columns(oracle):
    lib = fb.load()
    rng = np.random.default_rng(55)
    field, eta, h = _inputs(2, 20, 300, rng)
    out = np.empty((2, vo.DEPTHS16.size, 300), np.float32)
    for name in (OCEAN_SIGMA, OCEAN_S_G1, OCEAN_S_G2):
        terms, s, Cs, dc = _source(name, 20, False, rng)
        di = DepthInterpolator(name, terms, "linear", vo.DEPTHS16)
        assert lib.fb200_vinterp_interpolate_values(di._h, capi.ptr(field), capi.ptr(eta), 300, 2, capi.ptr(out)) == fb.MIFI_ERROR
        assert "sea-floor depth" in fb.last_error()
        assert lib.fb200_vinterp_get_data_slice(di._h, int(fb.DataType.FLOAT), capi.ptr(field), capi.ptr(eta), 300, 2, float("nan"),
                                                int(fb.DataType.FLOAT), capi.ptr(out)) == fb.MIFI_ERROR
        assert "sea-floor depth" in fb.last_error()
        with pytest.raises(fb.FimexB200Error, match="sea-floor depth"):
            di.interpolateValues(field, eta=eta)
    # depth levels need neither: the calls without _columns compute what the Python layer does, eta or not
    terms, s, Cs, dc = _source(DEPTH, 20, True, rng)
    dd = DepthInterpolator(DEPTH, terms, "nearestneighbor", vo.DEPTHS16, extrapolate=False)
    want = _oracle("nearestneighbor", DEPTH, s, Cs, dc, vo.DEPTHS16, field, None, None, extrapolate=False)
    for ps in (None, eta):
        assert lib.fb200_vinterp_interpolate_values(dd._h, capi.ptr(field), capi.ptr(ps), 300, 2, capi.ptr(out)) == fb.MIFI_OK
        assert_bit_equal(out, want, "depth levels on the call without _columns", nan_payload=True)
    import torch
    d_out = torch.empty(out.shape, device="cuda")
    d_field, = _cuda(field)
    assert lib.fb200_vinterp_interpolate_values_device(dd._h, capi.ptr(d_field), None, 300, 2, capi.ptr(d_out), None) == fb.MIFI_OK
    torch.cuda.synchronize()
    assert_bit_equal(d_out.cpu().numpy(), want, "depth levels on the device call without _columns", nan_payload=True)
    assert_bit_equal(dd.interpolateValues(field), want, "depth levels through the Python layer", nan_payload=True)
