"""A seeded differential fuzz of the three vertical branches on the GPU, and their edges.

Each fuzz case (tests/vertical_reference.py, draw_case: branch, converter or source coordinate, method, extrapolation, direction,
nk, np, nxy, nt, NaN shares, duplicate targets, targets on levels and beyond both ends, land, NaN eta / t / q / zs) is checked three
ways: the host path and the device path bit for bit against the C restatement, and both against the independent longdouble
reference within its derived bound.  ``FIMEX_B200_VFUZZ_SEEDS`` sets the number of seeds (default 60; more: a one-off soak run).

Edges, bit for bit against the restatement: nt = 70 000 (the launchers' loop over gridDim.y), nk = np = 1024 (and 1025 refused),
element offsets past 2^32 in one device call, the multi-chunk host pipeline with pinned and pageable arrays, every CDM type in and
out, and loglog at pressures <= 1 hPa (NaN or -+inf, not compared with the reference)."""
import ctypes as C
import gc
import os
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal
import vertical_depth_oracle as vdo
import vertical_height_oracle as vho
import vertical_oracle as vpo
import vertical_reference as vr

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import capi  # noqa: E402
from fimex_b200.vertical import HYBRID, OCEAN_S_G2, PRESSURE, DEPTH, DepthInterpolator, HeightInterpolator, VerticalInterpolator  # noqa: E402

SEEDS = int(os.environ.get("FIMEX_B200_VFUZZ_SEEDS", "60"))
G0 = vr.G0
_SUMMARY = {"cases": 0, "worst": 0.0, "share": 0.0}


def _cuda(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cuda_kw(kw):
    return {k: _cuda(v) for k, v in kw.items()}


@pytest.mark.parametrize("seed", range(SEEDS))
def test_fuzz(oracle, seed):
    case = vr.draw_case(10_000 + seed, budget=4_000_000)
    want = case.oracle(case.field)
    h = case.handle()
    host = h.interpolateValues(case.field, **case.kwargs)
    dev = h.interpolateValues(_cuda(case.field), **_cuda_kw(case.kwargs)).cpu().numpy()
    nn = case.method == "nearestneighbor"
    assert_bit_equal(host, want, case.what + " host", nan_payload=nn)
    assert_bit_equal(dev, want, case.what + " device", nan_payload=nn)
    ref = case.reference(case.field)
    for got, where in ((host, "host"), (dev, "device")):
        frac, share = vr.check(got, ref, f"{case.what} {where} vs the reference")
    _SUMMARY["cases"] += 1
    _SUMMARY["worst"] = max(_SUMMARY["worst"], frac)
    _SUMMARY["share"] = max(_SUMMARY["share"], share)


def test_fuzz_summary():
    """prints the largest error (as a fraction of its bound) and the largest ambiguous share of the fuzz cases that ran"""
    print(f"\nvertical fuzz: {_SUMMARY['cases']} cases, largest error {_SUMMARY['worst']:.3f} of the bound, "
          f"largest ambiguous share {_SUMMARY['share']:.4%}")


# ------------------------------------------------------------------------------------------------------------- fixed cases per branch
def _pressure(nt, nk, nxy, npt, rng, method="log"):
    ap, b = vr._hybrid_table(nk, rng)
    levels = rng.uniform(0.5, 1100, npt)
    field = rng.normal(250, 30, (nt, nk, nxy)).astype(np.float32)
    ps = rng.uniform(480, 1040, (nt, nxy)).astype(np.float32)
    h = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, method, levels)
    m = vr.METHOD_NAMES[method]
    return h, field, {"ps": ps}, lambda f, kw: vpo.vinterp(m, 1, ap, b, levels, f, ps=kw["ps"])


def _height(nt, nk, nxy, npt, rng, converter="hypsometric", target="altitude"):
    ap, b = vr._hybrid_table(nk, rng)
    levels = rng.uniform(-200, 16000, npt)
    field = rng.normal(250, 30, (nt, nk, nxy)).astype(np.float32)
    ps = rng.uniform(480, 1040, (nt, nxy)).astype(np.float32)
    p = ap[None, :, None] + b[None, :, None] * ps.astype(np.float64)[:, None, :]
    zstd = 44330.8 * (1 - (p / 1013.25) ** 0.190263)
    kw = {"zs": (rng.uniform(-50, 2500, nxy) * G0).astype(np.float32)}
    if converter == "hypsometric":
        kw.update(ps=ps, t=(np.maximum(288.15 - 6.5e-3 * zstd, 210.0) + rng.normal(0, 1.5, p.shape)).astype(np.float32),
                  q=(rng.uniform(0, 0.02, p.shape) * np.exp(-np.maximum(zstd, 0) / 2500)).astype(np.float32))
    else:
        kw["z"] = (zstd * G0).astype(np.float32)
    conv = {"standard": 0, "hypsometric": 1, "field": 2}[converter]
    tgt = {"altitude": 0, "height": 1}[target]
    if (tgt == 1) == (conv == 1):
        del kw["zs"]
    h = HeightInterpolator(HYBRID, {"ap": ap, "b": b}, "linear", levels, type=target, converter=converter, z_scale=1 / G0, zs_scale=1 / G0)
    return h, field, kw, lambda f, k: vho.vinterp_height(0, conv, tgt, 1, ap, b, levels, f, **k, z_scale=1 / G0, zs_scale=1 / G0)


def _depth(nt, nk, nxy, npt, rng):
    s, Cs = vdo.roms_stretching(nk)
    levels = rng.uniform(-5, 3600, npt)
    field = rng.normal(10, 5, (nt, nk, nxy)).astype(np.float32)
    hh = rng.uniform(5, 3000, nxy)
    hh[rng.random(nxy) < 0.2] = 0.0
    kw = {"eta": rng.uniform(-1.5, 1.5, (nt, nxy)).astype(np.float32), "depth": hh.astype(np.float32)}
    h = DepthInterpolator(OCEAN_S_G2, {"s": s, "C": Cs, "depth_c": 50.0}, "linear", levels)
    return h, field, kw, lambda f, k: vdo.vinterp_depth(0, vdo.OCEAN_S_G2, s, Cs, levels, f, eta=k["eta"], depth=k["depth"], depth_c=50.0)


BRANCHES = {"pressure": _pressure, "height": _height, "depth": _depth}


def _both_paths(h, field, kw, want, what, nan_payload=False):
    assert_bit_equal(h.interpolateValues(field, **kw), want, what + " host", nan_payload=nan_payload)
    assert_bit_equal(h.interpolateValues(_cuda(field), **_cuda_kw(kw)).cpu().numpy(), want, what + " device", nan_payload=nan_payload)


@pytest.mark.parametrize("branch", list(BRANCHES))
def test_70000_time_steps(oracle, branch):
    """nt = 70 000 > 65 535: the launchers loop over blockIdx.y in chunks of 65 535 steps"""
    h, field, kw, orc = BRANCHES[branch](70_000, 2, 3, 3, np.random.default_rng(7))
    want = orc(field, kw)
    assert np.isfinite(want[65_535:]).mean() > 0.3
    _both_paths(h, field, kw, want, f"{branch} nt=70000")


@pytest.mark.parametrize("branch", list(BRANCHES))
def test_1024_levels_and_targets(oracle, branch):
    """the table limit: nk = np = 1024 (40 KB of dynamic shared memory for the pressure kernel); 1025 is refused"""
    rng = np.random.default_rng(11)
    h, field, kw, orc = BRANCHES[branch](2, 1024, 37, 1024, rng)
    _both_paths(h, field, kw, orc(field, kw), f"{branch} nk=np=1024")
    lib = fb.load()
    handle = C.c_void_p()
    lev = np.linspace(1.0, 1000.0, 1025)
    for nk, npt in ((1025, 4), (4, 1025)):
        a, b = np.linspace(0.0, 1.0, nk), np.linspace(1.0, 0.0, nk)
        if branch == "pressure":
            rc = lib.fb200_vinterp_create_hybrid(0, capi.ptr(a), capi.ptr(b), nk, 1.0, capi.ptr(lev), npt, 1, C.byref(handle))
            with pytest.raises(fb.FimexB200Error, match="1024"):
                VerticalInterpolator(HYBRID, {"ap": a, "b": b}, "linear", lev[:npt])
        elif branch == "height":
            rc = lib.fb200_vinterp_create_height(0, 1, 0, 1, capi.ptr(a), capi.ptr(b), nk, 0.0, 1.0, 1.0, 1.0, capi.ptr(lev), npt, 1,
                                                 C.byref(handle))
            with pytest.raises(fb.FimexB200Error, match="1024"):
                HeightInterpolator(HYBRID, {"ap": a, "b": b}, "linear", lev[:npt])
        else:
            rc = lib.fb200_vinterp_create_depth(0, 3, capi.ptr(lev[:nk]), None, nk, 0.0, capi.ptr(lev), npt, 1, C.byref(handle))
            with pytest.raises(fb.FimexB200Error, match="1024"):
                DepthInterpolator(DEPTH, {"depth": lev[:nk]}, "linear", lev[:npt])
        assert rc == fb.MIFI_ERROR and not handle.value and "1024" in fb.last_error()


# ---------------------------------------------------------------------------------------------------- offsets past 2^32 elements
def _device_normal(shape, seed, mean, std):
    """float32 on the device, normal(mean, std) from a seeded torch.Generator"""
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.empty(shape, dtype=torch.float32, device="cuda").normal_(mean, std, generator=g)


@pytest.mark.parametrize("branch", list(BRANCHES))
def test_offsets_past_2_32(oracle, branch):
    """one device call whose last time step starts beyond 2^32 elements (about 18 GB of float32 input); the first and the last
    steps are compared with the restatement run on those steps alone"""
    import torch
    rng = np.random.default_rng(32)
    if branch == "depth":
        nt, nk, nxy = 54, 35, 2600 * 900
    else:
        nt, nk, nxy = 32, 137, 1440 * 721
    assert (nt - 1) * nk * nxy > 2 ** 32
    field = _device_normal((nt, nk, nxy), 2026 + len(branch), 250.0, 30.0)
    npt = 4
    if branch == "pressure":
        ap, b = vr._hybrid_table(nk, rng)
        levels = np.array([1000.0, 850.0, 500.0, 3.0])
        h = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, "log", levels)
        ps = _device_normal((nt, nxy), 5, 760.0, 120.0).clamp_(480.0, 1040.0)
        kw = {"ps": ps}
        orc = lambda f, k: vpo.vinterp(1, 1, ap, b, levels, f, ps=k["ps"])  # noqa: E731
    elif branch == "height":
        ap, b = vr._hybrid_table(nk, rng)
        p = ap + b * 1013.25
        levels = np.array([100.0, 1500.0, 9000.0, 30000.0])
        h = HeightInterpolator(PRESSURE, {"p": p}, "linear", levels, type="altitude", converter="standard")
        kw = {}
        orc = lambda f, k: vho.vinterp_height(0, 0, 0, 0, p, None, levels, f)  # noqa: E731
    else:
        s, Cs = vdo.roms_stretching(nk)
        levels = vdo.DEPTHS16[::4].copy()
        hh, eta = vdo.synthetic_ocean(2600, 900, rng)
        h = DepthInterpolator(OCEAN_S_G2, {"s": s, "C": Cs, "depth_c": 250.0}, "linear", levels)
        kw = {"eta": torch.from_numpy(np.tile(eta, (nt, 1))).cuda(), "depth": torch.from_numpy(hh).cuda()}
        orc = lambda f, k: vdo.vinterp_depth(0, vdo.OCEAN_S_G2, s, Cs, levels, f, eta=k["eta"], depth=k["depth"], depth_c=250.0)  # noqa: E731
    out = h.interpolateValues(field, **kw)
    torch.cuda.synchronize()
    assert out.shape == (nt, npt, nxy)
    for t in (0, nt - 1):
        k = {n: (v[t:t + 1] if v.shape[0] == nt and v.dim() == 2 else v).cpu().numpy() for n, v in kw.items()}
        want = orc(field[t:t + 1].cpu().numpy(), k)
        assert_bit_equal(out[t:t + 1].cpu().numpy(), want, f"{branch} step {t} of {nt}")
        assert np.isfinite(want).mean() > 0.5
    del field, out, kw
    gc.collect()
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------------------- the host pipeline in chunks
def _pinned(a, keep):
    """a copy of `a` in page-locked memory from fb200_host_alloc (freed by the caller through `keep`)"""
    lib = fb.load()
    p = lib.fb200_host_alloc(a.nbytes)
    assert p
    keep.append(p)
    out = np.frombuffer((C.c_char * a.nbytes).from_address(p), dtype=a.dtype).reshape(a.shape)
    out[...] = a
    return out


@pytest.mark.parametrize("memory", ["pinned", "pageable"])
@pytest.mark.parametrize("case", ["hypsometric", "field", "depth", "typed"])
def test_host_pipeline_in_chunks(oracle, monkeypatch, case, memory):
    """1 MB chunks of 3 to 9 time steps, the last one partial (31, 46, 75, 39 steps of 280, 194, 115, 225 KB); more than 8 MB per
    call, so pageable arrays go through the bounce buffers; the hypsometric call fills all four per-step slots (field, ps, t, q) and
    uploads zs once, the depth call stages eta and uploads the sea-floor depth once"""
    monkeypatch.setenv("FIMEX_B200_HOST_CHUNK_MB", "1")
    rng = np.random.default_rng(zlib_seed(case + memory))
    nt = {"hypsometric": 31, "field": 46, "depth": 75, "typed": 39}[case]
    nk, nxy, npt = 20, 1031, 7
    if case in ("hypsometric", "typed"):
        h, field, kw, orc = _height(nt, nk, nxy, npt, rng)
        assert set(kw) == {"ps", "t", "q", "zs"}
    elif case == "field":
        h, field, kw, orc = _height(nt, nk, nxy, npt, rng, converter="field", target="height")
    else:
        h, field, kw, orc = _depth(nt, nk, nxy, npt, rng)
    want = orc(field, kw)
    keep = []
    try:
        if memory == "pinned":
            field = _pinned(field, keep)
            kw = {k: _pinned(v, keep) for k, v in kw.items()}
        if case == "typed":
            packed = np.clip(np.round((np.nan_to_num(field, nan=250.0) - 250.0) * 100), -32000, 32000).astype(np.int16)
            packed = _pinned(packed, keep) if memory == "pinned" else packed
            want = oracle.from_float(orc(oracle.as_float(packed, -32767.0), kw), -32767.0, np.int16).reshape(nt, npt, nxy)
            got = h.getDataSlice(packed, bad_value=-32767.0, **kw)
            dev = h.getDataSlice(_cuda(packed), bad_value=-32767.0, **_cuda_kw(kw)).cpu().numpy()
            assert np.array_equal(got, want) and np.array_equal(dev, want)
        else:
            got = h.interpolateValues(field, **kw)
            dev = h.interpolateValues(_cuda(field), **_cuda_kw(kw)).cpu().numpy()
            assert_bit_equal(got, want, f"{case} {memory} host")
            assert_bit_equal(dev, want, f"{case} {memory} device")
            np.testing.assert_array_equal(got.view(np.uint32), dev.view(np.uint32))
        assert np.isfinite(want).mean() > 0.3
    finally:
        for p in keep:
            fb.load().fb200_host_free(p)


def zlib_seed(s):
    return zlib.crc32(s.encode())


# ------------------------------------------------------------------------------------------------------------------- every CDM type
_TYPED = [(np.float32, np.float32, None), (np.int16, np.int16, None), (np.float32, np.int16, -32767.0), (np.int16, np.float32, -32767.0),
          (np.float64, np.float64, None), (np.int32, np.int32, None), (np.uint8, np.uint8, None), (np.int8, np.int8, None),
          (np.uint16, np.uint16, None), (np.uint32, np.uint32, 4000000000.0), (np.int64, np.int64, -9999.0), (np.uint64, np.uint64, 12345.0),
          (np.float32, np.float32, np.nan)]


def _typed_field(rng, shape, dtype, fill):
    dt = np.dtype(dtype)
    if dt.kind == "f":
        a = rng.normal(250, 30, shape).astype(dt)
    else:
        info = np.iinfo(dt)
        a = rng.integers(max(info.min, -30000), min(info.max, 30000), shape, endpoint=True).astype(dt)
    a[rng.random(shape) < 0.03] = dt.type(fill)
    return a


@pytest.mark.parametrize("in_dtype,out_dtype,fill", _TYPED)
@pytest.mark.parametrize("branch", list(BRANCHES))
def test_every_cdm_type(oracle, branch, in_dtype, out_dtype, fill):
    """getDataSlice with every CDM type in and out (the horizontal suite's set): fill -> NaN, interpolate, NaN -> fill and cast, as the
    restatement's as_float / from_float around the vertical restatement; host and device"""
    rng = np.random.default_rng(zlib_seed(f"{branch}{np.dtype(in_dtype)}{np.dtype(out_dtype)}{fill}"))
    nt, nk, nxy, npt = 2, 17, 257, 9
    h, _, kw, orc = BRANCHES[branch](nt, nk, nxy, npt, rng)
    if fill is None:
        fill = fb.default_fill_value(in_dtype)
    data = _typed_field(rng, (nt, nk, nxy), in_dtype, fill)
    want = oracle.from_float(orc(oracle.as_float(data, fill), kw), fill, out_dtype).reshape(nt, npt, nxy)
    got = h.getDataSlice(data, bad_value=fill, out_dtype=out_dtype, **kw)
    import torch
    dev = h.getDataSlice(_cuda(data), bad_value=fill, out_dtype=getattr(torch, np.dtype(out_dtype).name), **_cuda_kw(kw)).cpu().numpy()
    for g, where in ((got, "host"), (dev, "device")):
        assert g.dtype == np.dtype(out_dtype) and g.shape == want.shape, where
        if np.dtype(out_dtype).kind == "f":
            bits = np.uint32 if g.itemsize == 4 else np.uint64
            assert ((g.view(bits) == want.view(bits)) | (np.isnan(g) & np.isnan(want))).all(), where
        else:
            assert np.array_equal(g, want), where
    if not np.isnan(fill):
        assert (want == np.dtype(out_dtype).type(fill)).any()


# ------------------------------------------------------------------------------------------------------------- loglog at <= 1 hPa
def test_loglog_at_and_below_one_hpa(oracle):
    """ERA5's 1 hPa level under a model top near 0.02 hPa: a pair with a level at or below 1 hPa gives NaN, a target of exactly 1 hPa
    extrapolated from levels above it -+inf; the GPU gives what the restatement gives (outside the reference's comparison)"""
    rng = np.random.default_rng(1)
    ap, b = vr._hybrid_table(137, rng)
    levels = np.array([1, 2, 3, 5, 7, 10, 20, 50, 100, 500, 850, 1000], dtype=np.float64)
    field = rng.normal(250, 30, (2, 137, 1031)).astype(np.float32)
    ps = rng.uniform(480, 1040, (2, 1031)).astype(np.float32)
    h = VerticalInterpolator(HYBRID, {"ap": ap, "b": b}, "loglog", levels)
    want = vpo.vinterp(2, 1, ap, b, levels, field, ps=ps)
    _both_paths(h, field, {"ps": ps}, want, "loglog, model top 0.02 hPa")
    assert np.isnan(want[:, 0]).all() and np.isfinite(want[:, 3:]).all()
    p = np.array([1.5, 2.0, 10.0, 50.0, 300.0, 1000.0])
    f = rng.normal(250, 30, (1, p.size, 64)).astype(np.float32)
    hp = VerticalInterpolator(PRESSURE, {"p": p}, "loglog", [1.0, 1.2, 700.0])
    want = vpo.vinterp(2, 0, p, None, [1.0, 1.2, 700.0], f)
    _both_paths(hp, f, {}, want, "loglog, 1 hPa extrapolated")
    assert np.isinf(want[0, 0]).all() and np.isfinite(want[0, 1:]).all()


def test_two_level_formula_is_not_contracted(oracle):
    """targets for which an FMA-contracted A + w (B - A) rounds to another float32 (vertical_reference.contraction_targets): the
    kernel gives the restatement's uncontracted value, host and device"""
    levels, A, B, targets = vr.contraction_targets()
    field = np.tile(np.array([[[A], [B]]], np.float32), (3, 1, 33))
    h = VerticalInterpolator(PRESSURE, {"p": levels}, "linear", targets)
    _both_paths(h, field, {}, vpo.vinterp(0, 0, levels, None, targets, field), "contraction targets")
