"""Vertical interpolation to height and altitude levels, CPU side: independent known answers for the restatement
(tests/vertical_height_oracle.c, orc_vinterp_height) of the contract in DESIGN.md section 2, the C ABI's and the Python layer's argument checks,
and the refusal without a GPU.  The GPU is compared with this restatement bit for bit in test_gpu_vertical_height.py."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import fimex_b200
import vertical_height_oracle as vo
from fimex_b200 import capi
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, HeightInterpolator

LIN, LOG, NN = 0, 1, 3
R, M, MW, G0 = 8.31432, 0.0289644, 0.01801528, 9.80665
H = R / (M * G0)
HB = np.array([0.0, 11000.0, 20000.0, 32000.0, 47000.0, 51000.0, 71000.0])
TB = np.array([288.15, 216.65, 216.65, 228.65, 270.65, 270.65, 214.65])
LB = np.array([-6.5e-3, 0.0, 1e-3, 2.8e-3, 0.0, -2.8e-3, -2e-3])
PB = np.array([1013.25, 226.3206, 54.74889, 8.680187, 1.109063, 0.6693887, 0.03956420])


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture
def quiet():
    os.environ["FIMEX_B200_QUIET"] = "1"
    yield
    os.environ.pop("FIMEX_B200_QUIET", None)


def hybrid_table(nk, rng):
    """the seeded L137-like table of test_gpu_vertical.py (hPa)"""
    u = np.cumsum(rng.uniform(0.6, 1.4, nk))
    u = (u - u[0]) / (u[-1] - u[0])
    eta = np.exp(np.log(2e-5) * (1 - u) ** 1.6)
    b = np.clip((eta - 0.2) / 0.8, 0, None)
    return 1013.25 * (eta - b), b


def zstd_libm(p):
    """the standard converter's formula in numpy with the C library's exp and log"""
    p = np.asarray(p, dtype=np.float64)
    b = np.zeros(p.shape, dtype=int)
    for layer in range(1, 7):
        b = np.where(p <= PB[layer], layer, b)
    L, T, h, P = LB[b], TB[b], HB[b], PB[b]
    with np.errstate(all="ignore"):
        poly = h + T / L * (np.exp(-(R * L) / (G0 * M) * np.log(p / P)) - 1.0)
        iso = h + H * T * np.log(P / p)
    return np.where(L != 0, poly, iso)


def t_std(z):
    b = np.clip(np.searchsorted(HB, z, side="right") - 1, 0, 6)
    return TB[b] + LB[b] * (z - HB[b])


def _field(converter, target, levels, field, z=None, **kw):
    """one or more columns of the field converter: field and z [nk][ncol]"""
    f = np.asarray(field, dtype=np.float32)
    zz = np.asarray(z, dtype=np.float32)
    return vo.vinterp_height(kw.pop("method", LIN), converter, target, vo.VCOORD_PRESSURE, None, None, levels, f.reshape(1, f.shape[0], -1),
                             z=zz.reshape(1, zz.shape[0], -1), **kw)[0]


# ---------------------------------------------------------------------------------------------- the standard converter
def test_base_pressures_approached_from_the_layer_below():
    for layer in range(1, 7):
        p = np.nextafter(PB[layer], np.inf)  # the formula of layer - 1
        assert abs(vo.zstd(p) - HB[layer]) <= 2e-3, (layer, vo.zstd(p))
        assert vo.zstd(PB[layer]) == HB[layer]  # ln 1 = 0 in the layer's own formula


def test_icao_heights():
    for p, h in zip([850, 700, 500, 300, 250, 200, 100, 50], [1457, 3012, 5574, 9164, 10363, 11784, 16180, 20576]):
        assert abs(vo.zstd(p) - h) <= 0.5, (p, vo.zstd(p))


def test_standard_matches_the_formula_with_libm():
    ps = np.concatenate([np.geomspace(0.01, 1100.0, 3001), PB, PB * (1 + 1e-9), PB * (1 - 1e-9)])
    got = np.array([vo.zstd(p) for p in ps])
    np.testing.assert_allclose(got, zstd_libm(ps), rtol=0, atol=1e-6)


def test_vexp_is_within_one_ulp_of_libm():
    xs = np.concatenate([np.linspace(-745, 709.7, 20001), np.linspace(-1, 1, 2001), np.geomspace(1e-300, 1, 301), -np.geomspace(1e-300, 1, 301),
                         [0.0, -0.0, 0.34657359, 1.03972077]])
    for x in xs:
        got, want = vo.vexp(x), math.exp(x)
        assert abs(got - want) <= math.ulp(want), (x, got, want)
    assert vo.vexp(math.inf) == math.inf and vo.vexp(-math.inf) == 0.0 and math.isnan(vo.vexp(math.nan))
    assert vo.vexp(710.0) == math.inf and vo.vexp(-800.0) == 0.0


# ---------------------------------------------------------------------------------------------- the hypsometric converter
def test_isothermal_column_is_the_closed_form():
    rng = np.random.default_rng(4)
    ap, b = hybrid_table(60, rng)
    ps = np.float32(987.5)
    p = ap + b * np.float64(ps)
    for q in (None, 0.004):
        T = np.full(60, 250.0, np.float32)
        qq = None if q is None else np.full(60, q, np.float32)
        zc, d = vo.height_column(vo.HYPSOMETRIC, vo.HEIGHT, vo.VCOORD_HYBRID, ap, b, ps=ps, t=T, q=qq)
        assert d == 0  # surface at k = nk - 1
        tv = 250.0 * (1 + (M / MW - 1) * np.float64(np.float32(q))) if q is not None else 250.0
        want = H * tv * np.log(np.float64(ps) / p)
        np.testing.assert_allclose(zc[:-1], want[:-1], rtol=1e-9)
        assert abs(zc[-1]) <= 1e-9  # the lowest level is at ps
        # altitude: the same plus the surface altitude
        za, _ = vo.height_column(vo.HYPSOMETRIC, vo.ALTITUDE, vo.VCOORD_HYBRID, ap, b, ps=ps, t=T, q=qq, zs=np.float32(1500.0))
        np.testing.assert_allclose(za, zc + 1500.0, rtol=1e-12, atol=1e-9)


def trapezoid_bound(p_walk):
    """DESIGN.md section 2: a bound on |hypsometric - standard| at every level (walk order, from the surface at the standard surface
    pressure), for T(p) of the standard atmosphere itself.  Per layer of the sum, of log-thickness d = ln(p_prev / p): the trapezoid rule
    on T(u), u = ln p, with T'' = kappa^2 T (kappa = -L_b H) gives H d^3 kappa^2 T_max / 12; a layer that holds a base altitude, where
    the slope of T(u) jumps by |kappa_b - kappa_b-1| T_b, adds H d^2 |jump| / 8.  Plus 2 mm per base altitude below (the published
    base pressures are rounded: the standard converter itself jumps there by up to 1.5 mm) and 2^-23 z for T rounded to float."""
    z = zstd_libm(p_walk)
    kappa = -LB * H
    jumps = np.abs(np.diff(kappa)) * TB[1:]
    bound = np.zeros(p_walk.size)
    acc = 0.0
    for m in range(1, p_walk.size):
        d = math.log(p_walk[m - 1] / p_walk[m])
        z0, z1 = z[m - 1], z[m]
        b0, b1 = np.clip(np.searchsorted(HB, [z0, z1], side="right") - 1, 0, 6)
        tmax = float(t_std(np.linspace(z0, z1, 9)).max())
        acc += H * d ** 3 * float((kappa[b0:b1 + 1] ** 2).max()) * tmax / 12
        if b1 > b0:
            acc += H * d ** 2 * float(jumps[b0:b1].max()) / 8
        bound[m] = acc + 2e-3 * np.count_nonzero(HB[1:] <= z1) + 2.0 ** -23 * abs(z1)
    return bound


def test_standard_temperatures_reproduce_the_standard_converter():
    rng = np.random.default_rng(1)
    ap, b = hybrid_table(137, rng)
    ps = np.float32(1013.25)
    p = ap + b * np.float64(ps)  # increasing with k: the surface is k = 136 (eta = 1, p = ps)
    T = t_std(zstd_libm(p)).astype(np.float32)
    zh, d = vo.height_column(vo.HYPSOMETRIC, vo.ALTITUDE, vo.VCOORD_HYBRID, ap, b, ps=ps, t=T, zs=np.float32(0.0))
    zs_, d2 = vo.height_column(vo.STANDARD, vo.ALTITUDE, vo.VCOORD_HYBRID, ap, b, ps=ps)
    assert d == d2 == 0
    diff = np.abs(zh - zs_)[::-1]  # walk order
    bound = trapezoid_bound(p[::-1])
    assert np.all(diff <= bound), np.max(diff - bound)
    low = zs_[::-1] < 20000
    assert diff[low].max() <= 0.75 and diff.max() <= 1.2, (diff[low].max(), diff.max())


# ---------------------------------------------------------------------------------------------- rules of the interpolation
def test_two_levels_linear_and_nearest():
    z = [[0.0], [100.0]]
    v = [[1.0], [3.0]]
    assert list(_field(vo.FIELD, vo.ALTITUDE, [25.0, 0.0, 100.0, 50.0], v, z)[:, 0]) == [1.5, 1.0, 3.0, 2.0]
    assert list(_field(vo.FIELD, vo.ALTITUDE, [49.0, 50.0, 51.0], v, z, method=NN)[:, 0]) == [1.0, 1.0, 3.0]  # a tie: the lower level
    # surface at k = nk - 1: the same answers
    assert list(_field(vo.FIELD, vo.ALTITUDE, [25.0, 50.0], v[::-1], z[::-1])[:, 0]) == [1.5, 2.0]
    assert list(_field(vo.FIELD, vo.ALTITUDE, [50.0, 51.0], v[::-1], z[::-1], method=NN)[:, 0]) == [1.0, 3.0]
    # geopotential with z_scale = 1 / g0, heights above a surface geopotential with zs_scale = 1 / g0
    phi = np.array([[0.0], [100.0 * G0]])
    got = _field(vo.FIELD, vo.HEIGHT, [15.0], v, phi, z_scale=1 / G0, zs=np.array([10.0 * G0], np.float32), zs_scale=1 / G0)
    assert abs(got[0, 0] - 1.5) < 1e-6


def test_extrapolation_modes():
    z = np.array([[10.0], [20.0], [40.0]])
    v = 2 * z + 1
    levels = [0.0, 10.0, 40.0, 50.0]
    assert list(_field(vo.FIELD, vo.ALTITUDE, levels, v, z)[:, 0]) == [1.0, 21.0, 81.0, 101.0]
    off = _field(vo.FIELD, vo.ALTITUDE, levels, v, z, extrapolate=False)[:, 0]
    assert np.isnan(off[0]) and np.isnan(off[3]) and list(off[1:3]) == [21.0, 81.0]
    assert list(_field(vo.FIELD, vo.ALTITUDE, levels, v, z, method=NN)[:, 0]) == [21.0, 21.0, 81.0, 81.0]


def test_nan_levels_end_the_column():
    z = np.array([[10.0], [20.0], [np.nan], [40.0]])
    v = np.array([[1.0], [2.0], [3.0], [4.0]])
    got = _field(vo.FIELD, vo.ALTITUDE, [5.0, 15.0, 20.0, 25.0, 45.0], v, z)[:, 0]
    assert got[0] == 0.5 and got[1] == 1.5 and got[2] == 2.0 and np.isnan(got[3:]).all()
    # equal or NaN ends: a NaN column
    assert np.isnan(_field(vo.FIELD, vo.ALTITUDE, [10.0], [[1.0], [2.0]], [[10.0], [10.0]])).all()
    assert np.isnan(_field(vo.FIELD, vo.ALTITUDE, [10.0], [[1.0], [2.0]], [[np.nan], [10.0]])).all()
    # a NaN surface altitude for heights
    assert np.isnan(_field(vo.FIELD, vo.HEIGHT, [10.0], [[1.0], [2.0]], [[0.0], [100.0]], zs=np.array([np.nan], np.float32))).all()
    # the hypsometric sum: a NaN temperature ends the column there; a NaN ps is a NaN column
    ap, b = np.array([0.0, 0.0, 0.0, 0.0]), np.array([0.5, 0.7, 0.9, 1.0])
    T = np.array([[[230.0], [np.nan], [260.0], [280.0]]], np.float32)
    f = np.array([[[4.0], [3.0], [2.0], [1.0]]], np.float32)
    z1 = H * 0.5 * (280 + 260) * math.log(1 / 0.9)
    got = vo.vinterp_height(LIN, vo.HYPSOMETRIC, vo.HEIGHT, vo.VCOORD_HYBRID, ap, b, [0.0, z1 / 2, z1 + 1.0], f, ps=np.array([[1000.0]], np.float32),
                            t=T)[0, :, 0]
    assert got[0] == 1.0 and abs(got[1] - 1.5) < 1e-6 and np.isnan(got[2])
    got = vo.vinterp_height(LIN, vo.HYPSOMETRIC, vo.HEIGHT, vo.VCOORD_HYBRID, ap, b, [0.0], f, ps=np.array([[np.nan]], np.float32), t=T)
    assert np.isnan(got).all()


def test_standard_height_is_altitude_minus_the_surface():
    p = np.array([1000.0, 850.0, 700.0, 500.0])
    f = zstd_libm(p).astype(np.float32)[None, :, None]  # the field is its own altitude
    alt = vo.vinterp_height(LIN, vo.STANDARD, vo.ALTITUDE, vo.VCOORD_PRESSURE, p, None, [1000.0, 3000.0], f)[0, :, 0]
    np.testing.assert_allclose(alt, [1000.0, 3000.0], rtol=1e-6)
    hgt = vo.vinterp_height(LIN, vo.STANDARD, vo.HEIGHT, vo.VCOORD_PRESSURE, p, None, [1000.0, 3000.0], f, zs=np.array([500.0], np.float32))[0, :, 0]
    np.testing.assert_allclose(hgt, [1500.0, 3500.0], rtol=1e-6)


# ---------------------------------------------------------------------------------------------- the C ABI and the Python layer
def test_height_symbols_are_declared_and_exported():
    names = capi.declared_symbols()
    want = ["fb200_vinterp_create_height", "fb200_vinterp_interpolate_values_columns", "fb200_vinterp_interpolate_values_columns_device",
            "fb200_vinterp_get_data_slice_columns", "fb200_vinterp_get_data_slice_columns_device"]
    lib = capi.load()
    for n in want:
        assert n in names and hasattr(lib, n), n


def _create(method=LIN, converter=1, target=1, vcoord=1, a=(0.0, 0.0), b=(0.5, 1.0), nk=2, ptop=0.0, ps_scale=1.0, z_scale=1.0, zs_scale=1.0,
            levels=(10.0,), handle=True):
    """fb200_vinterp_create_height with one argument changed from a valid hybrid / hypsometric / height call"""
    a, b, lev = (None if v is None else np.asarray(v, dtype=np.float64) for v in (a, b, levels))
    h = C.c_void_p()
    return capi.load().fb200_vinterp_create_height(method, converter, target, vcoord, capi.ptr(a), capi.ptr(b), nk, ptop, ps_scale, z_scale,
                                                   zs_scale, capi.ptr(lev), lev.size, 1, C.byref(h) if handle else None)


@pytest.mark.parametrize("kwargs, message", [
    (dict(method=LOG), "linear and nearestneighbor only"),
    (dict(method=2), "linear and nearestneighbor only"),
    (dict(converter=1, vcoord=0, b=None), "hypsometric converter needs a surface pressure"),
    (dict(converter=3), "unknown height converter"),
    (dict(target=2), "unknown height target"),
    (dict(converter=0, vcoord=5), "unknown source vertical coordinate"),
    (dict(nk=1), "number of source levels"),
    (dict(levels=()), "number of target levels"),
    (dict(levels=(np.nan,)), "target levels must be finite"),
    (dict(z_scale=np.inf), "must be finite"),
    (dict(zs_scale=np.nan), "must be finite"),
    (dict(a=None), "null ap"),
    (dict(vcoord=2, b=None), "null sigma"),
    (dict(handle=False), "null handle pointer"),
])
def test_argument_checks_of_the_c_abi(quiet, kwargs, message):
    assert _create(**kwargs) == fimex_b200.MIFI_ERROR
    assert message in fimex_b200.last_error()


def test_the_calls_refuse_a_null_handle(quiet):
    lib = capi.load()
    assert lib.fb200_vinterp_get_data_slice_columns(None, 5, None, None, 4, 1, 0.0, 5, None) == fimex_b200.MIFI_ERROR
    assert "null vertical interpolation handle" in fimex_b200.last_error()
    assert lib.fb200_vinterp_interpolate_values_columns(None, None, None, 4, 1, None) == fimex_b200.MIFI_ERROR


@pytest.mark.parametrize("kwargs, message", [
    (dict(method="log"), "linear and nearestneighbor only"),
    (dict(method="loglog"), "linear and nearestneighbor only"),
    (dict(standard_name=PRESSURE, terms={"p": [1000.0, 500.0]}), "hypsometric converter needs a surface pressure"),
    (dict(type="depth"), "unknown height target type"),
    (dict(converter="barometric"), "unknown height converter"),
    (dict(standard_name="ocean_s_coordinate", terms={}), "not supported"),
])
def test_argument_checks_of_the_python_layer(quiet, kwargs, message):
    args = dict(standard_name=HYBRID, terms={"ap": [0.0, 0.0], "b": [0.5, 1.0]}, method="linear", levels=[10.0])
    args.update(kwargs)
    with pytest.raises(fimex_b200.FimexB200Error, match=message):
        HeightInterpolator(**args)


def test_no_cpu_fallback_without_gpu(quiet):
    if _has_gpu():
        pytest.skip("a GPU is present; the refusal path cannot be exercised")
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        HeightInterpolator(SIGMA, {"sigma": [0.1, 0.5, 1.0], "ptop": 10.0}, "linear", [10.0, 100.0])
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        HeightInterpolator(PRESSURE, {"p": [1000.0, 500.0]}, "nearestneighbor", [3000.0], type="altitude", converter="standard")
    assert _create() == fimex_b200.MIFI_ERROR and "no usable CUDA device" in fimex_b200.last_error()
