"""Vertical interpolation to depth levels, CPU side: independent known answers for the restatement (tests/vertical_depth_oracle.c,
orc_vinterp_depth) of the contract in DESIGN.md section 2, the C ABI's and the Python layer's argument checks, and the refusal without a
GPU.  The GPU is compared with this restatement bit for bit in test_gpu_vertical_depth.py."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import fimex_b200
import vertical_depth_oracle as vo
from fimex_b200 import capi
from fimex_b200.vertical import DEPTH, OCEAN_S_G1, OCEAN_S_G2, OCEAN_SIGMA, DepthInterpolator
from vertical_depth_oracle import roms_stretching

LIN, LOG, NN = 0, 1, 3
U = 2.0 ** -53  # unit roundoff of fp64


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


# the CF conventions, appendix D, as written there (depth = h, the sea-floor depth)
def cf_sigma(sigma, eta, depth):
    return eta + sigma * (depth + eta)


def cf_g1(s, Cs, eta, depth, depth_c):
    S = depth_c * s + (depth - depth_c) * Cs
    return S + eta * (1 + S / depth)


def cf_g2(s, Cs, eta, depth, depth_c):
    S = (depth_c * s + depth * Cs) / (depth_c + depth)
    return eta + (eta + depth) * S


def _f32(x):
    return float(np.float32(x))


def _columns(seed, n=300):
    """seeded (h, eta, depth_c) triples, h and eta as float32 values (the library reads them as float)"""
    rng = np.random.default_rng(seed)
    return [(_f32(rng.uniform(5, 3000)), _f32(rng.uniform(-2.5, 2.5)), float(rng.uniform(0, 400))) for _ in range(n)]


# ---------------------------------------------------------------------------------------------- the formulas
def test_z_matches_the_cf_formulas():
    s, Cs = roms_stretching(35)
    sigma = np.linspace(-1, 0, 21)
    for h, eta, dc in _columns(1):
        scale = h + abs(eta)
        np.testing.assert_allclose(vo.column_z(vo.OCEAN_S_G2, s, Cs, dc, h, eta), cf_g2(s, Cs, eta, h, dc), rtol=1e-12, atol=1e-12 * scale)
        np.testing.assert_allclose(vo.column_z(vo.OCEAN_S_G1, s, Cs, dc, h, eta), cf_g1(s, Cs, eta, h, dc), rtol=1e-12, atol=1e-12 * scale)
        np.testing.assert_allclose(vo.column_z(vo.OCEAN_SIGMA, sigma, None, 0.0, h, eta), cf_sigma(sigma, eta, h), rtol=1e-12,
                                   atol=1e-12 * scale)
    lev = np.array([0.0, 3.0, 10.0, 3000.0])
    assert np.array_equal(vo.column_z(vo.DEPTH, lev), -lev)


def test_stretching_table_is_a_roms_table():
    s, Cs = roms_stretching(35, w=True)
    assert s[0] == -1.0 and s[-1] == 0.0 and Cs[0] == -1.0 and Cs[-1] == 0.0
    assert np.all(np.diff(Cs) > 0) and np.all(Cs >= -1) and np.all(Cs <= 0)


def test_g2_identities():
    for h, eta, dc in _columns(2):
        # s = C = 0: S = 0 exactly, so z = eta + (eta + h) * 0 = eta
        assert vo.column_z(vo.OCEAN_S_G2, [0.0, 0.0], [0.0, 0.0], dc, h, eta)[0] == eta
        # s = C = -1: S = (-depth_c - h) / (depth_c + h) = -1 exactly, so z = eta - (eta + h); -h is representable, so the two roundings
        # together are at most 2 * (ulp(eta + h) / 2) away from it
        z = vo.column_z(vo.OCEAN_S_G2, [-1.0, 0.0], [-1.0, 0.0], dc, h, eta)[0]
        assert z == eta - (eta + h)
        assert abs(z + h) <= math.ulp(eta + h), (h, eta, dc, z)


def test_g1_at_the_bottom():
    """s = C = -1.  S = -depth_c - fl(h - depth_c) is within e1 = ulp(|h - depth_c|) of -h (-h is representable); S / h is -1 within
    e1 / h + 2^-53, 1 + S / h is exact (Sterbenz), so eta * (1 + S / h) adds at most |eta| (e1 / h + 2^-52) and the last sum
    ulp(h)."""
    for h, eta, dc in _columns(3):
        z = vo.column_z(vo.OCEAN_S_G1, [-1.0, 0.0], [-1.0, 0.0], dc, h, eta)[0]
        e1 = math.ulp(abs(h - dc))
        bound = e1 + abs(eta) * (e1 / h + 2.0 ** -51) + math.ulp(h)
        assert abs(z + h) <= bound, (h, eta, dc, z + h, bound)
    # the surface: s = C = 0 gives S = 0 and z = eta
    for h, eta, dc in _columns(4, 50):
        assert vo.column_z(vo.OCEAN_S_G1, [0.0, -1.0], [0.0, -1.0], dc, h, eta)[0] == eta


def test_sigma_identities():
    for h, eta, dc in _columns(5):
        z = vo.column_z(vo.OCEAN_SIGMA, [0.0, -1.0], None, 0.0, h, eta)
        assert z[0] == eta
        assert z[1] == eta - (h + eta) and abs(z[1] + h) <= math.ulp(eta + h)


def test_g2_with_c_equal_s_and_no_eta_is_s_times_h():
    """eta = 0, C = s: S = (dc s + h s) / (dc + h); both products have the sign of s, so the numerator carries 3 roundings, the quotient
    one more and h * S the fifth: |z - s h| <= 5u |s h| to first order; 6u with numpy's own product s * h"""
    s, _ = roms_stretching(35)
    for h, _, dc in _columns(6):
        z = vo.column_z(vo.OCEAN_S_G2, s, s, dc, h, 0.0)
        assert np.all(np.abs(z - s * h) <= 6 * U * np.abs(s * h)), (h, dc)


def test_a_field_linear_in_depth_is_reproduced_at_interior_targets():
    s, Cs = roms_stretching(35)
    a, b = 12.5, -0.004  # e.g. temperature [degC] against depth [m]
    targets = np.array([0.0, 3.0, 10.0, 15.0, 25.0, 50.0, 75.0, 100.0, 150.0, 200.0, 250.0, 300.0, 500.0, 1000.0, 2000.0, 3000.0])
    for h, eta, dc in _columns(8, 40):
        for vcoord in (vo.OCEAN_S_G2, vo.OCEAN_S_G1):
            x = -vo.column_z(vcoord, s, Cs, dc, h, eta)
            f = (a + b * x).astype(np.float32)
            got = vo.vinterp_depth(LIN, vcoord, s, Cs, targets, f[None, :, None], eta=np.array([[eta]], np.float32),
                                   depth=np.array([h], np.float32), depth_c=dc, extrapolate=False)[0, :, 0]
            inside = (targets >= x.min()) & (targets <= x.max())
            assert np.isnan(got[~inside]).all()
            tol = 3 * 2.0 ** -24 * np.abs(f).max()  # the two float32 end values and the float32 result
            np.testing.assert_allclose(got[inside], a + b * targets[inside], rtol=0, atol=tol)


# ---------------------------------------------------------------------------------------------- rules of the interpolation
def _levels(levels, field, targets, **kw):
    f = np.asarray(field, dtype=np.float32)
    return vo.vinterp_depth(kw.pop("method", LIN), vo.DEPTH, levels, None, targets, f.reshape(1, f.size, 1), **kw)[0, :, 0]


def test_two_levels_linear_and_nearest():
    assert list(_levels([0.0, 100.0], [1.0, 3.0], [25.0, 0.0, 100.0, 50.0])) == [1.5, 1.0, 3.0, 2.0]
    assert list(_levels([0.0, 100.0], [1.0, 3.0], [49.0, 50.0, 51.0], method=NN)) == [1.0, 1.0, 3.0]  # a tie: the upper level
    # the surface at k = nk - 1: the same answers
    assert list(_levels([100.0, 0.0], [3.0, 1.0], [25.0, 50.0])) == [1.5, 2.0]
    assert list(_levels([100.0, 0.0], [3.0, 1.0], [50.0, 51.0], method=NN)) == [1.0, 3.0]


def test_extrapolation_modes():
    x = np.array([10.0, 20.0, 40.0])
    v = 2 * x + 1
    targets = [0.0, 10.0, 40.0, 50.0]
    assert list(_levels(x, v, targets)) == [1.0, 21.0, 81.0, 101.0]
    off = _levels(x, v, targets, extrapolate=False)
    assert np.isnan(off[0]) and np.isnan(off[3]) and list(off[1:3]) == [21.0, 81.0]
    assert list(_levels(x, v, targets, method=NN)) == [21.0, 21.0, 81.0, 81.0]
    assert list(_levels(x[::-1], v[::-1], targets)) == [1.0, 21.0, 81.0, 101.0]


def test_ocean_extrapolation_above_the_top_level_and_below_the_sea_floor():
    """sigma levels -0.9 ... -0.1 of a 100 m column with eta = 1: x from -1 + 0.1 * 101 = 9.1 m down to -1 + 0.9 * 101 = 89.9 m"""
    sigma = np.array([-0.9, -0.5, -0.1])
    f = np.array([[[9.0], [5.0], [1.0]]], np.float32)
    kw = dict(eta=np.array([[1.0]], np.float32), depth=np.array([100.0], np.float32))
    targets = [0.0, 9.2, 89.8, 100.0]
    on = vo.vinterp_depth(LIN, vo.OCEAN_SIGMA, sigma, None, targets, f, **kw)[0, :, 0]
    off = vo.vinterp_depth(LIN, vo.OCEAN_SIGMA, sigma, None, targets, f, extrapolate=False, **kw)[0, :, 0]
    assert np.isnan(off[[0, 3]]).all() and np.array_equal(off[1:3], on[1:3])
    np.testing.assert_allclose(on, [1 - 9.1 * 4 / 40.4, 1 + 0.1 * 4 / 40.4, 9 - 0.1 * 4 / 40.4, 9 + 10.1 * 4 / 40.4], rtol=1e-6)


def test_nan_columns():
    s, Cs = roms_stretching(10)
    f = np.arange(10, dtype=np.float32)[None, :, None].repeat(6, axis=2)
    depth = np.array([100.0, np.nan, 0.0, -5.0, 100.0, 100.0], np.float32)
    eta = np.array([[0.3, 0.3, 0.3, 0.3, np.nan, -0.2]], np.float32)
    for vcoord in (vo.OCEAN_SIGMA, vo.OCEAN_S_G1, vo.OCEAN_S_G2):
        got = vo.vinterp_depth(LIN, vcoord, s, Cs, [5.0, 50.0], f, eta=eta, depth=depth, depth_c=20.0)[0]
        assert np.isfinite(got[:, [0, 5]]).all() and np.isnan(got[:, 1:5]).all(), vcoord
        # eta not given: 0
        got0 = vo.vinterp_depth(LIN, vcoord, s, Cs, [5.0, 50.0], f, depth=depth, depth_c=20.0)[0]
        assert np.isfinite(got0[:, [0, 4, 5]]).all() and np.isnan(got0[:, 1:4]).all()
    # equal ends
    assert np.isnan(_levels([10.0, 10.0], [1.0, 2.0], [10.0])).all()


# ---------------------------------------------------------------------------------------------- the C ABI and the Python layer
def test_depth_symbols_are_declared_and_exported():
    assert "fb200_vinterp_create_depth" in capi.declared_symbols() and hasattr(capi.load(), "fb200_vinterp_create_depth")


def _create(method=LIN, vcoord=6, s=(-1.0, 0.0), Cs=(-1.0, 0.0), nk=2, depth_c=10.0, levels=(10.0,), handle=True):
    """fb200_vinterp_create_depth with one argument changed from a valid g2 call"""
    s, Cs, lev = (None if v is None else np.asarray(v, dtype=np.float64) for v in (s, Cs, levels))
    h = C.c_void_p()
    return capi.load().fb200_vinterp_create_depth(method, vcoord, capi.ptr(s), capi.ptr(Cs), nk, depth_c, capi.ptr(lev), lev.size, 1,
                                                  C.byref(h) if handle else None)


@pytest.mark.parametrize("kwargs, message", [
    (dict(method=LOG), "linear and nearestneighbor only"),
    (dict(method=2), "linear and nearestneighbor only"),
    (dict(vcoord=2), "unknown depth source vertical coordinate"),
    (dict(vcoord=7), "unknown depth source vertical coordinate"),
    (dict(Cs=None), "null C"),
    (dict(vcoord=5, Cs=None), "null C"),
    (dict(s=None), "null s"),
    (dict(vcoord=4, s=None), "null sigma"),
    (dict(depth_c=-1.0), "depth_c must be finite and >= 0"),
    (dict(depth_c=np.nan), "depth_c must be finite and >= 0"),
    (dict(depth_c=np.inf), "depth_c must be finite and >= 0"),
    (dict(nk=1), "number of source levels"),
    (dict(nk=1025, s=np.zeros(1025), Cs=np.zeros(1025)), "number of source levels"),
    (dict(levels=()), "number of target levels"),
    (dict(levels=np.zeros(1025)), "number of target levels"),
    (dict(levels=(np.nan,)), "target levels must be finite"),
    (dict(s=(-1.0, np.inf)), "must be finite"),
    (dict(handle=False), "null handle pointer"),
])
def test_argument_checks_of_the_c_abi(quiet, kwargs, message):
    assert _create(**kwargs) == fimex_b200.MIFI_ERROR
    assert message in fimex_b200.last_error()


@pytest.mark.parametrize("kwargs, message", [
    (dict(method="log"), "linear and nearestneighbor only"),
    (dict(method="loglog"), "linear and nearestneighbor only"),
    (dict(method="cubic"), "unknown vertical interpolation method"),
    (dict(standard_name="ocean_s_coordinate", terms={}), "not supported for depth levels"),
    (dict(standard_name="atmosphere_sigma_coordinate", terms={"sigma": [0.5, 1.0]}), "not supported for depth levels"),
    (dict(terms={"s": [-1.0, 0.0], "depth_c": 10.0}), "needs the terms s, C, depth_c"),
    (dict(terms={"s": [-1.0, 0.0], "C": [-1.0, -0.5, 0.0], "depth_c": 10.0}), "2 values of s but 3 of C"),
    (dict(standard_name=OCEAN_SIGMA, terms={"eta": 0.0, "depth": 1.0}), "needs the terms sigma"),
    (dict(standard_name=DEPTH, terms={"z": [0.0, 10.0]}), "needs the terms depth"),
])
def test_argument_checks_of_the_python_layer(quiet, kwargs, message):
    args = dict(standard_name=OCEAN_S_G2, terms={"s": [-1.0, 0.0], "C": [-1.0, 0.0], "depth_c": 10.0}, method="linear", levels=[10.0])
    args.update(kwargs)
    with pytest.raises(fimex_b200.FimexB200Error, match=message):
        DepthInterpolator(**args)


def test_no_cpu_fallback_without_gpu(quiet):
    if _has_gpu():
        pytest.skip("a GPU is present; the refusal path cannot be exercised")
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        DepthInterpolator(OCEAN_S_G1, {"s": [-1.0, 0.0], "C": [-1.0, 0.0], "depth_c": 10.0, "eta": None, "depth": None}, "linear", [10.0])
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        DepthInterpolator(DEPTH, {"depth": [0.0, 10.0, 50.0]}, "nearestneighbor", [3.0])
    assert _create() == fimex_b200.MIFI_ERROR and "no usable CUDA device" in fimex_b200.last_error()


def test_the_names_are_the_cf_standard_names():
    assert (DEPTH, OCEAN_SIGMA, OCEAN_S_G1, OCEAN_S_G2) == ("depth", "ocean_sigma_coordinate", "ocean_s_coordinate_g1", "ocean_s_coordinate_g2")
