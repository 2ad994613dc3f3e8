"""Vertical interpolation to pressure levels, CPU side: known answers of the oracle's restatement (tests/vertical_oracle.c,
orc_vinterp_pressure) of the semantics DESIGN.md section 2 commits to, the method-string parser, and the C ABI's argument checks
and its refusal without a GPU.  The GPU is compared with this oracle bit for bit in test_gpu_vertical.py."""
import math
import os

import numpy as np
import pytest

import fimex_b200
import vertical_oracle as vo
from fimex_b200 import capi
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, VerticalInterpolator, vertical_method

LIN, LOG, LOGLOG, NN = 0, 1, 2, 3


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


def _pressure(method, p, field, levels, extrapolate=True):
    """pressure levels p (one column per value of the trailing axis of field [nk][ncol])"""
    f = np.asarray(field, dtype=np.float32)
    return vo.vinterp(method, vo.VCOORD_PRESSURE, p, None, levels, f.reshape(1, len(p), -1), extrapolate=extrapolate)[0]


def test_vlog_is_within_one_ulp_of_libm():
    xs = np.concatenate([np.geomspace(1e-300, 1e300, 2001), np.linspace(0.5, 2.0, 2001), np.linspace(1 - 1e-6, 1 + 1e-6, 101), [5e-324, 1.0]])
    for x in xs:
        got, want = vo.vlog(x), math.log(x)
        assert abs(got - want) <= math.ulp(want) + 1e-300, (x, got, want)
    assert vo.vlog(0.0) == -math.inf and math.isnan(vo.vlog(-1.0)) and vo.vlog(math.inf) == math.inf


def test_linear_reproduces_a_field_linear_in_p():
    p = np.array([10.0, 50.0, 100.0, 300.0, 700.0, 1000.0])
    levels = np.array([10.0, 25.0, 99.5, 500.0, 850.0, 1000.0, 333.25])
    got = _pressure(LIN, p, (2 * p + 1)[:, None], levels)
    np.testing.assert_allclose(got[:, 0], 2 * levels + 1, rtol=1e-7)


def test_log_reproduces_a_field_linear_in_ln_p():
    p = np.array([1.0, 5.0, 30.0, 200.0, 600.0, 1013.0])
    levels = np.array([2.0, 10.0, 100.0, 500.0, 925.0, 1013.0, 1.0])
    field = (250 + 10 * np.log(p)).astype(np.float32)
    got = _pressure(LOG, p, field[:, None], levels)
    # the inputs are float32: the error is that of the field's rounding, not of the weights
    np.testing.assert_allclose(got[:, 0], 250 + 10 * np.log(levels), rtol=2e-7)


def test_loglog_is_linear_in_ln_ln_p():
    p = np.array([2.0, 10.0, 100.0, 1000.0])
    field = (np.log(np.log(p)) * 4).astype(np.float32)
    levels = np.array([5.0, 50.0, 500.0])
    got = _pressure(LOGLOG, p, field[:, None], levels)
    np.testing.assert_allclose(got[:, 0], 4 * np.log(np.log(levels)), rtol=1e-6)


def test_nearest_neighbour_picks_and_ties():
    p = np.array([100.0, 200.0, 300.0])
    vals = np.array([1.0, 2.0, 3.0])
    levels = np.array([149.0, 150.0, 151.0, 250.0, 299.0, 100.0])
    got = _pressure(NN, p, vals[:, None], levels)[:, 0]
    assert list(got) == [1.0, 1.0, 2.0, 2.0, 3.0, 1.0]  # 150 and 250 are ties: the lower k
    # decreasing column: the tie at 150 (between k = 1 at 200 and k = 2 at 100) takes k = 1
    got = _pressure(NN, p[::-1], vals[::-1, None], levels)[:, 0]
    assert list(got) == [1.0, 2.0, 2.0, 3.0, 3.0, 1.0]


def test_extrapolation_modes():
    p = np.array([100.0, 200.0, 400.0])
    field = (2 * p + 1)[:, None]
    levels = np.array([50.0, 100.0, 400.0, 500.0])
    on = _pressure(LIN, p, field, levels, extrapolate=True)[:, 0]
    assert list(on) == [101.0, 201.0, 801.0, 1001.0]  # the end pair on each side, continued linearly
    off = _pressure(LIN, p, field, levels, extrapolate=False)[:, 0]
    assert np.isnan(off[0]) and np.isnan(off[3]) and list(off[1:3]) == [201.0, 801.0]
    nn = _pressure(NN, p, field, levels, extrapolate=True)[:, 0]
    assert list(nn) == [201.0, 201.0, 801.0, 801.0]  # the end level


def test_increasing_and_decreasing_columns_agree():
    rng = np.random.default_rng(3)
    p = np.sort(rng.uniform(1, 1100, 40))
    field = rng.normal(250, 20, (40, 7)).astype(np.float32)
    levels = rng.uniform(0.5, 1200, 30)
    for m in (LIN, LOG, NN):
        up = _pressure(m, p, field, levels)
        down = _pressure(m, p[::-1].copy(), field[::-1].copy(), levels)
        np.testing.assert_array_equal(up, down)


def test_hybrid_sigma_and_ps_scale():
    ap = np.array([0.0, 50.0, 100.0, 60.0, 0.0])
    b = np.array([0.0, 0.1, 0.4, 0.8, 1.0])
    ps_hpa = np.array([1000.0, 850.0, 600.0], dtype=np.float32)
    levels = np.array([1000.0, 700.0, 500.0, 300.0, 10.0])
    p = ap[:, None] + b[:, None] * ps_hpa.astype(np.float64)[None, :]  # [nk][ncol]
    field = (p * 3 - 7).astype(np.float32)
    got = vo.vinterp(LIN, vo.VCOORD_HYBRID, ap, b, levels, field[None], ps=ps_hpa[None])[0]
    want = np.empty_like(got)
    for c in range(3):
        want[:, c] = np.interp(levels, p[:, c], p[:, c] * 3 - 7)  # inside the column everywhere except 1000 hPa over 850 / 600
    inside = levels[:, None] <= ps_hpa[None, :]
    np.testing.assert_allclose(got[inside], want[inside], rtol=1e-6)
    # a Pa field with ps_scale 0.01
    ps_pa = (ps_hpa.astype(np.float64) * 100).astype(np.float32)
    got_pa = vo.vinterp(LIN, vo.VCOORD_HYBRID, ap, b, levels, field[None], ps=ps_pa[None], ps_scale=0.01)[0]
    np.testing.assert_allclose(got_pa[inside], want[inside], rtol=1e-6)
    # sigma: p = ptop + sigma (ps - ptop)
    sigma = np.array([0.0, 0.25, 0.5, 1.0])
    ptop = 10.0
    ps = np.array([1000.0], dtype=np.float32)
    ps_col = ptop + sigma * (1000.0 - ptop)
    got = vo.vinterp(LIN, vo.VCOORD_SIGMA, None, sigma, [505.0, 257.5], (2 * ps_col + 1).astype(np.float32)[None, :, None], ps=ps[None],
                         ptop=ptop)[0]
    np.testing.assert_allclose(got[:, 0], [1011.0, 516.0], rtol=1e-7)


def test_nan_cases():
    # a flat column
    got = _pressure(LIN, np.array([500.0, 500.0, 500.0]), np.ones((3, 1)), [500.0])
    assert np.isnan(got).all()
    # loglog at p <= 1: ln ln p is NaN (p < 1) or -inf (p == 1)
    p = np.array([0.5, 2.0, 10.0])
    got = _pressure(LOGLOG, p, np.array([[1.0], [2.0], [3.0]]), [0.8, 1.5])
    assert np.isnan(got).all()
    # NaN inputs propagate through the weights; nearest neighbour only when the NaN is the level it picks
    p = np.array([100.0, 200.0, 300.0])
    field = np.array([[np.nan], [2.0], [3.0]])
    assert np.isnan(_pressure(LIN, p, field, [150.0])).all()
    assert _pressure(LIN, p, field, [250.0])[0, 0] == 2.5
    assert _pressure(NN, p, field, [160.0])[0, 0] == 2.0
    assert np.isnan(_pressure(NN, p, field, [140.0])).all()
    # a NaN surface pressure
    got = vo.vinterp(LIN, vo.VCOORD_HYBRID, [0.0, 0.0], [0.5, 1.0], [500.0], np.ones((1, 2, 1), np.float32),
                         ps=np.array([[np.nan]], np.float32))
    assert np.isnan(got).all()


def test_method_strings():
    assert [vertical_method(s) for s in ("linear", "log", "loglog", "nearestneighbor")] == [0, 1, 2, 3]
    for bad in ("Linear", "nearest", "", "log-log"):
        with pytest.raises(fimex_b200.FimexB200Error):
            vertical_method(bad)


def test_vertical_symbols_are_declared_and_exported():
    names = capi.declared_symbols()
    want = ["fb200_vinterp_create_hybrid", "fb200_vinterp_create_sigma", "fb200_vinterp_destroy", "fb200_vinterp_interpolate_values",
            "fb200_vinterp_interpolate_values_device", "fb200_vinterp_get_data_slice", "fb200_vinterp_get_data_slice_device"]
    lib = capi.load()
    for n in want:
        assert n in names and hasattr(lib, n), n


@pytest.mark.parametrize("kwargs, message", [
    (dict(terms={"p": [500.0]}), "number of source levels"),
    (dict(levels=[]), "number of target levels"),
    (dict(levels=[500.0, np.nan]), "target levels must be finite"),
    (dict(levels=[np.inf]), "target levels must be finite"),
    (dict(terms={"p": [1000.0, np.nan]}), "must be finite"),
    (dict(ps_scale=np.nan), "ps_scale"),
])
def test_argument_checks(quiet, kwargs, message):
    args = dict(standard_name=PRESSURE, terms={"p": [1000.0, 500.0]}, method="linear", levels=[700.0])
    args.update(kwargs)
    with pytest.raises(fimex_b200.FimexB200Error, match=message):
        VerticalInterpolator(**args)


def test_argument_checks_of_the_c_abi(quiet):
    import ctypes as C
    lib = capi.load()
    h = C.c_void_p()
    lev = np.array([500.0])
    p = np.array([1000.0, 100.0])
    assert lib.fb200_vinterp_create_hybrid(7, capi.ptr(p), None, 2, 1.0, capi.ptr(lev), 1, 1, C.byref(h)) == fimex_b200.MIFI_ERROR
    assert "unknown vertical interpolation method" in fimex_b200.last_error()
    assert lib.fb200_vinterp_create_hybrid(0, None, None, 2, 1.0, capi.ptr(lev), 1, 1, C.byref(h)) == fimex_b200.MIFI_ERROR
    assert "null ap" in fimex_b200.last_error()
    assert lib.fb200_vinterp_create_sigma(0, capi.ptr(p), 2, 1.0, 1.0, None, 1, 1, C.byref(h)) == fimex_b200.MIFI_ERROR
    assert "null target levels" in fimex_b200.last_error()
    assert lib.fb200_vinterp_create_sigma(0, capi.ptr(p), 2, 1.0, 1.0, capi.ptr(lev), 1, 1, None) == fimex_b200.MIFI_ERROR
    assert "null handle pointer" in fimex_b200.last_error()
    assert lib.fb200_vinterp_interpolate_values(None, None, None, 4, 1, None) == fimex_b200.MIFI_ERROR
    assert "null vertical interpolation handle" in fimex_b200.last_error()
    with pytest.raises(fimex_b200.FimexB200Error, match="needs the terms"):
        VerticalInterpolator(HYBRID, {"b": [0.0, 1.0]}, "log", [500.0])
    with pytest.raises(fimex_b200.FimexB200Error, match="not supported"):
        VerticalInterpolator("ocean_s_coordinate", {}, "log", [500.0])


def test_no_cpu_fallback_without_gpu(quiet):
    if _has_gpu():
        pytest.skip("a GPU is present; the refusal path cannot be exercised")
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        VerticalInterpolator(SIGMA, {"sigma": [0.1, 0.5, 1.0], "ptop": 10.0}, "log", [850.0, 500.0])
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        VerticalInterpolator(HYBRID, {"a": [0.0, 0.1], "p0": 1000.0, "b": [0.5, 1.0]}, "nearestneighbor", [850.0])


def _reference_header():
    path = os.path.join(os.environ.get("REFERENCE", "/root/reference"), "include", "fimex", "interpolation.h")
    return open(path).read() if os.path.exists(path) else None


def test_two_level_formula_against_the_reference(reference):
    """The reference's own mifi_get_values_linear_f / _log_f / _log_log_f against the oracle's two-level step: pins the operation
    order of the formula (DESIGN.md section 2 marks it unpinned where the reference is not compiled)."""
    import ctypes as C
    import re
    header = _reference_header()
    if header is None:
        pytest.skip("reference header not available")
    names = {LIN: "mifi_get_values_linear_f", LOG: "mifi_get_values_log_f", LOGLOG: "mifi_get_values_log_log_f"}
    for name in names.values():
        m = re.search(r"int\s+" + name + r"\s*\(([^)]*)\)", header)
        if m is None or not hasattr(reference.lib, name):
            pytest.skip(f"{name} not in the reference")
        params = [p.strip() for p in m.group(1).split(",")]
        assert len(params) == 7 and "float" in params[0] and "float" in params[2] and "double" in params[4], params
    rng = np.random.default_rng(11)
    A = rng.normal(250, 30, 4096).astype(np.float32)
    B = rng.normal(250, 30, 4096).astype(np.float32)
    for method, name in names.items():
        f = getattr(reference.lib, name)
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_double, C.c_double, C.c_double]
        for a, b, x in ((300.0, 500.0, 400.0), (500.0, 300.0, 350.0), (850.0, 925.0, 1000.0), (2.0, 3.0, 2.5)):
            ref = np.empty_like(A)
            f(A.ctypes.data, B.ctypes.data, ref.ctypes.data, A.size, a, b, x)
            orc = vo.vint_values(method, A, B, a, b, x)
            if method == LIN:
                np.testing.assert_array_equal(orc.view(np.uint32), ref.view(np.uint32))
            else:  # the reference's ln() is the C library's
                np.testing.assert_allclose(orc, ref, rtol=2e-7)
