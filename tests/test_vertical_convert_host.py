"""The vertical interpolator's data conversions (theta2T, omega2vwind, add4Dpressure), CPU side: the restatement
(tests/vertical_convert_oracle.c, orc_vconvert) of the contract in DESIGN.md section 2 against the independent longdouble reference and
known answers, the C ABI's and the Python layer's argument checks, and the refusal without a GPU.  The GPU is compared with this
restatement bit for bit in test_gpu_vertical_convert.py."""
import ctypes as C
import os

import numpy as np
import pytest

import fimex_b200
import vertical_convert_oracle as vc
import vertical_convert_reference as vcr
from fimex_b200 import capi
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, PressureConversion

R_STAR, M_AIR, G0 = 8.31432, 0.0289644, 9.80665


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


def _restate(case):
    return vc.vconvert(case.op, case.kind, case.a, case.b, case.nk, field=case.field, ps=case.ps, t=case.t, nt=1, nxy=7, **case.args())


def _reference(case):
    return vcr.reference(case.op, case.kind, case.a, case.b, case.nk, field=case.field, ps=case.ps, t=case.t, nt=1, nxy=7, **case.args())


# ---------------------------------------------------------------------------------------------- the restatement against the reference
def test_restatement_within_the_reference_bound():
    """200 seeded cases, every op x source coordinate more than 20 times"""
    seen, worst = {}, 0.0
    for seed in range(200):
        case = vcr.draw_case(seed, op=seed % 3, kind=(seed // 3) % 3)
        seen[(case.op, case.kind)] = seen.get((case.op, case.kind), 0) + 1
        worst = max(worst, vcr.check(_restate(case), _reference(case), f"seed {seed}"))
    assert len(seen) == 9 and min(seen.values()) >= 20
    assert 0.3 < worst <= 1.0  # the bound is tight enough to see the float32 rounding


def test_the_bound_catches_a_wrong_kappa():
    """theta2T with kappa = 0.286 instead of 2/7 leaves the bound on an ordinary column"""
    case = vcr.draw_case(3, op=vcr.THETA2T, kind=vcr.VCOORD_HYBRID)
    ref = _reference(case)
    p, _ = vcr.pressure(case.kind, case.a, case.b, case.ptop, case.ps_scale, case.ps, case.nk, *ref.ideal.shape[::2])
    wrong = (case.field.reshape(ref.ideal.shape).astype(np.float64) * np.power(p.astype(np.float64) / 1000.0, 0.286)).astype(np.float32)
    with pytest.raises(AssertionError, match="exceeds the bound"):
        vcr.check(wrong, ref, "kappa 0.286")


# ---------------------------------------------------------------------------------------------- known answers
def test_theta_at_1000_hpa_is_t_bit_for_bit():
    theta = np.random.default_rng(1).uniform(150, 2000, (2, 1, 999)).astype(np.float32)
    got = vc.vconvert(vc.THETA2T, vc.VCOORD_PRESSURE, [1000.0], None, 1, field=theta)
    assert got.tobytes() == theta.tobytes()
    ps = np.full((2, 999), 1000.0, np.float32)  # hybrid level with p_k = 0 + 1 * ps = 1000
    assert vc.vconvert(vc.THETA2T, vc.VCOORD_HYBRID, [0.0], [1.0], 1, field=theta, ps=ps).tobytes() == theta.tobytes()


def test_theta2t_against_numpy_power():
    """theta (p / 1000)^(2/7) in numpy float64, rounded to float32: within 1 float32 step over 1e5 random p in [1, 1100] hPa"""
    rng = np.random.default_rng(2)
    p = rng.uniform(1, 1100, 100_000)
    theta = rng.uniform(180, 1500, (1, p.size, 1)).astype(np.float32)
    got = vc.vconvert(vc.THETA2T, vc.VCOORD_PRESSURE, p, None, p.size, field=theta).ravel()
    want = (theta.ravel().astype(np.float64) * np.power(p / 1000.0, 2.0 / 7.0)).astype(np.float32)
    steps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert steps.max() <= 1 and (steps == 0).mean() > 0.99


def test_omega2vwind_against_the_textbook_formula():
    """w = -omega R_d T / (g p), R_d = R* / M written separately, p in Pa: within 1e-12 relative in fp64"""
    rng = np.random.default_rng(3)
    R_d = R_STAR / M_AIR
    for omega, T, p in zip(rng.normal(0, 2, 2000), rng.uniform(180, 320, 2000), rng.uniform(1, 1100, 2000)):
        want = -omega * R_d * T / (G0 * p * 100.0)
        got = vc.value(vc.OMEGA2VWIND, omega, T, p)
        assert abs(got - want) <= 1e-12 * abs(want), (omega, T, p, got, want)


def test_the_pressure_field_interpolated_back_gives_the_targets():
    """add4Dpressure on hybrid levels, then the pressure branch's restatement (linear) interpolates that field to targets inside each
    column: each comes back within the float rounding of its bracket"""
    rng = np.random.default_rng(4)
    ap, b = vcr.vr._hybrid_table(60, rng)
    ps = rng.uniform(500, 1050, (2, 301)).astype(np.float32)
    pf = vc.vconvert(vc.PRESSURE, vc.VCOORD_HYBRID, ap, b, 60, ps=ps)
    assert pf.shape == (2, 60, 301)
    targets = np.array([0.5, 3.0, 10.0, 100.0, 250.0, 480.0])
    got = vc.vinterp_pressure(0, vc.VCOORD_HYBRID, ap, b, targets, pf, ps=ps, extrapolate=False)
    assert np.isfinite(got).all()
    step = np.spacing(np.float32(targets)).astype(np.float64)[None, :, None]
    assert (np.abs(got.astype(np.float64) - targets[None, :, None]) <= step).all()


def test_nan_inputs_give_nan():
    ps = np.array([[np.nan, 1000.0]], np.float32)
    th = np.array([[[300.0, np.nan]]], np.float32)
    out = vc.vconvert(vc.THETA2T, vc.VCOORD_HYBRID, [10.0], [0.9], 1, field=th, ps=ps)
    assert np.isnan(out).all()
    out = vc.vconvert(vc.OMEGA2VWIND, vc.VCOORD_SIGMA, None, [0.5], 1, field=np.array([[[1.0, np.nan, 1.0]]], np.float32),
                      ps=np.array([[900.0, 900.0, 900.0]], np.float32), t=np.array([[[np.nan, 250.0, 250.0]]], np.float32), ptop=10.0)
    assert np.isnan(out.ravel()[:2]).all() and np.isfinite(out.ravel()[2])


# ---------------------------------------------------------------------------------------------- the C ABI and the Python layer
def test_conversion_symbols_are_declared_and_exported():
    names = ("fb200_vconvert_create", "fb200_vconvert_destroy", "fb200_vconvert_values", "fb200_vconvert_values_device")
    assert all(n in capi.declared_symbols() and hasattr(capi.load(), n) for n in names)
    assert "PressureConversion" in fimex_b200.__all__


def _create(op=0, vcoord=1, a=(10.0, 0.0), b=(0.5, 1.0), nk=2, ptop=0.0, ps_scale=1.0, handle=True):
    """fb200_vconvert_create with one argument changed from a valid hybrid theta2T call"""
    a, b = (None if v is None else np.asarray(v, dtype=np.float64) for v in (a, b))
    h = C.c_void_p()
    return capi.load().fb200_vconvert_create(op, vcoord, capi.ptr(a), capi.ptr(b), nk, ptop, ps_scale, C.byref(h) if handle else None)


@pytest.mark.parametrize("kwargs, message", [
    (dict(op=3), "unknown data conversion"),
    (dict(op=-1), "unknown data conversion"),
    (dict(vcoord=3), "unknown source vertical coordinate"),
    (dict(vcoord=-1), "unknown source vertical coordinate"),
    (dict(nk=0), "number of levels must be in [1, 1024]"),
    (dict(nk=1025, a=np.zeros(1025), b=np.zeros(1025)), "number of levels must be in [1, 1024]"),
    (dict(a=None), "null ap"),
    (dict(b=None), "null b"),
    (dict(vcoord=2, b=None), "null sigma"),
    (dict(vcoord=0, a=None), "null ap"),
    (dict(a=(np.nan, 0.0)), "must be finite"),
    (dict(b=(np.inf, 1.0)), "must be finite"),
    (dict(ps_scale=np.nan), "ps_scale and ptop must be finite"),
    (dict(vcoord=2, ptop=np.inf), "ps_scale and ptop must be finite"),
    (dict(handle=False), "null handle pointer"),
])
def test_argument_checks_of_the_c_abi(quiet, kwargs, message):
    assert _create(**kwargs) == fimex_b200.MIFI_ERROR
    assert message in fimex_b200.last_error()


@pytest.mark.parametrize("kwargs, message", [
    (dict(operation="T2theta"), "unknown data conversion"),
    (dict(operation="theta2t"), "unknown data conversion"),
    (dict(standard_name="height", terms={"p": [1.0]}), "not supported"),
    (dict(terms={"ap": [1.0, 2.0]}), "'b'"),
    (dict(terms={"ap": [1.0, 2.0], "b": [0.0]}), "2 values of ap but 1 of b"),
    (dict(terms={"b": [0.0, 1.0]}), "needs the terms ap, b or a, p0, b"),
])
def test_argument_checks_of_the_python_layer(quiet, kwargs, message):
    args = dict(standard_name=HYBRID, terms={"ap": [1.0, 2.0], "b": [0.0, 1.0]}, operation="theta2T")
    args.update(kwargs)
    with pytest.raises((fimex_b200.FimexB200Error, KeyError), match=message):
        PressureConversion(**args)


def test_no_cpu_fallback_without_gpu(quiet):
    if _has_gpu():
        pytest.skip("a GPU is present; the refusal path cannot be exercised")
    for name, terms in ((HYBRID, {"ap": [1.0, 2.0], "b": [0.0, 1.0]}), (SIGMA, {"sigma": [0.5, 1.0], "ptop": 10.0}), (PRESSURE, {"p": [500.0]})):
        for op in ("theta2T", "omega2vwind", "add4Dpressure"):
            with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
                PressureConversion(name, terms, op)
    assert _create() == fimex_b200.MIFI_ERROR and "no usable CUDA device" in fimex_b200.last_error()
    lib = capi.load()
    out = np.empty(4, np.float32)
    field = np.ones(4, np.float32)
    # a handle never exists without a device: the calls refuse the null handle before anything else
    assert lib.fb200_vconvert_values(None, capi.ptr(field), None, 4, 1, capi.ptr(out)) == fimex_b200.MIFI_ERROR
    assert "null data conversion handle" in fimex_b200.last_error()
    assert lib.fb200_vconvert_values_device(None, capi.ptr(field), None, 4, 1, capi.ptr(out), None) == fimex_b200.MIFI_ERROR
    assert "null data conversion handle" in fimex_b200.last_error()
    lib.fb200_vconvert_destroy(None)  # no-op


def test_the_operation_names_are_the_options():
    assert list(fimex_b200.vertical.CONVERSIONS) == ["theta2T", "omega2vwind", "add4Dpressure"]
    assert fimex_b200.vertical.CONVERSIONS == vc.OPS == vcr.OPS
