"""Time interpolation (CDMTimeInterpolator's linear change of the time axis), CPU side: known answers of the time-change map and of the
time specification, the restatement (tests/time_interp_oracle.py) against an independent reference in exact rationals and against the
reference's own mifi_get_values_linear_f, the C ABI's and the Python layer's argument checks, and the refusal without a GPU.  The GPU
is compared with the restatement bit for bit in test_gpu_time_interp.py."""
import ctypes as C
import os
from fractions import Fraction

import numpy as np
import pytest

import fimex_b200
import time_interp_oracle as to
import vertical_oracle as vo
from fimex_b200 import capi
from fimex_b200.timeinterp import TimeInterpolator, expand_sequence, expand_time_spec, parse_time_unit

HOURS = "hours since 1970-01-01 00:00:00"


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


# ---------------------------------------------------------------------------------------------- the time-change map
def test_three_hourly_to_hourly():
    ia, ib, w = to.time_map([0.0, 3.0, 6.0], np.arange(7.0))
    assert ia.tolist() == [0, 0, 0, 0, 1, 1, 1] and ib.tolist() == [1, 1, 1, 1, 2, 2, 2]
    assert w.tolist() == [0.0, 1 / 3, 2 / 3, 1.0, 1 / 3, 2 / 3, 1.0]


def test_extrapolation_uses_the_end_pairs_and_nan_rows_without_it():
    times = [0.0, 3.0, 6.0, 12.0]
    ia, ib, w = to.time_map(times, [-3.0, 15.0, 12.0, 0.0])
    assert ia.tolist() == [0, 2, 2, 0] and ib.tolist() == [1, 3, 3, 1]
    assert w.tolist() == [-1.0, 1.5, 1.0, 0.0]
    ia, ib, w = to.time_map(times, [-3.0, 15.0, 12.0, -1e-300])
    ia_off, ib_off, _ = to.time_map(times, [-3.0, 15.0, 12.0, -1e-300], extrapolate=False)
    assert ia_off.tolist() == [-1, -1, 2, -1] and ib_off.tolist() == [-1, -1, 3, -1]


def test_unsorted_and_repeated_targets():
    ia, ib, w = to.time_map([0.0, 10.0, 20.0], [15.0, 5.0, 15.0, 10.0, 10.0, 0.0])
    assert ia.tolist() == [1, 0, 1, 0, 0, 0]  # 10 is in [0, 10] first
    assert w.tolist() == [0.5, 0.5, 0.5, 1.0, 1.0, 0.0]


def test_an_exact_hit_blends_and_propagates_nan():
    """a target on a source time goes through the formula: the other step of its bracket enters as 0 * (B - A)"""
    A = np.array([1.0, 2.0], np.float32)
    B = np.array([np.nan, np.inf], np.float32)
    got = vo.vint_values(vo.LIN, A, B, 0.0, 3.0, 0.0)
    assert np.isnan(got).all()


def test_signed_zero_follows_the_sign_of_b_minus_a():
    """A = -0, w = 0: -0 + 0 * (B - A) is -0 for B < 0 and +0 for B > 0 (before the store, which adds +0)"""
    A = np.array([-0.0, -0.0], np.float32)
    got = vo.vint_values(vo.LIN, A, np.array([-1.0, 1.0], np.float32), 0.0, 1.0, 0.0)
    assert np.signbit(got).tolist() == [True, False]


# ---------------------------------------------------------------------------------------------- the time specification
def test_absolute_time_in_hours_since_1970():
    got = expand_time_spec("2000-01-01 00:00:00", [0.0, 1.0], HOURS)
    assert got.tolist() == [262968.0]
    got = expand_time_spec("2000-01-01 00:00:00,2000-01-01 06:00:00,...,2000-01-02 00:00:00", [262968.0, 262992.0], HOURS)
    assert got.tolist() == [262968.0 + 6 * i for i in range(5)]
    assert expand_time_spec("1970-01-02 00:00:00", [0.0, 1.0], "days since 1970-01-01").tolist() == [1.0]
    assert expand_time_spec("2000-01-01 00:00:30", [0.0, 1.0], "minutes since 2000-01-01 00:00:00").tolist() == [0.5]


def test_sequence_expansion():
    assert expand_sequence(["0", "3", "...", "12"], None) == [0, 3, 6, 9, 12]
    assert expand_sequence(["0", "3", "...", "13"], None) == [0, 3, 6, 9, 12]
    assert expand_sequence(["1", "5", "7", "...", "11"], None) == [1, 5, 7, 9, 11]
    assert expand_sequence(["0", "0.1", "...", "0.3"], None) == [0.0, 0.1, 0.2, 0.30000000000000004]
    assert expand_sequence(["2", "4"], None) == [2.0, 4.0]


def test_a_sequence_beyond_the_target_limit_raises_before_it_is_formed():
    """0,1e-6,...,1e6 would be 10^12 values: refused at once, as are 2^20 + 1; 2^20 values are accepted"""
    import time
    t0 = time.perf_counter()
    with pytest.raises(fimex_b200.FimexB200Error, match="more than 1048576"):
        expand_time_spec("0,1e-6,...,1e6;unit=hours", [0.0, 1.0], HOURS)
    with pytest.raises(fimex_b200.FimexB200Error, match="more than 1048576"):
        expand_sequence(["0", "1", "...", str(2 ** 20)], None)
    assert time.perf_counter() - t0 < 1.0
    assert len(expand_sequence(["0", "1", "...", str(2 ** 20 - 1)], None)) == 2 ** 20


def test_x_is_the_last_source_time():
    src = [262968.0, 262971.0, 262974.0, 262977.0]
    got = expand_time_spec("2000-01-01 00:00:00,2000-01-01 01:00:00,...,x", src, HOURS)
    assert got.tolist() == [262968.0 + i for i in range(10)]
    got = expand_time_spec("0,1,...,x;unit=hours", src, HOURS)  # base: the first source time rounded down to a whole hour
    assert got.tolist() == [262968.0 + i for i in range(10)]
    got = expand_time_spec("0,2,...,x;relativeStart=1;unit=hours", [262968.5, 262977.0], HOURS)
    assert got.tolist() == [262969.0, 262971.0, 262973.0, 262975.0, 262977.0]
    got = expand_time_spec("0,30,...,90;unit=minutes", [262968.26, 262977.0], HOURS)  # 15.6 minutes past the hour: base at 15
    assert got.tolist() == [262968.25, 262968.75, 262969.25, 262969.75]


@pytest.mark.parametrize("spec", ["", "0,3,...,12", "2000-01-01", "2000-01-01T00:00:00", "2000-13-01 00:00:00", "2000-01-01 00:00:00,,x",
                                  "0,...,12;unit=hours", "0,3,...;unit=hours", "3,0,...,12;unit=hours", "0,3,...,12,...,24;unit=hours",
                                  "0,3;unit=weeks", "0,3;unit=hours;unit=hours", "0,3;step=1;unit=hours", "a,b;unit=hours", "0,3;relativeStart=z;unit=hours"])
def test_malformed_specifications_raise(spec):
    with pytest.raises(fimex_b200.FimexB200Error):
        expand_time_spec(spec, [0.0, 24.0], HOURS)


@pytest.mark.parametrize("unit, calendar", [("hours", "standard"), ("weeks since 2000-01-01", "standard"), ("hours since 2000-1-1 0:0", "noleap"),
                                            ("hours after 2000-01-01", "standard"), ("hours since 2000-02-30", "standard")])
def test_unsupported_units_and_calendars_raise(unit, calendar):
    with pytest.raises(fimex_b200.FimexB200Error):
        parse_time_unit(unit, calendar)


def test_units_parse():
    assert parse_time_unit("hours since 2000-1-1 0:0")[0] == 3600
    assert parse_time_unit("days since 1970-01-01T00:00:00Z", "proleptic_gregorian") == (86400, np.datetime64("1970-01-01T00:00:00", "s"))
    assert parse_time_unit("seconds since 1850-01-01", "gregorian")[0] == 1
    with pytest.raises(fimex_b200.FimexB200Error, match="1582-10-15"):
        expand_time_spec("1500-01-01 00:00:00", [0.0, 1.0], "days since 1400-01-01")
    assert expand_time_spec("1400-01-02 00:00:00", [0.0, 1.0], "days since 1400-01-01", "proleptic_gregorian").tolist() == [1.0]


# ---------------------------------------------------------------------------------------------- the restatement
def _exact(times, tau, A, B):
    """the definition in exact rationals: the smallest bracket, or the end pair outside; A + (tau - t_k) / (t_k+1 - t_k) (B - A)"""
    t = [Fraction(float(x)) for x in times]
    x = Fraction(float(tau))
    if x < t[0]:
        k = 0
    elif x > t[-1]:
        k = len(t) - 2
    else:
        k = min(i for i in range(len(t) - 1) if t[i] <= x <= t[i + 1])
    w = (x - t[k]) / (t[k + 1] - t[k])
    return k, [Fraction(float(a)) + w * (Fraction(float(b)) - Fraction(float(a))) for a, b in zip(A, B)]


def test_restatement_against_exact_rationals():
    """200 seeded cases: the same bracket, and the float32 result within half a float32 step of the exact value plus the fp64 rounding
    of the blend (2^-50 (|A| + |w (B - A)|)); nearly always the correctly rounded value itself"""
    total = exact_hits = 0
    for seed in range(200):
        r = np.random.default_rng(seed)
        nt = int(r.integers(2, 9))
        times = np.cumsum(r.choice([1.0, 3.0, 6.0, r.uniform(0.1, 10)], nt)) + r.uniform(-1e5, 1e5)
        taus = np.concatenate([r.uniform(times[0] - 5, times[-1] + 5, 4), r.choice(times, 2)])
        ia, ib, w = to.time_map(times, taus)
        for j, tau in enumerate(taus):
            A = r.normal(250, 80, 16).astype(np.float32)
            B = (A + r.normal(0, 10, 16)).astype(np.float32) if seed % 2 else r.normal(0, 1e3, 16).astype(np.float32)
            k, want = _exact(times, tau, A, B)
            assert ia[j] == k and ib[j] == k + 1
            got = vo.vint_values(vo.LIN, A, B, times[k], times[k + 1], tau)
            for g, e, a, b in zip(got, want, A, B):
                err = abs(Fraction(float(g)) - e)
                bound = Fraction(float(np.spacing(np.float32(abs(float(e)))))) / 2 + Fraction(2.0 ** -50) * (abs(Fraction(float(a))) + abs(e - Fraction(float(a))))
                assert err <= bound, (seed, j, g, float(e))
                exact_hits += float(g) == float(np.float32(float(e)))
                total += 1
    assert total >= 200 * 6 * 16 and exact_hits / total > 0.999


def test_two_level_step_against_the_reference(reference):
    """the reference's own mifi_get_values_linear_f with time arguments (a = t_k, b = t_k+1, x = tau) against the restatement's step"""
    f = getattr(reference.lib, "mifi_get_values_linear_f", None)
    if f is None:
        pytest.skip("mifi_get_values_linear_f not in the reference")
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_double, C.c_double, C.c_double]
    rng = np.random.default_rng(12)
    A = rng.normal(250, 30, 4096).astype(np.float32)
    B = rng.normal(250, 30, 4096).astype(np.float32)
    for a, b, x in ((0.0, 3.0, 1.0), (262968.0, 262974.0, 262969.0), (0.0, 3.0, -1.0), (0.0, 3.0, 3.0), (10.5, 11.0, 12.25)):
        ref = np.empty_like(A)
        f(A.ctypes.data, B.ctypes.data, ref.ctypes.data, A.size, a, b, x)
        np.testing.assert_array_equal(vo.vint_values(vo.LIN, A, B, a, b, x).view(np.uint32), ref.view(np.uint32))


def test_typed_restatement_goes_through_the_adapters(oracle):
    """int16 with a fill value: the fill enters as NaN and leaves as the fill; values are rounded half away from zero"""
    a = np.array([10, -32767, 11, 0], np.int16)
    b = np.array([20, 5, -32767, 1], np.int16)
    got = to.step(oracle, [0.0, 4.0], 1.0, 0, a, b, -32767.0, np.int16)
    assert got.tolist() == [13, -32767, -32767, 0]  # 12.5 rounds away from zero


# ---------------------------------------------------------------------------------------------- the C ABI and the Python layer
def test_time_interpolation_symbols_are_declared_and_exported():
    names = ("fb200_tinterp_create", "fb200_tinterp_destroy", "fb200_tinterp_source_steps", "fb200_tinterp_get_step",
             "fb200_tinterp_get_step_device", "fb200_tinterp_get_data_slice_device")
    assert all(n in capi.declared_symbols() and hasattr(capi.load(), n) for n in names)
    assert "TimeInterpolator" in fimex_b200.__all__


def _create(times=(0.0, 3.0, 6.0), new_times=(1.0, 2.0), nt=None, nj=None, handle=True):
    """fb200_tinterp_create with one argument changed from a valid call"""
    t, n = (None if v is None else np.asarray(v, dtype=np.float64) for v in (times, new_times))
    h = C.c_void_p()
    return capi.load().fb200_tinterp_create(capi.ptr(t), len(times) if nt is None else nt, capi.ptr(n),
                                            len(new_times) if nj is None else nj, 1, C.byref(h) if handle else None)


@pytest.mark.parametrize("kwargs, message", [
    (dict(times=(0.0,)), "number of source times must be at least 2"),
    (dict(nt=-1), "number of source times must be at least 2"),
    (dict(new_times=(), nj=0), "number of target times must be in [1, 1048576]"),
    (dict(new_times=np.zeros(1048577)), "number of target times must be in [1, 1048576]"),
    (dict(times=None, nt=3), "null time axis"),
    (dict(new_times=None, nj=2), "null time axis"),
    (dict(times=(0.0, np.nan, 6.0)), "times must be finite"),
    (dict(new_times=(1.0, np.inf)), "times must be finite"),
    (dict(times=(0.0, 3.0, 3.0)), "strictly increasing"),
    (dict(times=(6.0, 3.0, 0.0)), "strictly increasing"),
    (dict(handle=False), "null handle pointer"),
])
def test_argument_checks_of_the_c_abi(quiet, kwargs, message):
    assert _create(**kwargs) == fimex_b200.MIFI_ERROR
    assert message in fimex_b200.last_error()


@pytest.mark.parametrize("kwargs, error", [
    (dict(), "either new_times or time_spec"),
    (dict(new_times=[1.0], time_spec="0,1;unit=hours"), "either new_times or time_spec"),
    (dict(new_times=[1.0], unit="hours"), "is not '<seconds|minutes|hours|days> since"),
    (dict(new_times=[1.0], calendar="360_day"), "calendar '360_day' is not supported"),
    (dict(time_spec="0,3,...,12"), "needs ';unit='"),
])
def test_argument_checks_of_the_python_layer(quiet, kwargs, error):
    args = dict(times=[0.0, 3.0, 6.0], unit=HOURS)
    args.update(kwargs)
    with pytest.raises(fimex_b200.FimexB200Error, match=error.replace("(", r"\(").replace("|", r"\|").replace("[", r"\[")):
        TimeInterpolator(**args)


def test_no_cpu_fallback_without_gpu(quiet):
    if _has_gpu():
        pytest.skip("a GPU is present; the refusal path cannot be exercised")
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        TimeInterpolator([0.0, 3.0, 6.0], HOURS, new_times=np.arange(7.0))
    with pytest.raises(fimex_b200.FimexB200Error, match="no usable CUDA device"):
        TimeInterpolator([0.0, 3.0, 6.0], HOURS, time_spec="0,1,...,x;unit=hours")
    assert _create() == fimex_b200.MIFI_ERROR and "no usable CUDA device" in fimex_b200.last_error()
    lib = capi.load()
    a = np.ones(4, np.float32)
    out = np.empty(4, np.float32)
    ia, ib, w = C.c_int(), C.c_int(), C.c_double()
    # a handle never exists without a device: the calls refuse the null handle before anything else
    assert lib.fb200_tinterp_source_steps(None, 0, C.byref(ia), C.byref(ib), C.byref(w)) == fimex_b200.MIFI_ERROR
    assert "null time interpolation handle" in fimex_b200.last_error()
    assert lib.fb200_tinterp_get_step(None, 0, 4, capi.ptr(a), capi.ptr(a), 4, np.nan, 4, capi.ptr(out)) == fimex_b200.MIFI_ERROR
    assert "null time interpolation handle" in fimex_b200.last_error()
    assert lib.fb200_tinterp_get_step_device(None, 0, 4, capi.ptr(a), capi.ptr(a), 4, np.nan, 4, capi.ptr(out), None) == fimex_b200.MIFI_ERROR
    assert "null time interpolation handle" in fimex_b200.last_error()
    assert lib.fb200_tinterp_get_data_slice_device(None, 4, capi.ptr(a), 4, np.nan, 4, capi.ptr(out), None) == fimex_b200.MIFI_ERROR
    assert "null time interpolation handle" in fimex_b200.last_error()
    lib.fb200_tinterp_destroy(None)  # no-op
