"""Time interpolation on the GPU against the restatement (tests/time_interp_oracle.py), bit for bit with identical NaN masks: every
in/out type pair of (1c) with fill values on the host, device and stack entry points; NaN, +-inf and +-0 inputs; n = 1, 3 and unaligned
pointers (the scalar path); J = 70 000; a stack beyond 2^32 elements; concurrent calls on one handle; a seeded fuzz; and a device
chain time -> horizontal -> vertical interpolation to pressure levels."""
import os
import threading

import numpy as np
import pytest

import time_interp_oracle as to
import vertical_oracle as vo

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200.timeinterp import TimeInterpolator  # noqa: E402
from fimex_b200.vertical import HYBRID, VerticalInterpolator  # noqa: E402

HOURS = "hours since 1970-01-01 00:00:00"
SEEDS = int(os.environ.get("FIMEX_B200_TFUZZ_SEEDS", "40"))
DTYPES = [np.int8, np.int16, np.int32, np.float32, np.float64, np.uint8, np.uint16, np.uint32, np.int64, np.uint64]
ERA5_LEVELS = np.array([1, 2, 3, 5, 7, 10, 20, 30, 50, 70, 100, 125, 150, 175, 200, 225, 250, 300, 350, 400, 450, 500, 550, 600, 650, 700,
                        750, 775, 800, 825, 850, 875, 900, 925, 950, 975, 1000], dtype=np.float64)


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
        differ = got.view(np.uint8).reshape(got.size, -1) != want.view(np.uint8).reshape(want.size, -1)
        differ = differ.any(axis=-1) if got.size else differ
    bad = np.flatnonzero(differ)
    assert bad.size == 0, f"{what}: {bad.size} of {got.size} differ, first at {bad[0]}: {got.ravel()[bad[0]]} vs {want.ravel()[bad[0]]}"


def _fits(v, dtype):
    dt = np.dtype(dtype)
    if np.isnan(v):
        return dt.kind == "f"
    return dt.kind == "f" or np.iinfo(dt).min <= v <= np.iinfo(dt).max


def _fill(in_dtype, out_dtype=None):
    """the input type's default fill value where both types hold it (static_cast of an out-of-range fill is undefined), else 127"""
    f = fb.default_fill_value(in_dtype)
    return f if _fits(f, in_dtype) and _fits(f, out_dtype or in_dtype) else 127.0


def _data(rng, shape, dtype, fill, fill_share=0.05):
    """values in [0, 60] (every type holds them and every blend below stays inside int8 after rounding), with fill values"""
    dt = np.dtype(dtype)
    v = rng.uniform(0, 60, shape)
    v = v.astype(dt) if dt.kind == "f" else np.round(v).astype(dt)
    v[rng.random(shape) < fill_share] = dt.type(fill)
    return v


def _targets(rng, times, nj, outside=True):
    """targets in any order with repeats, exact hits on source times and (outside) up to 0.9 of a step beyond each end: the blends of
    values in [0, 60] stay in [-54, 114]"""
    t0, t1 = times[0], times[-1]
    d0, d1 = (times[1] - t0) * 0.9, (t1 - times[-2]) * 0.9
    taus = rng.uniform(t0 - d0 if outside else t0, t1 + d1 if outside else t1, nj)
    hits = rng.random(nj) < 0.25
    taus[hits] = rng.choice(times, int(hits.sum()))
    if nj > 3:
        taus[1] = taus[0]
    return taus


def _times(rng, nt):
    return 262968.0 + np.cumsum(rng.choice([1.0, 3.0, 6.0], nt)) - 1.0


def _torch(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _check_all_paths(oracle, ti, data, bad, out_dtype, what, host_steps=True):
    """the stack call, every step on the device and (host_steps) every step from host buffers, against the restatement"""
    want = to.stack(oracle, ti.source_times, ti.times, data, bad, out_dtype, extrapolate=ti.extrapolate)
    d = _torch(data)
    got = ti.get_data_slice(d, bad_value=bad, out_dtype=_torch_dtype(out_dtype)).cpu().numpy()
    _same(got, want, f"{what} stack")
    for j in range(ti.times.size):
        ia, ib, w = ti.source_steps(j)
        a, b = data[max(ia, 0)], data[max(ia, 0) + 1]
        got = ti.get_data_slice_step(j, d[max(ia, 0)], d[max(ia, 0) + 1], bad_value=bad, out_dtype=_torch_dtype(out_dtype)).cpu().numpy()
        _same(got, want[j], f"{what} device step {j}")
        if host_steps:
            _same(ti.get_data_slice_step(j, a, b, bad_value=bad, out_dtype=out_dtype), want[j], f"{what} host step {j}")


def _torch_dtype(dtype):
    import torch
    return getattr(torch, np.dtype(dtype).name)


def _make(times, taus, extrapolate=True):
    return TimeInterpolator(times, HOURS, new_times=taus, extrapolate=extrapolate)


# ---------------------------------------------------------------------------------------------- types and entry points
def test_source_steps_match_the_restatement():
    rng = np.random.default_rng(1)
    times = _times(rng, 9)
    taus = _targets(rng, times, 200)
    for extrapolate in (True, False):
        ti = _make(times, taus, extrapolate)
        ia, ib, w = to.time_map(times, taus, extrapolate)
        got = np.array([ti.source_steps(j) for j in range(taus.size)])
        assert got[:, 0].tolist() == ia.tolist() and got[:, 1].tolist() == ib.tolist()
        assert got[:, 2].tobytes() == w.tobytes()
    ti = TimeInterpolator([0.0, 3.0, 6.0], HOURS, time_spec="0,1,...,x;unit=hours")
    assert [ti.source_steps(j)[:2] for j in range(7)] == [(0, 1)] * 4 + [(1, 2)] * 3
    with pytest.raises(fb.FimexB200Error, match="out of range"):
        ti.source_steps(7)


@pytest.mark.parametrize("in_dtype", DTYPES, ids=lambda d: np.dtype(d).name)
def test_every_type_pair_with_fill_values(oracle, in_dtype):
    rng = np.random.default_rng(np.dtype(in_dtype).num)
    times = _times(rng, 5)
    ti = _make(times, _targets(rng, times, 9))
    for out_dtype in DTYPES:
        bad = _fill(in_dtype, out_dtype)
        data = _data(rng, (5, 2, 517), in_dtype, bad)
        host = np.dtype(out_dtype) in (np.dtype(np.float32), np.dtype(np.int16), np.dtype(in_dtype))
        what = f"{np.dtype(in_dtype).name}->{np.dtype(out_dtype).name}"
        _check_all_paths(oracle, ti, data, bad, out_dtype, what, host_steps=host)
        got = ti.get_data_slice(_torch(data), bad_value=bad, out_dtype=_torch_dtype(out_dtype)).cpu().numpy()
        assert (got == np.dtype(out_dtype).type(bad)).any()  # the fill value came through both adapters
        if np.dtype(out_dtype).kind == "f":  # a NaN fill value switches the input pass off: the fill values in the data are values
            want = to.stack(oracle, times, ti.times, data, float("nan"), out_dtype)
            got = ti.get_data_slice(_torch(data), bad_value=float("nan"), out_dtype=_torch_dtype(out_dtype)).cpu().numpy()
            _same(got, want, f"{what} no fill value")


def test_without_extrapolation_the_rows_outside_are_fill(oracle):
    rng = np.random.default_rng(2)
    times = _times(rng, 4)
    taus = np.array([times[0] - 1, times[1], times[-1] + 1, times[2] + 0.5, times[0] - 2])
    ti = _make(times, taus, extrapolate=False)
    data = _data(rng, (4, 1001), np.int16, -32767.0)
    _check_all_paths(oracle, ti, data, -32767.0, np.int16, "no extrapolation")
    got = ti.get_data_slice(_torch(data), bad_value=-32767.0).cpu().numpy()
    assert (got[[0, 2, 4]] == -32767).all()
    # a target without a bracket reads no source step: the C ABI takes NULL slices for it
    import ctypes as C
    out = np.empty(1001, np.int16)
    lib = fb.load()
    assert lib.fb200_tinterp_get_step(ti._h, 0, 2, None, None, out.size, -32767.0, 2, out.ctypes.data_as(C.c_void_p)) == fb.MIFI_OK
    assert (out == -32767).all()
    assert lib.fb200_tinterp_get_step(ti._h, 1, 2, None, None, out.size, -32767.0, 2, out.ctypes.data_as(C.c_void_p)) == fb.MIFI_ERROR
    assert "null data pointer" in fb.last_error()


def test_nan_inf_and_signed_zeros(oracle):
    """NaN and +-inf propagate through the blend (also into an exact hit through its other step); A = -0 with w = 0 gives -0 or +0 by the
    sign of B - A before the store, whose '+ 0' makes both +0 on every typed output (restatement and kernel alike)"""
    times = np.array([0.0, 3.0, 6.0])
    taus = np.array([0.0, 1.0, 3.0, 6.0, 7.5, -1.0])
    specials = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -1.0, 3e38, -3e38], np.float32)
    a, b, c = np.meshgrid(specials, specials, specials, indexing="ij")
    data = np.stack([a.ravel(), b.ravel(), c.ravel()])
    ti = _make(times, taus)
    for out_dtype in (np.float32, np.float64):
        _check_all_paths(oracle, ti, data, float("nan"), out_dtype, f"specials -> {np.dtype(out_dtype).name}")
    f = vo.vint_values(vo.LIN, np.array([-0.0, -0.0], np.float32), np.array([-1.0, 1.0], np.float32), 0.0, 3.0, 0.0)
    assert np.signbit(f).tolist() == [True, False]
    got = ti.get_data_slice(_torch(np.array([[-0.0, -0.0], [-1.0, 1.0], [0.0, 0.0]], np.float32)), bad_value=float("nan")).cpu().numpy()
    assert not np.signbit(got[0]).any()


@pytest.mark.parametrize("n", [1, 3, 4, 5, 1027])
def test_small_and_odd_n_and_unaligned_pointers(oracle, n):
    import torch
    rng = np.random.default_rng(n)
    times = _times(rng, 6)
    ti = _make(times, _targets(rng, times, 11))
    for dtype in (np.float32, np.int16, np.uint8, np.float64):
        data = _data(rng, (6, n), dtype, _fill(dtype))
        _check_all_paths(oracle, ti, data, _fill(dtype), dtype, f"n={n} {np.dtype(dtype).name}")
        # every pointer one element off the four-element alignment
        buf = torch.zeros(6 * n + 1, dtype=_torch_dtype(dtype), device="cuda")
        buf[1:] = _torch(data.ravel())
        stack = buf[1:].view(6, n)
        out = torch.zeros(ti.times.size * n + 1, dtype=_torch_dtype(dtype), device="cuda")
        lib = fb.load()
        tcode = int(fb.cdm_type(dtype))
        assert lib.fb200_tinterp_get_data_slice_device(ti._h, tcode, fb.capi.ptr(stack), n, _fill(dtype), tcode, fb.capi.ptr(out[1:]),
                                                       None) == fb.MIFI_OK
        want = to.stack(oracle, times, ti.times, data, _fill(dtype), dtype)
        _same(out[1:].cpu().numpy().reshape(want.shape), want, f"n={n} unaligned {np.dtype(dtype).name}")
        assert out[0].item() == 0
        got = ti.get_data_slice_step(3, stack[ti.source_steps(3)[0]], stack[ti.source_steps(3)[1]], bad_value=_fill(dtype)).cpu().numpy()
        _same(got, want[3], f"n={n} unaligned step")


def test_aligned_n_with_unaligned_output(oracle):
    import torch
    rng = np.random.default_rng(4)
    times = _times(rng, 3)
    ti = _make(times, _targets(rng, times, 5))
    data = _data(rng, (3, 4096), np.float32, _fill(np.float32))
    out = torch.zeros(5 * 4096 + 2, dtype=torch.float32, device="cuda")
    assert fb.load().fb200_tinterp_get_data_slice_device(ti._h, 4, fb.capi.ptr(_torch(data)), 4096, np.nan, 4, fb.capi.ptr(out[2:]),
                                                         None) == fb.MIFI_OK
    _same(out[2:].cpu().numpy().reshape(5, 4096), to.stack(oracle, times, ti.times, data, np.nan, np.float32), "unaligned output")


# ---------------------------------------------------------------------------------------------- sizes
@pytest.mark.parametrize("in_dtype, out_dtype", [(np.float32, np.float32), (np.int16, np.int16), (np.uint8, np.float64), (np.float64, np.int8)],
                         ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("extrapolate", [True, False])
@pytest.mark.parametrize("odd", [False, True], ids=["vector", "scalar"])
def test_one_segment_walks_every_target(oracle, in_dtype, out_dtype, extrapolate, odd):
    """n large enough that the sorted targets are not split over gridDim.y: one thread walks all of them, through repeated brackets,
    moves up by one (the old B becomes the new A), jumps over source steps, and (without extrapolation) on to targets without a
    bracket.  The odd n takes the scalar path."""
    import torch
    n = torch.cuda.get_device_properties(0).multi_processor_count * 8 * 1024 + (3 if odd else 0)
    times = np.array([0.0, 3.0, 6.0, 9.0, 12.0, 15.0, 18.0]) + 262968.0
    offs = [1.0, 2.0, 2.0, 3.0, 4.0, 5.0, 6.0, 10.0, 17.0, 18.0, -1.5, 19.5, 0.0, 13.0]  # unsorted; two outside the range
    taus = times[0] + np.array(offs)
    ti = _make(times, taus, extrapolate)
    ia, _, _ = to.time_map(times, taus, extrapolate)
    assert (ia < 0).sum() == (0 if extrapolate else 2)
    rng = np.random.default_rng(7)
    bad = _fill(in_dtype, out_dtype)
    data = _data(rng, (times.size, n), in_dtype, bad, fill_share=0.01)
    got = ti.get_data_slice(_torch(data), bad_value=bad, out_dtype=_torch_dtype(out_dtype)).cpu().numpy()
    _same(got, to.stack(oracle, times, taus, data, bad, out_dtype, extrapolate), f"one segment, n = {n}")


def test_70000_targets(oracle):
    rng = np.random.default_rng(7)
    times = _times(rng, 50)
    taus = _targets(rng, times, 70_000)
    ti = _make(times, taus)
    data = _data(rng, (50, 5), np.float32, _fill(np.float32))
    got = ti.get_data_slice(_torch(data), bad_value=_fill(np.float32)).cpu().numpy()
    # the restatement, vectorised over the targets: float in and out, so the adapters are the identity but for fill <-> NaN
    ia, ib, w = to.time_map(times, taus)
    A = oracle.as_float(data, _fill(np.float32))
    want = np.empty((taus.size, 5), np.float32)
    for j in range(taus.size):
        want[j] = vo.vint_values(vo.LIN, A[ia[j]], A[ib[j]], times[ia[j]], times[ib[j]], taus[j])
    _same(got, oracle.from_float(want, _fill(np.float32), np.float32), "J = 70 000")
    for j in (0, 12_345, 69_999):
        ia_j, ib_j, _ = ti.source_steps(j)
        _same(ti.get_data_slice_step(j, data[ia_j], data[ib_j], bad_value=_fill(np.float32)), got[j], f"J = 70 000 step {j}")


def test_stack_beyond_2_pow_32_elements(oracle):
    """int8 [3][2^31 + 8]: the last step starts beyond 2^32 elements; sampled windows against the restatement"""
    import torch
    n = (1 << 31) + 8
    times = np.array([0.0, 3.0, 6.0])
    taus = np.array([5.0, 1.0, 7.0])
    ti = _make(times, taus)
    g = torch.Generator(device="cuda").manual_seed(5)
    stack = torch.randint(-20, 60, (3, n), dtype=torch.int8, device="cuda", generator=g)
    stack[:, ::97] = -127
    out = ti.get_data_slice(stack, bad_value=-127.0)
    torch.cuda.synchronize()
    for lo in (0, (1 << 31) - 4096, n - 65536):
        win = stack[:, lo:lo + 65536].cpu().numpy()
        want = to.stack(oracle, times, taus, win, -127.0, np.int8)
        _same(out[:, lo:lo + 65536].cpu().numpy(), want, f"window at {lo}")
    del stack, out
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- concurrency and the fuzz
def test_concurrent_calls_on_one_handle(oracle):
    import torch
    rng = np.random.default_rng(9)
    times = _times(rng, 8)
    ti = _make(times, _targets(rng, times, 24))
    data = _data(rng, (8, 64, 333), np.int16, -32767.0)
    want = to.stack(oracle, times, ti.times, data, -32767.0, np.int16)
    d = _torch(data)
    torch.cuda.synchronize()  # the threads' streams do not order after the upload
    errors = []

    def work(k):
        try:
            fb.set_device(0)
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for rep in range(3):
                    got = ti.get_data_slice(d, bad_value=-32767.0, stream=s)
                    s.synchronize()
                    _same(got.cpu().numpy(), want, f"thread {k} stack")
                    j = (k * 7 + rep) % ti.times.size
                    ia, ib, _ = ti.source_steps(j)
                    _same(ti.get_data_slice_step(j, data[ia], data[ib], bad_value=-32767.0), want[j], f"thread {k} host step {j}")
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=work, args=(k,)) for k in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[0]


@pytest.mark.parametrize("seed", range(SEEDS))
def test_fuzz(oracle, seed):
    rng = np.random.default_rng(1000 + seed)
    nt = int(rng.integers(2, 12))
    times = _times(rng, nt)
    extrapolate = bool(rng.integers(0, 2))
    taus = _targets(rng, times, int(rng.integers(1, 30)))
    ti = _make(times, taus, extrapolate)
    in_dtype, out_dtype = DTYPES[int(rng.integers(0, 10))], DTYPES[int(rng.integers(0, 10))]
    shape = (nt,) + tuple(int(x) for x in rng.integers(1, 40, int(rng.integers(1, 3))))
    bad = _fill(in_dtype, out_dtype)
    data = _data(rng, shape, in_dtype, bad, fill_share=float(rng.uniform(0, 0.2)))
    if np.dtype(out_dtype).kind == "f" and rng.random() < 0.2:
        bad = float("nan")  # no input pass; a NaN fill value is only cast to floating outputs
    _check_all_paths(oracle, ti, data, bad, out_dtype, f"seed {seed}", host_steps=seed % 4 == 0)


# ---------------------------------------------------------------------------------------------- a device chain
def test_chain_time_then_horizontal_then_pressure_levels(oracle):
    """3-hourly model-level temperature and surface pressure to hourly steps, through the horizontal bilinear get_data_slice_device over
    all J x nz levels, then the vertical linear interpolation to the 37 ERA5 levels, all on the device; against the three restatements"""
    import torch
    import vertical_convert_oracle as vc
    import vertical_reference as vr
    rng = np.random.default_rng(43)
    nt, nk = 3, 30
    inX, inY, outX, outY = 97, 61, 83, 45
    px = rng.uniform(-0.5, inX - 0.5, outX * outY)
    py = rng.uniform(-0.5, inY - 0.5, outX * outY)
    ci = fb.CachedInterpolation("x", "y", fb.Method.BILINEAR, px, py, inX, inY, outX, outY)
    ap, b = vr._hybrid_table(nk, rng)
    terms = {"ap": ap, "b": b}
    times = np.array([0.0, 3.0, 6.0]) + 262968.0
    ti = TimeInterpolator(times, HOURS, time_spec="0,1,...,x;unit=hours")
    J = ti.times.size
    T = rng.uniform(200, 300, (nt, nk, inY, inX)).astype(np.float32)
    T[rng.random(T.shape) < 0.01] = np.nan
    ps = rng.uniform(900, 1040, (nt, inY, inX)).astype(np.float32)
    nan = float("nan")
    t_T = ti.get_data_slice(_torch(T), bad_value=nan)
    t_ps = ti.get_data_slice(_torch(ps), bad_value=nan)
    h_T = ci.getDataSlice(t_T.reshape(J * nk, inY, inX), nan).reshape(J, nk, outY * outX).contiguous()
    h_ps = ci.getDataSlice(t_ps.reshape(J, inY, inX), nan).reshape(J, outY * outX).contiguous()
    got = VerticalInterpolator(HYBRID, terms, "linear", ERA5_LEVELS).getDataSlice(h_T, ps=h_ps, bad_value=nan).cpu().numpy()
    o_T = to.stack(oracle, times, ti.times, T, nan, np.float32)
    o_ps = to.stack(oracle, times, ti.times, ps, nan, np.float32)
    o_hT = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, o_T.reshape(-1, inY, inX)).reshape(J, nk, -1)
    o_hps = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, o_ps.reshape(-1, inY, inX)).reshape(J, -1)
    want = vc.vinterp_pressure(0, vc.VCOORD_HYBRID, ap, b, ERA5_LEVELS, o_hT, ps=o_hps)
    _same(got.reshape(want.shape), want, "time -> horizontal -> vertical")
    assert J == 7 and np.isfinite(want).mean() > 0.5
