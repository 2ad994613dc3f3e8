"""The vertical interpolator's data conversions (theta2T, omega2vwind, add4Dpressure) on the GPU against the restatement
(orc_vconvert, tests/vertical_convert_oracle.c), bit for bit with identical NaN masks: every op x source coordinate on the host, device
and in-place entry points, NaN in ps, theta, omega and T; concurrent calls on one handle; nt = 70 000, a step beyond 2^32 elements,
nk = 1 and 1024; the host pipeline in chunks on pinned and pageable arrays; a seeded fuzz against the independent reference's bound;
one whole ERA5-size step; and two device chains horizontal -> conversion -> vertical interpolation."""
import ctypes as C
import gc
import os
import threading
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal
import vertical_convert_oracle as vc
import vertical_convert_reference as vcr
import vertical_reference as vr

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import capi  # noqa: E402
from fimex_b200.vertical import HYBRID, PRESSURE, SIGMA, PressureConversion, VerticalInterpolator, _Columns  # noqa: E402

OPS = list(vc.OPS)
NAMES = {PRESSURE: vc.VCOORD_PRESSURE, HYBRID: vc.VCOORD_HYBRID, SIGMA: vc.VCOORD_SIGMA}
SEEDS = int(os.environ.get("FIMEX_B200_VCONV_SEEDS", "40"))
ERA5_LEVELS = np.array([1, 2, 3, 5, 7, 10, 20, 30, 50, 70, 100, 125, 150, 175, 200, 225, 250, 300, 350, 400, 450, 500, 550, 600, 650, 700,
                        750, 775, 800, 825, 850, 875, 900, 925, 950, 975, 1000], dtype=np.float64)


def _source(name, nk, rng):
    """(terms, a, b, ptop) of a monotone column of nk levels"""
    if name == PRESSURE:
        p = np.sort(rng.uniform(1, 1100, nk))
        return {"p": p}, p, None, 0.0
    if name == HYBRID:
        ap, b = vr._hybrid_table(max(nk, 2), rng)
        ap, b = ap[:nk].copy(), b[:nk].copy()
        return {"ap": ap, "b": b}, ap, b, 0.0
    sigma, ptop = np.sort(rng.uniform(0.01, 1.0, nk)), float(rng.uniform(0, 50))
    return {"sigma": sigma, "ptop": ptop}, None, sigma, ptop


def _inputs(op, name, nt, nk, nxy, rng, nan_share=0.01, pa=False):
    """(field, ps, t) float32, seeded, with a share of NaN in each; None where the op or coordinate reads nothing"""
    shape = (nt, nk, nxy)
    field = t = ps = None
    if op == "theta2T":
        field = rng.uniform(180, 1500, shape).astype(np.float32)
    elif op == "omega2vwind":
        field = rng.normal(0, 1.5, shape).astype(np.float32)
        t = rng.uniform(180, 320, shape).astype(np.float32)
    if name != PRESSURE:
        ps = (rng.uniform(480, 1060, (nt, nxy)) * (100.0 if pa else 1.0)).astype(np.float32)
    for a in (field, t, ps):
        if a is not None and nan_share:
            a[rng.random(a.shape) < nan_share] = np.nan
    return field, ps, t


def _oracle(op, name, a, b, nk, field, ps, t, ptop, ps_scale=1.0, nt=None, nxy=None):
    return vc.vconvert(vc.OPS[op], NAMES[name], a, b, nk, field=field, ps=ps, t=t, ptop=ptop, ps_scale=ps_scale, nt=nt, nxy=nxy)


def _cuda(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _in_place(pc, d_field, d_ps, d_t, nxy, nt):
    """fb200_vconvert_values_device with d_out == d_in"""
    cols = _Columns()
    cols.ps = capi.ptr(d_ps).value if d_ps is not None else None
    cols.t = capi.ptr(d_t).value if d_t is not None else None
    capi.check(fb.load().fb200_vconvert_values_device(pc._h, capi.ptr(d_field), C.byref(cols), nxy, nt, capi.ptr(d_field), None), "in place")
    import torch
    torch.cuda.synchronize()
    return d_field


@pytest.mark.parametrize("pa", [False, True], ids=["hPa", "Pa"])
@pytest.mark.parametrize("name", list(NAMES))
@pytest.mark.parametrize("op", OPS)
def test_bit_identical_to_restatement(oracle, op, name, pa):
    """host, device and in-place entry points; NaN in ps and in every input field"""
    rng = np.random.default_rng(zlib.crc32(repr((op, name, pa)).encode()))
    nt, nk, nxy = 3, 37, 517
    terms, a, b, ptop = _source(name, nk, rng)
    field, ps, t = _inputs(op, name, nt, nk, nxy, rng, pa=pa)
    s = 0.01 if pa else 1.0
    want = _oracle(op, name, a, b, nk, field, ps, t, ptop, s, nt=nt, nxy=nxy)
    pc = PressureConversion(name, terms, op, ps_scale=s)
    what = f"{op} {name} {'Pa' if pa else 'hPa'}"
    host = pc.convert(field, ps=ps, t=t, nt=nt if field is None and ps is None else None)
    if op == "add4Dpressure" and name == PRESSURE:  # no field and no ps: [nt][nk], one value per level and step
        assert host.shape == (nt, nk)
        assert_bit_equal(host, want[:, :, 0], what + " host")
        return
    assert_bit_equal(host.reshape(want.shape), want, what + " host")
    dev = pc.convert(_cuda(field), ps=_cuda(ps), t=_cuda(t)).cpu().numpy()
    assert_bit_equal(dev.reshape(want.shape), want, what + " device")
    if field is not None:
        d = _in_place(pc, _cuda(field), _cuda(ps), _cuda(t), nxy, nt).cpu().numpy()
        assert_bit_equal(d, want, what + " in place")
    assert 0.8 < np.isfinite(want).mean() < 1.0, what  # values and NaN both exercised


def test_nan_propagation_is_per_value_and_per_column(oracle):
    """a NaN ps makes its whole column and step NaN; a NaN theta, omega or T only its own value"""
    rng = np.random.default_rng(8)
    terms, a, b, ptop = _source(HYBRID, 20, rng)
    field, ps, t = _inputs("omega2vwind", HYBRID, 2, 20, 64, rng, nan_share=0.0)
    ps[1, 5] = np.nan
    field[0, 3, 7] = np.nan
    t[0, 4, 9] = np.nan
    got = PressureConversion(HYBRID, terms, "omega2vwind").convert(_cuda(field), ps=_cuda(ps), t=_cuda(t)).cpu().numpy()
    assert_bit_equal(got, _oracle("omega2vwind", HYBRID, a, b, 20, field, ps, t, ptop), "nan")
    mask = np.zeros(got.shape, bool)
    mask[1, :, 5] = mask[0, 3, 7] = mask[0, 4, 9] = True
    assert np.array_equal(np.isnan(got), mask)


def test_concurrent_calls_on_one_handle(oracle):
    rng = np.random.default_rng(21)
    terms, a, b, ptop = _source(SIGMA, 40, rng)
    pc = PressureConversion(SIGMA, terms, "theta2T")
    cases = [_inputs("theta2T", SIGMA, 3, 40, 2053 + 7 * i, np.random.default_rng(100 + i)) for i in range(6)]
    results = [None] * len(cases)

    def work(i):
        field, ps, t = cases[i]
        for _ in range(3):
            results[i] = pc.convert(field, ps=ps)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for i, (field, ps, t) in enumerate(cases):
        assert_bit_equal(results[i], _oracle("theta2T", SIGMA, a, b, 40, field, ps, None, ptop), f"thread {i}")


# ------------------------------------------------------------------------------------------------------------------------- edges
@pytest.mark.parametrize("op", OPS)
def test_more_steps_than_one_launch_takes(oracle, op):
    """nt = 70 000 > 65 535, the limit of gridDim.y: device and host entry points"""
    rng = np.random.default_rng(zlib.crc32(op.encode()))
    nt, nk, nxy = 70_000, 3, 33
    terms, a, b, ptop = _source(HYBRID, nk, rng)
    field, ps, t = _inputs(op, HYBRID, nt, nk, nxy, rng, nan_share=0.0)
    want = _oracle(op, HYBRID, a, b, nk, field, ps, t, ptop)
    pc = PressureConversion(HYBRID, terms, op)
    assert_bit_equal(pc.convert(_cuda(field), ps=_cuda(ps), t=_cuda(t)).cpu().numpy(), want, f"{op} nt=70000 device")
    assert_bit_equal(pc.convert(field, ps=ps, t=t), want, f"{op} nt=70000 host")


def test_last_step_beyond_two_to_the_32_elements(oracle):
    """theta2T in place on [65][64][2^20 + 3]: the last step starts beyond 2^32 elements (17.4 GB)"""
    import torch
    nt, nk, nxy = 65, 64, (1 << 20) + 3
    assert (nt - 1) * nk * nxy > 2 ** 32
    rng = np.random.default_rng(32)
    terms, a, b, ptop = _source(HYBRID, nk, rng)
    g = torch.Generator(device="cuda").manual_seed(5)
    field = torch.rand((nt, nk, nxy), device="cuda", generator=g).mul_(1300).add_(200)
    ps = torch.rand((nt, nxy), device="cuda", generator=g).mul_(560).add_(480)
    first, last = field[0:1].cpu().numpy(), field[nt - 1:nt].cpu().numpy()
    pc = PressureConversion(HYBRID, terms, "theta2T")
    _in_place(pc, field, ps, None, nxy, nt)
    for step, before in ((0, first), (nt - 1, last)):
        want = _oracle("theta2T", HYBRID, a, b, nk, before, ps[step:step + 1].cpu().numpy(), None, ptop)
        assert_bit_equal(field[step:step + 1].cpu().numpy(), want, f"step {step} of {nt}")
    del field, ps
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("nk", [1, 1024])
@pytest.mark.parametrize("name", list(NAMES))
def test_one_and_1024_levels(oracle, name, nk):
    rng = np.random.default_rng(nk + len(name))
    terms, a, b, ptop = _source(name, nk, rng)
    for op in ("theta2T", "omega2vwind"):
        field, ps, t = _inputs(op, name, 2, nk, 129, rng)
        pc = PressureConversion(name, terms, op)
        want = _oracle(op, name, a, b, nk, field, ps, t, ptop)
        assert_bit_equal(pc.convert(field, ps=ps, t=t), want, f"{op} {name} nk={nk} host")
        assert_bit_equal(pc.convert(_cuda(field), ps=_cuda(ps), t=_cuda(t)).cpu().numpy(), want, f"{op} {name} nk={nk} device")


def test_1025_levels_are_refused():
    with pytest.raises(fb.FimexB200Error, match=r"number of levels must be in \[1, 1024\]"):
        PressureConversion(PRESSURE, {"p": np.linspace(1, 1000, 1025)}, "add4Dpressure")
    h = C.c_void_p()
    p = np.linspace(1, 1000, 1025)
    assert fb.load().fb200_vconvert_create(2, 0, capi.ptr(p), None, 1025, 0.0, 1.0, C.byref(h)) == fb.MIFI_ERROR


def test_calls_refuse_missing_inputs():
    rng = np.random.default_rng(9)
    terms, a, b, ptop = _source(HYBRID, 5, rng)
    field, ps, t = _inputs("omega2vwind", HYBRID, 1, 5, 10, rng)
    pc = PressureConversion(HYBRID, terms, "omega2vwind")
    with pytest.raises(fb.FimexB200Error, match="air temperature t"):
        pc.convert(field, ps=ps)
    with pytest.raises(fb.FimexB200Error, match="surface pressure ps"):
        pc.convert(field, t=t)
    with pytest.raises(fb.FimexB200Error, match="float32 CUDA tensor"):
        pc.convert(_cuda(field), ps=_cuda(ps).double(), t=_cuda(t))
    with pytest.raises(fb.FimexB200Error, match="float32 CUDA tensor"):
        pc.convert(_cuda(field), ps=ps, t=_cuda(t))
    lib = fb.load()
    out = np.empty_like(field)
    cols = _Columns()
    cols.ps = capi.ptr(ps).value
    assert lib.fb200_vconvert_values(pc._h, capi.ptr(field), C.byref(cols), 10, 1, capi.ptr(out)) == fb.MIFI_ERROR
    assert "omega2vwind needs the air temperature t" in fb.last_error()


def _pinned(a, keep):
    lib = fb.load()
    p = lib.fb200_host_alloc(a.nbytes)
    assert p
    keep.append(p)
    out = np.frombuffer((C.c_char * a.nbytes).from_address(p), dtype=a.dtype).reshape(a.shape)
    out[...] = a
    return out


@pytest.mark.parametrize("memory", ["pinned", "pageable"])
@pytest.mark.parametrize("op", ["omega2vwind", "add4Dpressure", "theta2T"])
def test_host_pipeline_in_chunks(oracle, monkeypatch, op, memory):
    """1 MB chunks, the last one partial; more than 8 MB per call, so pageable arrays go through the bounce buffers"""
    monkeypatch.setenv("FIMEX_B200_HOST_CHUNK_MB", "1")
    rng = np.random.default_rng(zlib.crc32((op + memory).encode()))
    nt, nk, nxy = {"omega2vwind": 37, "add4Dpressure": 61, "theta2T": 43}[op], 20, 1031
    terms, a, b, ptop = _source(SIGMA, nk, rng)
    field, ps, t = _inputs(op, SIGMA, nt, nk, nxy, rng)
    want = _oracle(op, SIGMA, a, b, nk, field, ps, t, ptop)
    keep = []
    try:
        if memory == "pinned":
            field, ps, t = (None if x is None else _pinned(x, keep) for x in (field, ps, t))
        got = PressureConversion(SIGMA, terms, op).convert(field, ps=ps, t=t)
        assert_bit_equal(got, want, f"{op} {memory}")
        assert np.isfinite(want).mean() > 0.9
    finally:
        for p in keep:
            fb.load().fb200_host_free(p)


def contraction_cases(n=8):
    """(ap, b, ps, omega, T) with hybrid p_k = ap + b ps for which an FMA-contracted p_k (one rounding instead of two) moves w across
    a float32 rounding boundary: a search over ap, one fp64 step at a time, near the p that puts w on a float32 midpoint"""
    from fractions import Fraction
    H = 8.31432 / (0.0289644 * 9.80665)
    rng = np.random.default_rng(77)
    found = []
    while len(found) < n:
        omega, T, ps = float(np.float32(rng.normal(0, 2))), float(np.float32(rng.uniform(200, 300))), float(np.float32(rng.uniform(500, 1000)))
        b = float(rng.uniform(0.1, 0.9))
        w0 = -(omega * (H * T)) / (100.0 * 500.0)
        lo = float(np.float32(w0))
        mid = 0.5 * (lo + float(np.nextafter(np.float32(lo), np.float32(np.inf))))
        pstar = -(omega * (H * T)) / (100.0 * mid)
        a = pstar - b * ps
        for step in range(-64, 65):
            ap = a + step * float(np.spacing(np.abs(pstar)))
            p_two = ap + b * ps
            p_fma = float(Fraction(ap) + Fraction(b) * Fraction(ps))
            if p_two == p_fma:
                continue
            w_two = -(omega * (H * T)) / (100.0 * p_two)
            w_fma = -(omega * (H * T)) / (100.0 * p_fma)
            if np.float32(w_two) != np.float32(w_fma):
                found.append((ap, b, ps, omega, T))
                break
    return found


def test_omega2vwind_pressure_is_not_contracted(oracle):
    """columns for which an FMA-contracted p_k = ap + b ps gives another float32 w: the kernel gives the restatement's uncontracted
    value, host and device"""
    for ap, b, ps, omega, T in contraction_cases():
        pc = PressureConversion(HYBRID, {"ap": [ap], "b": [b]}, "omega2vwind")
        f, p, t = (np.full(s, v, np.float32) for s, v in (((2, 1, 33), omega), ((2, 33), ps), ((2, 1, 33), T)))
        want = _oracle("omega2vwind", HYBRID, [ap], [b], 1, f, p, t, 0.0)
        assert_bit_equal(pc.convert(f, ps=p, t=t), want, "contraction host")
        assert_bit_equal(pc.convert(_cuda(f), ps=_cuda(p), t=_cuda(t)).cpu().numpy(), want, "contraction device")


# --------------------------------------------------------------------------------------------------- the independent reference
@pytest.mark.parametrize("seed", range(SEEDS))
def test_fuzz_against_the_reference(oracle, seed):
    case = vcr.draw_case(10_000 + seed)
    op = list(vc.OPS)[case.op]
    name = list(NAMES)[case.kind]
    terms = {PRESSURE: lambda: {"p": case.a}, HYBRID: lambda: {"ap": case.a, "b": case.b},
             SIGMA: lambda: {"sigma": case.b, "ptop": case.ptop}}[name]()
    nt = None if case.field is not None or case.ps is not None else 2
    pc = PressureConversion(name, terms, op, ps_scale=case.ps_scale)
    host = pc.convert(case.field, ps=case.ps, t=case.t, nt=nt)
    want = vc.vconvert(case.op, case.kind, case.a, case.b, case.nk, field=case.field, ps=case.ps, t=case.t, nt=nt, nxy=1, **case.args())
    assert_bit_equal(host.reshape(want.shape), want, f"seed {seed} host")
    if nt is None:
        dev = pc.convert(_cuda(case.field), ps=_cuda(case.ps), t=_cuda(case.t)).cpu().numpy()
        assert_bit_equal(dev.reshape(want.shape), want, f"seed {seed} device")
    ref = vcr.reference(case.op, case.kind, case.a, case.b, case.nk, field=case.field, ps=case.ps, t=case.t, nt=nt, nxy=1, **case.args())
    assert vcr.check(host, ref, f"seed {seed}") <= 1.0


# ------------------------------------------------------------------------------------------------------------ whole step, chains
def test_era5_step_memcmp_equal(oracle):
    """one whole step of profiles/tools/vertical_convert_time.py's workload: 1440 x 721 columns, 137 hybrid levels, theta2T, host
    buffers"""
    rng = np.random.default_rng(20261021)
    ap, b = vr._hybrid_table(137, rng)
    nxy = 1440 * 721
    ps = rng.uniform(480, 1040, (1, nxy)).astype(np.float32)
    field = rng.uniform(180, 1500, (1, 137, nxy)).astype(np.float32)
    got = PressureConversion(HYBRID, {"ap": ap, "b": b}, "theta2T").convert(field.reshape(1, 137, 721, 1440), ps=ps.reshape(1, 721, 1440))
    want = vc.vconvert(vc.THETA2T, vc.VCOORD_HYBRID, ap, b, 137, field=field, ps=ps)
    assert got.shape == (1, 137, 721, 1440)
    assert got.tobytes() == want.tobytes()


def _horizontal(rng):
    inX, inY, outX, outY = 97, 61, 83, 45
    px = rng.uniform(-0.5, inX - 0.5, outX * outY)
    py = rng.uniform(-0.5, inY - 0.5, outX * outY)
    return fb.CachedInterpolation("x", "y", fb.Method.BILINEAR, px, py, inX, inY, outX, outY), (px, py, inX, inY, outX, outY)


def test_chain_theta_to_t_in_place_then_log_to_pressure_levels(oracle):
    """theta and ps through the horizontal bilinear get_data_slice_device, theta2T in place, then the vertical log to the 37 ERA5
    levels, all on the device; against the same chain of restatements"""
    import torch
    rng = np.random.default_rng(41)
    nt, nk = 2, 60
    ci, geo = _horizontal(rng)
    px, py, inX, inY, outX, outY = geo
    terms, ap, b, ptop = _source(HYBRID, nk, rng)
    theta, ps, _ = _inputs("theta2T", HYBRID, nt, nk, inX * inY, rng)
    nan = float("nan")
    h_theta = ci.getDataSlice(torch.from_numpy(theta.reshape(nt * nk, inY, inX)).cuda(), nan).reshape(nt, nk, outY * outX).contiguous()
    h_ps = ci.getDataSlice(torch.from_numpy(ps.reshape(nt, inY, inX)).cuda(), nan).reshape(nt, outY * outX).contiguous()
    _in_place(PressureConversion(HYBRID, terms, "theta2T"), h_theta, h_ps, None, outX * outY, nt)
    vi = VerticalInterpolator(HYBRID, terms, "log", ERA5_LEVELS)
    got = vi.getDataSlice(h_theta, ps=h_ps, bad_value=nan).cpu().numpy()
    o_theta = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, theta.reshape(-1, inY, inX)).reshape(nt, nk, -1)
    o_ps = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, ps.reshape(-1, inY, inX)).reshape(nt, -1)
    T = vc.vconvert(vc.THETA2T, vc.VCOORD_HYBRID, ap, b, nk, field=o_theta, ps=o_ps)
    want = vc.vinterp_pressure(1, vc.VCOORD_HYBRID, ap, b, ERA5_LEVELS, T, ps=o_ps)
    assert_bit_equal(got.reshape(want.shape), want, "theta chain")
    assert np.isfinite(want).mean() > 0.5


def test_chain_omega_to_w_then_linear(oracle):
    """omega, T and ps through the horizontal call, omega2vwind on the device, then the vertical linear to the 37 ERA5 levels"""
    import torch
    rng = np.random.default_rng(42)
    nt, nk = 2, 60
    ci, geo = _horizontal(rng)
    px, py, inX, inY, outX, outY = geo
    terms, ap, b, ptop = _source(HYBRID, nk, rng)
    omega, ps, t = _inputs("omega2vwind", HYBRID, nt, nk, inX * inY, rng)
    nan = float("nan")

    def horiz(x, lead):
        return ci.getDataSlice(torch.from_numpy(x.reshape(-1, inY, inX)).cuda(), nan).reshape(*lead, outY * outX).contiguous()

    h_omega, h_t, h_ps = horiz(omega, (nt, nk)), horiz(t, (nt, nk)), horiz(ps, (nt,))
    w = PressureConversion(HYBRID, terms, "omega2vwind").convert(h_omega, ps=h_ps, t=h_t)
    got = VerticalInterpolator(HYBRID, terms, "linear", ERA5_LEVELS).getDataSlice(w, ps=h_ps, bad_value=nan).cpu().numpy()

    def orc(x):
        return oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, x.reshape(-1, inY, inX))

    o_ps = orc(ps).reshape(nt, -1)
    W = vc.vconvert(vc.OMEGA2VWIND, vc.VCOORD_HYBRID, ap, b, nk, field=orc(omega).reshape(nt, nk, -1), ps=o_ps, t=orc(t).reshape(nt, nk, -1))
    want = vc.vinterp_pressure(0, vc.VCOORD_HYBRID, ap, b, ERA5_LEVELS, W, ps=o_ps)
    assert_bit_equal(got.reshape(want.shape), want, "omega chain")
    assert np.isfinite(want).mean() > 0.5
