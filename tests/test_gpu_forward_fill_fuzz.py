"""A seeded differential fuzz of forward interpolation and of the fill processes on the GPU, and their edges.

Forward (K8, CachedForwardInterpolation): each case of tests/forward_reference.py's generator (one of the ten methods, source and
target sizes, nz, points uniform / clustered into a few cells / over every edge, x.5 ties, NaN and huge positions, 0 / 1 / 30 % NaN
values with several payloads, repeats and both signs of zero) runs through the host and the device path and is compared bit for bit
with the C restatement and with the independent reference.  ``FIMEX_B200_FFUZZ_SEEDS`` sets the number of seeds (default 60).
NaN payloads are compared for the medians, whose result is a copied input value; sum and mean compute their NaN (the GPU returns
0x7fffffff) and max / min may select theirs with a min/max instruction, so there only the NaN masks are compared.
Edges: the level loop past one launch (nz up to 300; 130 for the medians), 1, 3, 2^12 and 2^12 + 1 cells, an output that is not
16-byte aligned, no point mapped, every point in one cell, typed getDataSlice for every method, the chunked host pipeline, and the
two buckets where std::nth_element differs from a sort and from rank selection.

Fill (fill2d, creepfill2d, creepfillval2d): a seeded fuzz of about 40 cases (``FIMEX_B200_FILLFUZZ_SEEDS``) over shapes in both
orientations, 1-5 levels, hole patterns and parameters, through the device and the host-pointer forms, bit for bit against the
restatement including the changed counts; every case again with the simple kernel forced.  Fixed shapes sit on both sides of each
kernel switch (min(nx, ny) = 799 | 800 and 1599 | 1600), on skewed<16> in both orientations, at config 2's 2000 x 2000 target and
at 30 x 700 / 700 x 30."""
import ctypes as C
import os

import numpy as np
import pytest

import forward_reference as fr

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import Method  # noqa: E402

FWD_SEEDS = int(os.environ.get("FIMEX_B200_FFUZZ_SEEDS", "60"))
FILL_SEEDS = int(os.environ.get("FIMEX_B200_FILLFUZZ_SEEDS", "40"))
ALL = [Method(m) for m in fr.METHODS]


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _gpu_equal(got, want, method, what):
    fr.assert_forward_equal(got, want, int(method), what, nan_payload=int(method) in fr.MEDIANS)


def _forward_all_paths(oracle, method, px, py, inX, inY, outX, outY, data, what, reference=True):
    """host and device path against the restatement (and the independent reference); returns the restatement's result"""
    want = oracle.forward_interpolate(int(method), px, py, inX, inY, outX, outY, data)
    if reference:
        fr.assert_forward_equal(want, fr.forward(int(method), px, py, outX, outY, data), int(method), f"{what}: restatement vs reference")
    cfi = fb.CachedForwardInterpolation("x", "y", method, px, py, inX, inY, outX, outY)
    _gpu_equal(cfi.interpolateValues(data), want, method, f"{what}: host path")
    _gpu_equal(cfi.interpolateValues(_cuda(data)).cpu().numpy(), want, method, f"{what}: device path")
    return want


# ================================================================================================================ forward: the fuzz
@pytest.mark.parametrize("seed", range(FWD_SEEDS))
def test_forward_fuzz(oracle, seed):
    c = fr.make_case(100_000 + seed)
    _forward_all_paths(oracle, Method(c["method"]), c["px"], c["py"], c["inX"], c["inY"], c["outX"], c["outY"], c["data"],
                       f"seed {seed}")


# ================================================================================================================ forward: the edges
def _dense_case(rng, nz, inX=40, inY=20, outX=13, outY=11):
    px = rng.uniform(-0.6, outX - 0.4, inX * inY)
    py = rng.uniform(-0.6, outY - 0.4, inX * inY)
    data = rng.normal(0, 3, (nz, inY, inX)).astype(np.float32)
    data[rng.random(data.shape) < 0.05] = np.nan
    data[rng.random(data.shape) < 0.05] = -0.0
    data[rng.random(data.shape) < 0.05] = 0.0
    return px, py, data


@pytest.mark.parametrize("method", [Method.FORWARD_SUM, Method.FORWARD_MEAN, Method.FORWARD_MAX, Method.FORWARD_MIN, Method.FORWARD_UNDEF_SUM,
                                    Method.FORWARD_UNDEF_MEAN, Method.FORWARD_UNDEF_MAX, Method.FORWARD_UNDEF_MIN])
@pytest.mark.parametrize("nz", [1, 2, 3, 4, 5, 255, 256, 257, 300])
def test_forward_level_counts(oracle, method, nz):
    """ZL = 1 for nz < 4, four levels per pass and a tail otherwise; gridDim.y = 64 passes cover 256 levels, 257 and 300 loop"""
    px, py, data = _dense_case(np.random.default_rng(nz * 31 + int(method)), nz)
    _forward_all_paths(oracle, method, px, py, 40, 20, 13, 11, data, f"nz {nz}", reference=nz <= 5)


@pytest.mark.parametrize("method", [Method.FORWARD_MEDIAN, Method.FORWARD_UNDEF_MEDIAN])
@pytest.mark.parametrize("nz", [1, 64, 65, 130])
def test_forward_median_level_counts(oracle, method, nz):
    """the median goes level by level: gridDim.y = 64 covers 64 levels, 65 and 130 loop through the same scratch slots"""
    px, py, data = _dense_case(np.random.default_rng(nz * 37 + int(method)), nz)
    _forward_all_paths(oracle, method, px, py, 40, 20, 13, 11, data, f"nz {nz}", reference=nz <= 65)


@pytest.mark.parametrize("outX,outY", [(1, 1), (3, 1), (64, 64), (4097, 1)])
def test_forward_cell_counts(oracle, outX, outY):
    """1 and 3 cells (one partial thread), 2^12 (a power of two: the radix sort's end_bit) and 2^12 + 1 (a partial last thread)"""
    rng = np.random.default_rng(outX * 7 + outY)
    inX, inY = 97, 43
    px = rng.uniform(-1.0, outX, inX * inY)
    py = rng.uniform(-1.0, outY, inX * inY)
    data = rng.normal(0, 3, (5, inY, inX)).astype(np.float32)
    data[rng.random(data.shape) < 0.1] = np.nan
    data[rng.random(data.shape) < 0.05] = -0.0
    for method in ALL:
        _forward_all_paths(oracle, method, px, py, inX, inY, outX, outY, data, f"{outX} x {outY} cells", reference=outX * outY < 4096)


def test_forward_unaligned_output(oracle):
    """out = buf[1:]: 4 bytes past a 16-byte boundary with n_cells % 4 == 0, so only the alignment turns the vector store off"""
    import torch
    rng = np.random.default_rng(5)
    inX, inY, outX, outY = 60, 30, 16, 9
    px, py, data = _dense_case(rng, 6, inX, inY, outX, outY)
    for method in ALL:
        want = oracle.forward_interpolate(int(method), px, py, inX, inY, outX, outY, data)
        cfi = fb.CachedForwardInterpolation("x", "y", method, px, py, inX, inY, outX, outY)
        buf = torch.full((outX * outY * 6 + 1,), 7.0, device="cuda")
        assert (buf[1:].data_ptr() & 15) == 4
        got = cfi.interpolateValues(_cuda(data), out=buf[1:])
        _gpu_equal(got.cpu().numpy(), want, method, "unaligned output")
        assert buf[0].item() == 7.0


def test_forward_nothing_mapped(oracle):
    rng = np.random.default_rng(6)
    px = np.full(300, -5.0)
    py = rng.uniform(0, 4, 300)
    data = rng.normal(0, 1, (3, 10, 30)).astype(np.float32)
    for method in ALL:
        want = _forward_all_paths(oracle, method, px, py, 30, 10, 5, 4, data, "nothing mapped")
        assert np.isnan(want).all()


@pytest.mark.parametrize("values", ["normal", "nan_and_zeros"])
def test_forward_every_point_in_one_cell(oracle, values):
    """~5000 points in one segment: the sums run 5000 steps, the median's rank selection 5000^2 compares or, with NaN or both
    signs of zero, the introselect on the cell's scratch copy"""
    rng = np.random.default_rng(7)
    inX, inY, outX, outY = 100, 50, 3, 2
    px = rng.uniform(0.6, 1.4, inX * inY)  # all in cell (1, 0)
    py = rng.uniform(-0.4, 0.4, inX * inY)
    data = rng.normal(0, 3, (2, inY, inX)).astype(np.float32)
    if values == "nan_and_zeros":
        data[rng.random(data.shape) < 0.2] = np.nan
        data[rng.random(data.shape) < 0.2] = -0.0
        data[rng.random(data.shape) < 0.2] = 0.0
    for method in ALL:
        want = _forward_all_paths(oracle, method, px, py, inX, inY, outX, outY, data, f"one cell, {values}")
        assert np.isnan(want[:, 0, 0]).all() and np.isnan(want[:, 1, :]).all()


def test_forward_median_known_answers(oracle):
    """std::nth_element selects NaN from {NaN, 3, 1, 2} (forward_undef_median) and +0 from {-0, +0, +0, -0, 1}; a sort selects 2,
    and rank selection with the first equal element in input order 3 and -0"""
    for method, vals in ((Method.FORWARD_UNDEF_MEDIAN, [np.nan, 3, 1, 2]), (Method.FORWARD_MEDIAN, [-0.0, 0.0, 0.0, -0.0, 1.0])):
        v = np.array(vals, dtype=np.float32)[None]
        px = np.zeros(v.size)
        want = _forward_all_paths(oracle, method, px, px, v.size, 1, 2, 1, v, "known answer")
        if method == Method.FORWARD_UNDEF_MEDIAN:
            assert np.isnan(want[0, 0, 0])
        else:
            assert want[0, 0, 0].view(np.uint32) == 0


@pytest.mark.parametrize("method", ALL)
@pytest.mark.parametrize("dtype", [np.int16, np.float64])
def test_forward_typed_get_data_slice(oracle, method, dtype):
    """fill -> NaN, aggregate, NaN -> fill + round + cast, host and device, for every forward method"""
    rng = np.random.default_rng(int(method) * 3 + np.dtype(dtype).itemsize)
    inX, inY, inZ, outX, outY = 60, 40, 5, 37, 21
    fill = -32767.0 if dtype == np.int16 else fb.default_fill_value(np.float64)
    px = rng.uniform(-1, outX, inX * inY)
    py = rng.uniform(-1, outY, inX * inY)
    if dtype == np.int16:
        data = rng.integers(-3000, 3000, (inZ, inY, inX)).astype(np.int16)
    else:
        data = rng.normal(0, 100, (inZ, inY, inX))
        data[rng.random(data.shape) < 0.05] = -0.0
    data[rng.random(data.shape) < 0.05] = dtype(fill)
    want = oracle.from_float(oracle.forward_interpolate(int(method), px, py, inX, inY, outX, outY, oracle.as_float(data, fill)), fill,
                             dtype).reshape(inZ, outY, outX)
    cfi = fb.CachedForwardInterpolation("x", "y", method, px, py, inX, inY, outX, outY)
    for got in (cfi.getDataSlice(data, fill), cfi.getDataSlice(_cuda(data), fill).cpu().numpy()):
        assert got.dtype == np.dtype(dtype)
        bits = np.uint16 if dtype == np.int16 else np.uint64
        assert np.array_equal(got.view(bits), want.view(bits))
    assert (want == dtype(fill)).any()


def _pinned(a, keep):
    """a copy of `a` in page-locked memory from fb200_host_alloc (freed by the caller through `keep`)"""
    p = fb.load().fb200_host_alloc(a.nbytes)
    assert p
    keep.append(p)
    out = np.frombuffer((C.c_char * a.nbytes).from_address(p), dtype=a.dtype).reshape(a.shape)
    out[...] = a
    return out


@pytest.mark.parametrize("memory", ["pinned", "pageable"])
def test_forward_host_pipeline_in_chunks(oracle, monkeypatch, memory):
    """1 MB chunks of 20 levels of 12 000 points (+ 600 cells), the last one partial; 9.6 MB per call, so pageable arrays go
    through the bounce buffers"""
    monkeypatch.setenv("FIMEX_B200_HOST_CHUNK_MB", "1")
    rng = np.random.default_rng(8 if memory == "pinned" else 9)
    inX, inY, nz, outX, outY = 120, 100, 203, 30, 20
    px, py, data = _dense_case(rng, nz, inX, inY, outX, outY)
    keep = []
    try:
        if memory == "pinned":
            data = _pinned(data, keep)
        for method in (Method.FORWARD_MEAN, Method.FORWARD_UNDEF_MEDIAN, Method.FORWARD_MAX):
            want = oracle.forward_interpolate(int(method), px, py, inX, inY, outX, outY, data)
            cfi = fb.CachedForwardInterpolation("x", "y", method, px, py, inX, inY, outX, outY)
            _gpu_equal(cfi.interpolateValues(data), want, method, f"{memory} chunks")
    finally:
        for p in keep:
            fb.load().fb200_host_free(p)


# ==================================================================================================================== fill: the fuzz
def _fill_field(rng, nz, ny, nx, pattern):
    yy, xx = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    f = (280 + 10 * np.sin(xx / 7.0) * np.cos(yy / 5.0) + rng.normal(0, 0.5, (nz, ny, nx))).astype(np.float32)
    if pattern.startswith("random"):
        f[rng.random(f.shape) < float(pattern.split(":")[1])] = np.nan
    elif pattern == "big_hole":
        y0, x0 = rng.integers(0, ny), rng.integers(0, nx)
        f[:, y0:y0 + max(1, ny // 2), x0:x0 + max(1, nx // 2)] = np.nan
    elif pattern == "borders":
        f[:, 0, :] = np.nan
        f[:, :, -1] = np.nan
        f[:, -1, : nx // 2] = np.nan
        f[:, : ny // 2, 0] = np.nan
        f[:, 0, 0] = f[:, -1, -1] = np.nan
    elif pattern == "one_defined":
        keep = f[:, ny // 3, nx // 2].copy()
        f[:] = np.nan
        f[:, ny // 3, nx // 2] = keep
    else:  # "one_undefined"
        f[:, rng.integers(0, ny), rng.integers(0, nx)] = np.nan
    return f


def _fill_case(seed):
    rng = np.random.default_rng(50_000 + seed)
    a = int(rng.choice([2, 3, 4, 5, 9, 17, 33, 64, 100, 150, 257]))
    b = int(rng.choice([2, 3, 5, 31, 77, 130, 300, 600]))
    nx, ny = (a, b) if rng.random() < 0.5 else (b, a)
    if rng.random() < 0.2:
        ny = nx
    nz = int(rng.integers(1, 6))
    pattern = str(rng.choice(["random:0.001", "random:0.1", "random:0.6", "big_hole", "borders", "one_defined", "one_undefined"]))
    f = _fill_field(rng, nz, ny, nx, pattern)
    fill_args = (np.float32(10 ** rng.uniform(-6, 0)), np.float32(rng.uniform(0.5, 2.0)), int(rng.choice([0, 1, 3, 4, 5, 9, 10, 11, 100])))
    repeat = int(rng.integers(0, 31))
    weight = int(rng.choice([1, 2, 3, 4, 5, 200]))  # 200: the char -56
    default = None if rng.random() < 0.5 else float(rng.normal(0, 10))
    return f, fill_args, repeat, weight, default, pattern


def _check_fill(oracle, f, fill_args, repeat, weight, default, what):
    want, counts = oracle.fill2d(f, *fill_args)
    dev = fb.fill2d_device(_cuda(f), *fill_args).cpu().numpy()
    assert np.array_equal(dev.view(np.uint32), want.view(np.uint32)), ("fill2d", what, fill_args)
    rc, one, n = fb.mifi_fill2d_f(f[-1], *fill_args)  # the reference's own host-pointer prototype
    assert rc == fb.MIFI_OK and n == counts[-1] and np.array_equal(one.view(np.uint32), want[-1].view(np.uint32)), ("mifi_fill2d_f", what)
    want, counts = oracle.creepfill2d(f, repeat, weight, default)
    dev = fb.creepfill2d_device(_cuda(f), repeat, weight, default).cpu().numpy()
    assert np.array_equal(dev.view(np.uint32), want.view(np.uint32)), ("creepfill2d", what, repeat, weight, default)
    rc, one, n = fb.mifi_creepfill2d_f(f[-1], repeat, weight, default)
    assert rc == fb.MIFI_OK and n == counts[-1] and np.array_equal(one.view(np.uint32), want[-1].view(np.uint32)), ("mifi_creepfill", what)


@pytest.mark.parametrize("simple", [False, True], ids=["chosen_kernel", "simple_kernel"])
@pytest.mark.parametrize("seed", range(FILL_SEEDS))
def test_fill_fuzz(oracle, monkeypatch, seed, simple):
    if simple:
        monkeypatch.setenv("FIMEX_B200_FILL_SIMPLE", "1")
    f, fill_args, repeat, weight, default, pattern = _fill_case(seed)
    _check_fill(oracle, f, fill_args, repeat, weight, default, f"seed {seed}: {f.shape} {pattern}")


def test_fill_generator_covers_the_edges():
    cases = [_fill_case(s) for s in range(FILL_SEEDS)]
    assert {c[5] for c in cases} >= {"random:0.6", "big_hole", "borders", "one_defined", "one_undefined"}
    assert any(c[0].shape[1] > c[0].shape[2] > 3 for c in cases) and any(c[0].shape[2] > c[0].shape[1] for c in cases)
    assert any(c[3] == 200 for c in cases) and {c[1][2] for c in cases} >= {0, 1, 100}


# ============================================================================================================= fill: the kernel switches
@pytest.mark.parametrize("nx,ny", [(799, 799), (800, 800), (1599, 1600), (1600, 1599), (1000, 1000), (1200, 900), (900, 1200),
                                   (2000, 2000), (30, 700), (700, 30)])
def test_fill_kernel_switches(oracle, nx, ny):
    """skewed<32> up to min(nx, ny) = 799, skewed<16> from 800 to 1599, the simple kernel from 1600 (config 2's 2000 x 2000
    target); by_y = 0 (ny > nx) at 30 x 700"""
    rng = np.random.default_rng(nx * 3 + ny)
    f = _fill_field(rng, 1, ny, nx, "random:0.1")
    f[0, ny // 4: ny // 4 + ny // 5, nx // 3: nx // 3 + nx // 6] = np.nan
    f[0, 0, :] = np.nan
    f[0, :, -1] = np.nan
    _check_fill(oracle, f, (np.float32(0.01), np.float32(1.6), 100), 20, 2, None, f"{nx} x {ny}")
    if min(nx, ny) >= 800:  # the other two process forms, once each
        want, _ = oracle.creepfill2d(f, 5, 200, -3.5)
        dev = fb.creepfill2d_device(_cuda(f), 5, 200, -3.5).cpu().numpy()
        assert np.array_equal(dev.view(np.uint32), want.view(np.uint32))


def test_get_data_slice_with_fill_processes_1000x1000(oracle):
    """a 1000 x 1000 x 4 target (skewed<16>): creepfill2d as preprocess on the source, fill2d as postprocess on the target,
    against the oracle chain"""
    from test_gpu_parity import _smooth_positions, _typed_field
    inX, inY, inZ, outX, outY = 300, 250, 4, 1000, 1000
    px, py = _smooth_positions(inX, inY, outX, outY, 17.0, 2.8, 3)  # part of the target hangs over the source grid
    rng = np.random.default_rng(10)
    fill = -32767.0
    data = _typed_field(rng, (inZ, inY, inX), np.int16, fill)
    data[:, 40:90, 60:140] = -32767
    ci = fb.CachedInterpolation("x", "y", Method.BILINEAR, px, py, inX, inY, outX, outY)
    ci.addPreprocess("creepfill2d(3,2)")
    ci.addPostprocess("fill2d(0.01,1.6,100)")
    got = ci.getDataSlice(data, fill)
    a = oracle.as_float(data, fill)
    a, _ = oracle.creepfill2d(a, 3, ord("2"))
    o = oracle.cached_interpolate(1, px, py, inX, inY, outX, outY, a)
    assert np.isnan(o).any()
    o, _ = oracle.fill2d(o.reshape(inZ, outY, outX), np.float32(0.01), np.float32(1.6), 100)
    want = oracle.from_float(o, fill, np.int16).reshape(got.shape)
    assert np.array_equal(got, want)
    assert not (got == -32767).any()
