"""BASELINE.json configs 2, 3(i), 3(ii) and 4: the WHOLE output field of one time step (137 levels; 5.48e8 values for the
2000 x 2000 grids, 2 x 1.23e9 for config 4) compared bit for bit with the reference's own CPU kernels -- oracle/_ref =
src/interpolation.c compiled unmodified, inside the restated CachedInterpolation.cc:118-147 loop -- on identical inputs:
the same field and the same fp64 position tables (the GPU's, downloaded).  The position tables themselves are compared
with the CPU pipeline (project_axes -> points2position -> createReducedDomain) over the whole grid, with the count of
index flips bounded by the number of positions within 4e-9 cells (1e-9 degree on the 0.25-degree axes) of a cell or half-cell
boundary.

Where oracle/_ref is not built (it needs the reference's sources, which the repository does not hold), the same comparison
runs against the restatement (oracle/liboracle.so), which tests/test_oracle_golden.py pins to vectors the reference computed.

Levels are compared in chunks so the host never holds more than one chunk of the reference's output.
"""
import os
import time

import numpy as np
import pytest

from conftest import ROOT  # noqa: F401

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import Method  # noqa: E402

SRC_LL = "+proj=latlong +a=6371000 +e=0 +no_defs"
ROTPOLE = "+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +R=6.371e+06 +no_defs"
STERE = "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0"
WGS84 = "+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs"
LON = np.arange(1440) * 0.25
LAT = 90 - np.arange(721) * 0.25
AX2 = (np.arange(2000) - 999.5) * 0.0225
NZ = 137


@pytest.fixture(scope="module")
def cpu_kernels(oracle):
    """the reference's own kernels where oracle/_ref is built, else the restatement: the same Python surface"""
    from oracle import oracle as orc
    return orc.Reference() if orc.Reference.available() else oracle


def _cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _bilinear_ub_count(oracle, px, py, inX, inY):
    """size of the set where the reference itself reads out of bounds (src/interpolation.c:936, SURVEY.md 8a trap 4):
    x in an outer half cell and y within half a cell of row iy.  Candidates by numpy, confirmed one by one."""
    cand = np.flatnonzero(((np.floor(px) < 0) | (np.floor(px) + 1 >= inX)) & (py >= inY - 1.0))
    return sum(1 for i in cand if oracle.bilinear_is_ub(px[i], py[i], inX, inY))


def _compare_levels(cpu_kernels, method, gx, gy, inX, inY, outX, outY, d_in, d_out, nan_payload, chunk=16, post=None):
    """d_in: list of device tensors [nz][inY][inX] (one per field), d_out: matching list [nz][outY][outX].  Returns the number
    of differing values over the whole stack.  post(list of host arrays) -> list of host arrays (e.g. the rotation)."""
    import torch
    nz = d_in[0].shape[0]
    differing, compared = 0, 0
    for z0 in range(0, nz, chunk):
        z1 = min(nz, z0 + chunk)
        want = [cpu_kernels.cached_interpolate(int(method), gx, gy, inX, inY, outX, outY, f[z0:z1].cpu().numpy(), nthreads=_cores()) for f in d_in]
        if post is not None:
            want = post(want, z1 - z0)
        for w, out in zip(want, d_out):
            w = torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).cuda().view(z1 - z0, outY, outX)
            got = out[z0:z1]
            diff = got.view(torch.int32) != w.view(torch.int32)
            if not nan_payload:  # arithmetic NaNs: x86 propagates the operand's payload, the GPU emits the canonical one
                diff &= ~(torch.isnan(got) & torch.isnan(w))
            differing += int(diff.sum().item())
            compared += got.numel()
    return differing, compared


def _cpu_positions(oracle, proj, ax, xdeg):
    rc, x, y = oracle.project_axes(proj, SRC_LL, np.radians(ax) if xdeg else ax, np.radians(ax) if xdeg else ax)
    assert rc == 1
    px = oracle.points2position(x, np.radians(LON), 1)
    py = oracle.points2position(y, np.radians(LAT), 2)
    return oracle.reduced_domain(px, py, 1440, 721)


def _field(inX, inY, seed, nan_frac=0.01):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo = torch.linspace(0, 6.28, inX, device="cuda")[None, None, :]
    la = torch.linspace(0, 1.0, inY, device="cuda")[None, :, None]
    z = torch.arange(NZ, device="cuda", dtype=torch.float32)[:, None, None]
    f = 250 + 30 * torch.sin(la) * torch.cos(2 * lo) + 0.1 * z + 0.5 * torch.randn((NZ, inY, inX), generator=g, device="cuda")
    if nan_frac:
        f[torch.rand(f.shape, generator=g, device="cuda") < nan_frac] = float("nan")
    return f.contiguous()


@pytest.mark.parametrize("method", [Method.BILINEAR, Method.NEAREST_NEIGHBOR], ids=["config2-bilinear", "config3i-nearestneighbor"])
def test_full_field_rotated_pole(oracle, cpu_kernels, method):
    """configs 2 and 3(i): every one of the 137 x 2000 x 2000 output values equals the reference's, bit for bit (NaN payload
    included for nearest neighbour); the index tables equal the CPU pipeline's except at positions within 1e-9 degree of a
    (half-)cell boundary"""
    t0 = time.perf_counter()
    ci = fb.CachedInterpolation.fromProjection(method, ROTPOLE, AX2, AX2, True, True, SRC_LL, LON, LAT, True)
    assert ci.createReducedDomain()
    inX, inY = ci.getInX(), ci.getInY()
    gx, gy = ci.points()
    # ---- tables vs the CPU pipeline, whole grid ----
    red, ox, oy, oinX, oinY, x0, y0 = _cpu_positions(oracle, ROTPOLE, AX2, True)
    assert red and (oinX, oinY) == (inX, inY) and (x0, y0) == tuple(ci.reducedDomain()[2:4])
    assert np.abs(gx - ox).max() <= 4e-9 and np.abs(gy - oy).max() <= 4e-9  # 1e-9 degree on a 0.25-degree axis
    if method == Method.NEAREST_NEIGHBOR:
        lr = lambda v: np.where(v >= 0, np.floor(v + 0.5), np.ceil(v - 0.5))  # lround
        flips = int(((lr(gx) != lr(ox)) | (lr(gy) != lr(oy))).sum())
        near = int(((np.abs(gx - np.floor(gx) - 0.5) < 4e-9) | (np.abs(gy - np.floor(gy) - 0.5) < 4e-9)).sum())
    else:
        flips = int(((np.floor(gx) != np.floor(ox)) | (np.floor(gy) != np.floor(oy))).sum())
        near = int(((np.abs(gx - np.round(gx)) < 4e-9) | (np.abs(gy - np.round(gy)) < 4e-9)).sum())
    assert flips <= near, (flips, near)
    if method == Method.BILINEAR:
        assert _bilinear_ub_count(oracle, gx, gy, inX, inY) == 0  # nothing to mask on this grid
    # ---- values, whole field ----
    field = _field(inX, inY, 20261018)
    out = ci.interpolateValues(field)
    differing, compared = _compare_levels(cpu_kernels, method, gx, gy, inX, inY, 2000, 2000, [field], [out],
                                          nan_payload=(method == Method.NEAREST_NEIGHBOR))
    assert compared == NZ * 4_000_000
    assert differing == 0, f"{differing} of {compared} values differ from the reference"
    print(f"full field {method.name}: {compared} values identical, {flips} index flips / {near} near a boundary, {time.perf_counter() - t0:.1f} s")


def test_full_field_coord_nearestneighbor(oracle, cpu_kernels):
    """config 3(ii): coord_nearestneighbor over the uncropped 1440 x 721 source: whole field memcmp-equal to the reference's
    mifi_get_values_f on the GPU's index table; the table itself against the CPU search on 20000 sampled targets"""
    lon2d, lat2d = oracle.lonlat_to_matrix(np.radians(LON), np.radians(LAT))
    ci = fb.CachedInterpolation.fromCoordinates(Method.COORD_NN, ROTPOLE, AX2, AX2, True, True, np.degrees(lon2d), np.degrees(lat2d), 1440, 721)
    gx, gy = ci.points()
    rc, tx, ty = oracle.project_axes(ROTPOLE, WGS84, np.radians(AX2), np.radians(AX2))
    rng = np.random.default_rng(55)
    sample = rng.integers(0, 4_000_000, 20000)
    wx, wy, ties = oracle.coordnn(tx[sample], ty[sample], lon2d, lat2d, 1440, 721)
    differ = int(((gx[sample] != wx) | (gy[sample] != wy)).sum())
    assert differ <= max(3, ties), (differ, ties)
    field = _field(1440, 721, 33)
    out = ci.interpolateValues(field)
    differing, compared = _compare_levels(cpu_kernels, Method.COORD_NN, gx, gy, 1440, 721, 2000, 2000, [field], [out], nan_payload=True)
    assert compared == NZ * 4_000_000 and differing == 0, f"{differing} of {compared} values differ from the reference"


def test_full_field_bicubic_vector_polar_stereographic(oracle, cpu_kernels):
    """config 4: bicubic x_wind / y_wind, 137 levels, to the 3000 x 3000 polar-stereographic grid, rotated by
    CachedVectorReprojection: both whole output fields (2 x 1.23e9 values) equal the reference's mifi_get_values_bicubic_f +
    mifi_vector_reproject_values_by_matrix_f, bit for bit, NaN wedges included"""
    import torch
    ax = -3748750.0 + 2500.0 * np.arange(3000)
    ci = fb.CachedInterpolation.fromProjection(Method.BICUBIC, STERE, ax, ax, False, False, SRC_LL, LON, LAT, True)
    assert ci.createReducedDomain()
    cvr = fb.CachedVectorReprojection.fromProjection(fb.MIFI_VECTOR_KEEP_SIZE, SRC_LL, STERE, ax, ax, fb.PROJ_AXIS, fb.PROJ_AXIS)
    inX, inY = ci.getInX(), ci.getInY()
    gx, gy = ci.points()
    red, ox, oy, oinX, oinY, x0, y0 = _cpu_positions(oracle, STERE, ax, False)
    assert (oinX, oinY) == (inX, inY)
    assert np.abs(gx - ox).max() <= 4e-9 and np.abs(gy - oy).max() <= 4e-9
    matrix = cvr.getMatrix()
    g = torch.Generator(device="cuda").manual_seed(4)
    u = (torch.randn((NZ, inY, inX), generator=g, device="cuda") * 10).contiguous()
    v = (torch.randn((NZ, inY, inX), generator=g, device="cuda") * 10).contiguous()
    u[torch.rand(u.shape, generator=g, device="cuda") < 0.002] = float("nan")
    uo, vo = ci.interpolateVector(u, v, cvr)

    def rotate(want, nz):
        wu, wv = cpu_kernels.vector_reproject_by_matrix(matrix, want[0], want[1], 3000, 3000, nz)
        return [wu, wv]

    differing, compared = _compare_levels(cpu_kernels, Method.BICUBIC, gx, gy, inX, inY, 3000, 3000, [u, v], [uo, vo], nan_payload=False,
                                          chunk=8, post=rotate)
    assert compared == 2 * NZ * 9_000_000 and differing == 0, f"{differing} of {compared} values differ from the reference"


def test_full_field_bicubic_fp32_mode_error(cpu_kernels, monkeypatch):
    """config 4 in the opt-in fp32 arithmetic (FIMEX_B200_BICUBIC_FP32=1): the whole 137 x 3000 x 3000 field of each component
    against the reference: identical NaN masks, and max |error| <= 1e-5 x D, D = the largest |tap| of the point's own 4 x 4
    stencil (for the rotated pair: of both components) -- the denominator of north_star's "<= 1e-5 relative"."""
    import torch
    import torch.nn.functional as F
    ax = -3748750.0 + 2500.0 * np.arange(3000)
    ci = fb.CachedInterpolation.fromProjection(Method.BICUBIC, STERE, ax, ax, False, False, SRC_LL, LON, LAT, True)
    assert ci.createReducedDomain()
    cvr = fb.CachedVectorReprojection.fromProjection(fb.MIFI_VECTOR_KEEP_SIZE, SRC_LL, STERE, ax, ax, fb.PROJ_AXIS, fb.PROJ_AXIS)
    inX, inY = ci.getInX(), ci.getInY()
    gx, gy = ci.points()
    matrix = cvr.getMatrix()
    g = torch.Generator(device="cuda").manual_seed(44)
    u = (torch.randn((NZ, inY, inX), generator=g, device="cuda") * 10).contiguous()
    v = (torch.randn((NZ, inY, inX), generator=g, device="cuda") * 10 + 3).contiguous()
    monkeypatch.setenv("FIMEX_B200_BICUBIC_FP32", "1")
    uo, vo = ci.interpolateVector(u, v, cvr)
    monkeypatch.delenv("FIMEX_B200_BICUBIC_FP32")
    # D per target point and level: max over the stencil of max(|u|, |v|)
    x0 = torch.from_numpy(np.floor(gx).astype(np.int64) - 1).cuda()
    y0 = torch.from_numpy(np.floor(gy).astype(np.int64) - 1).cuda()
    valid = (x0 >= 0) & (x0 + 3 < inX) & (y0 >= 0) & (y0 + 3 < inY)
    flat = (y0.clamp(0, inY - 4) * (inX - 3) + x0.clamp(0, inX - 4))
    worst, chunk = 0.0, 8
    for z0 in range(0, NZ, chunk):
        z1 = min(NZ, z0 + chunk)
        nz = z1 - z0
        hu, hv = u[z0:z1].cpu().numpy(), v[z0:z1].cpu().numpy()
        wu = cpu_kernels.cached_interpolate(2, gx, gy, inX, inY, 3000, 3000, hu, nthreads=_cores())
        wv = cpu_kernels.cached_interpolate(2, gx, gy, inX, inY, 3000, 3000, hv, nthreads=_cores())
        wu, wv = cpu_kernels.vector_reproject_by_matrix(matrix, wu, wv, 3000, 3000, nz)
        amax = torch.maximum(u[z0:z1].abs(), v[z0:z1].abs())
        win = F.max_pool2d(amax[None], kernel_size=4, stride=1)[0].reshape(nz, -1)  # [nz][(inY-3)*(inX-3)]
        D = win[:, flat]  # [nz][9e6]
        for w, out in ((wu, uo), (wv, vo)):
            w = torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).cuda().view(nz, -1)
            got = out[z0:z1].reshape(nz, -1)
            assert torch.equal(torch.isnan(got), torch.isnan(w)), "NaN masks differ"
            assert torch.equal(torch.isnan(w[0]), ~valid)
            err = ((got.double() - w.double()).abs() / D.double())[:, valid]
            worst = max(worst, float(err.max().item()))
    assert worst <= 1e-5, worst
    print(f"config 4, fp32 bicubic + rotation: max |error| / (largest |tap| of the stencil) = {worst:.3e} over 2 x {NZ} x 9e6 values")
