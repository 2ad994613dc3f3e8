"""The GPU's 3- and 7-parameter datum shifts (proj.cuh datum_shift, chosen by needs_datum_shift) against the independent
reference of tests/datum_reference.py, and their failure masks against the CPU oracle: the values and mesh kernels on random
CRS pairs, edge inputs, the vector matrices, and every table producer as a whole chain.  `FIMEX_B200_DATUM_SEEDS` sets the
number of random pairs."""
import os

import numpy as np
import pytest

import datum_reference as ref
from conftest import assert_bit_equal

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import Method  # noqa: E402

GPU_BAR_DEG = 1e-9
DEG = np.pi / 180
WGS84 = "+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs"
INTL7 = "+ellps=intl +towgs84=-87,-98,-121,0.4,-0.3,0.8,1.5"
SRC_0_360 = f"+proj=latlong {INTL7} +no_defs"  # a lat/lon source on 0..360 carrying a 7-parameter shift
STERE_NAD = "+proj=stere +lat_0=90 +lon_0=-32 +lat_ts=60 +ellps=bessel +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7 +no_defs"
ROT_SHIFT = "+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +R=6371000 +towgs84=120,-40,310 +no_defs"
SEEDS = int(os.environ.get("FIMEX_B200_DATUM_SEEDS", "48"))


def gpu_project(a, b, x, y):
    rc, gx, gy = fb.mifi_project_values(a, b, x, y)
    return (1 if rc == fb.MIFI_OK else rc), gx, gy


@pytest.fixture(scope="module")
def cases():
    return [ref.fuzz_case(7000 + s) for s in range(SEEDS)]


@pytest.mark.parametrize("seed", range(SEEDS))
def test_project_values_against_reference(oracle, cases, seed):
    src, dst, lon, lat = cases[seed]
    sx, sy, glon, glat = ref.source_points(gpu_project, src, lon, lat)
    gx, gy = ref.check(gpu_project, src, dst, sx, sy, glon, glat, GPU_BAR_DEG, f"seed {seed}")
    rc, wx, wy = oracle.project_values(src.proj, dst.proj, sx, sy)
    assert rc == 1
    assert np.array_equal(np.isfinite(gx), np.isfinite(wx)) and np.array_equal(np.isfinite(gy), np.isfinite(wy)), (src.proj, dst.proj)


@pytest.mark.parametrize("seed", range(0, SEEDS, 4))
def test_project_axes_against_reference(oracle, cases, seed):
    src, dst, lon, lat = cases[seed]
    sx, sy, _, _ = ref.source_points(gpu_project, src, lon, lat)
    xa = np.linspace(sx.min(), sx.max(), 23)
    ya = np.linspace(sy.min(), sy.max(), 19)
    rc, gx, gy = fb.mifi_project_axes(src.proj, dst.proj, xa, ya)
    assert rc == fb.MIFI_OK
    mx, my = (a.ravel() for a in np.meshgrid(xa, ya))
    if src.family == "ll":
        glon, glat = mx, my
    else:
        _, glon, glat = gpu_project(src.plain, src.geographic, mx, my)
    rlon, rlat = ref.shift(src.fig, src.datum, dst.fig, dst.datum, glon, glat)
    live = np.isfinite(rlon)
    err = ref.arc_error_deg(gpu_project, dst, gx[live], gy[live], rlon[live], rlat[live])
    assert np.nanmax(err, initial=0.0) <= GPU_BAR_DEG, (src.proj, dst.proj)
    rc, wx, wy = oracle.project_axes(src.proj, dst.proj, xa, ya)
    assert rc == 1 and np.array_equal(np.isfinite(gx), np.isfinite(wx)) and np.array_equal(np.isfinite(gy), np.isfinite(wy))


def test_parser_semantics_on_the_device():
    ref.check_first_key_wins_and_datum_figures(gpu_project, GPU_BAR_DEG)
    ref.check_towgs84_forms(gpu_project, GPU_BAR_DEG)
    x, y = np.radians([10.0, 20.0]), np.radians([50.0, 60.0])
    for bad in ("+proj=latlong +ellps=WGS84 +nadgrids=@null +no_defs", "+proj=latlong +datum=ED50 +no_defs"):
        assert fb.mifi_project_values(bad, WGS84, x, y)[0] != fb.MIFI_OK, bad
        assert fb.mifi_project_values(WGS84, bad, x, y)[0] != fb.MIFI_OK, bad


@pytest.mark.parametrize("case", range(len(ref.IDENTITY)))
def test_identity_cases_are_bitwise_datum_free(case):
    src, dst = ref.IDENTITY[case]
    x, y = ref.identity_inputs(gpu_project, src)
    a = fb.mifi_project_values(src, dst, x, y)
    b = fb.mifi_project_values(ref.strip_datum(src), ref.strip_datum(dst), x, y)
    assert a[0] == b[0] == fb.MIFI_OK
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64)) and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))


@pytest.mark.parametrize("case", range(3))
def test_edge_inputs(oracle, case):
    """latitudes just past a pole (clamped) and further (failed), longitudes outside (-180, 180], exact poles, a pure
    z-translation that keeps a pole on the axis"""
    src, dst, lon, lat = ref.edge_cases()[case]
    x, y = np.radians(lon), np.radians(lat)
    rc, gx, gy = fb.mifi_project_values(src.proj, dst.proj, x, y)
    assert rc == fb.MIFI_OK
    rlon, rlat = ref.shift(src.fig, src.datum, dst.fig, dst.datum, x, y)
    _, wx, wy = oracle.project_values(src.proj, dst.proj, x, y)
    for g, w, r in ((gx, wx, rlon), (gy, wy, rlat)):
        assert np.array_equal(np.isfinite(g), np.isfinite(w)) and np.array_equal(np.isfinite(g), np.isfinite(r))
    ok = np.isfinite(rlon)
    assert (np.abs(gx[ok]) <= np.pi).all()
    assert ref.arc_error_deg(gpu_project, dst, gx[ok], gy[ok], rlon[ok], rlat[ok]).max() <= GPU_BAR_DEG
    pole = ok & (np.abs(np.abs(rlat) - np.pi / 2) < 1e-15)
    assert (case != 2 or pole.sum() == 5) and (gx[pole] == 0).all() and (np.abs(gy[pole]) == np.pi / 2).all()
    # one point at a time: the datum step never fails a call, so every point gives what it gave in the batch
    for i in range(lon.size):
        rc1, g1x, g1y = fb.mifi_project_values(src.proj, dst.proj, x[i:i + 1], y[i:i + 1])
        assert rc1 == fb.MIFI_OK and g1x[0].tobytes() == gx[i].tobytes() and g1y[0].tobytes() == gy[i].tobytes()


def test_failed_inverse_and_single_point_errors(oracle):
    """points whose source inverse already failed stay failed through the shift; a single point whose destination
    projection fails fails the call (n == 1), in a batch it only fails itself"""
    lcc = "+proj=lcc +lat_1=50 +lat_2=60 +lon_0=10 +ellps=bessel +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7 +no_defs"
    lon = np.radians([10.0, 40.0, -20.0, 10.0, 170.0])
    lat = np.radians([-90.0, 55.0, 30.0, 89.0, -90.0])
    _, sx, sy = oracle.project_values("+proj=latlong +ellps=bessel +no_defs", lcc.replace(" +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7", ""),
                                      lon, lat)
    assert not np.isfinite(sx[0]) and np.isfinite(sx[1])  # the far pole has no lcc image
    rc, gx, gy = fb.mifi_project_values(lcc, WGS84, sx, sy)
    rc2, wx, wy = oracle.project_values(lcc, WGS84, sx, sy)
    assert rc == fb.MIFI_OK and rc2 == 1
    assert np.array_equal(np.isfinite(gx), np.isfinite(wx)) and not np.isfinite(gx[[0, 4]]).any() and np.isfinite(gx[1:4]).all()
    _, glon, glat = gpu_project(lcc.replace(" +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7", ""), "+proj=latlong +ellps=bessel +no_defs",
                                sx[1:4], sy[1:4])
    rlon, rlat = ref.shift(ref.figure_of_ellps("bessel"), ref.Datum(ref.REALISTIC[0]), ref.figure_of_ellps("WGS84"),
                           ref.Datum((0.0, 0.0, 0.0)), glon, glat)
    wgs = ref.latlong_crs("+ellps=WGS84", ref.figure_of_ellps("WGS84"), (0.0, 0.0, 0.0))
    assert ref.arc_error_deg(gpu_project, wgs, gx[1:4], gy[1:4], rlon, rlat).max() <= GPU_BAR_DEG
    # destination failure: the south pole, kept on the axis by a pure z-translation, has no image in a north lcc
    to_lcc = ("+proj=latlong +R=6371000 +towgs84=0,0,120 +no_defs", "+proj=lcc +lat_1=50 +lat_2=60 +lon_0=10 +R=6371000 +towgs84=0,0,0 +no_defs")
    lon, lat = np.radians([30.0, 30.0]), np.radians([-90.0, 60.0])
    rc, bx, _ = fb.mifi_project_values(*to_lcc, lon, lat)
    assert rc == fb.MIFI_OK and not np.isfinite(bx[0]) and np.isfinite(bx[1])
    for i in range(2):
        g1 = fb.mifi_project_values(*to_lcc, lon[i:i + 1], lat[i:i + 1])[0]
        w1 = oracle.project_values(*to_lcc, lon[i:i + 1], lat[i:i + 1])[0]
        assert (g1 == fb.MIFI_OK) == (w1 == 1) == (i == 1)


# --------------------------------------------------------------------------------------------------------- vector matrices
def _angles_close(got, want):
    fin = np.isfinite(want[3::4])
    assert np.array_equal(np.isfinite(got[3::4]), fin)
    d = np.remainder(got[3::4][fin] - want[3::4][fin] + np.pi, 2 * np.pi) - np.pi
    assert np.abs(d).max(initial=0.0) <= 1e-7 * DEG
    assert np.abs(got[0::4][fin]**2 + got[1::4][fin]**2 - 1).max(initial=0.0) < 1e-14


LONLAT_FIELD = (np.radians(np.linspace(-40, 20, 25)), np.radians(np.linspace(50, 85, 19)))
VECTOR_PAIRS = [  # (input CRS, output CRS, output axes, their types, a field of input-CRS positions)
    (SRC_0_360, STERE_NAD, (np.linspace(-2e6, 2e6, 31), np.linspace(-3e6, 1e6, 27)), (0, 0), LONLAT_FIELD),
    ("+proj=latlong +R=6371000 +towgs84=0,0,0 +no_defs", ROT_SHIFT, (np.linspace(-10, 10, 21), np.linspace(-8, 8, 17)), (1, 2), LONLAT_FIELD),
    (STERE_NAD, f"+proj=lcc +lat_1=45 +lat_2=65 +lon_0=15 {INTL7} +no_defs", (np.linspace(-1e6, 1e6, 25), np.linspace(-2e6, 2e6, 23)),
     (0, 0), (np.linspace(-1.5e6, 1.5e6, 21), np.linspace(-3e6, 0, 17))),
]


@pytest.mark.parametrize("case", range(len(VECTOR_PAIRS)))
def test_vector_matrices_on_shifted_pairs(oracle, case):
    src, dst, (ax, ay), types, (fx, fy) = VECTOR_PAIRS[case]
    rc, want = oracle.vector_matrix(src, dst, ax, ay, types[0], types[1])
    assert rc == 1
    rc, got = fb.mifi_get_vector_reproject_matrix(src, dst, ax, ay, types[0], types[1])
    assert rc == fb.MIFI_OK
    _angles_close(got, want)
    cvr = fb.CachedVectorReprojection.fromProjection(0, src, dst, ax, ay, types[0], types[1])
    _angles_close(cvr.getMatrix(), want)
    # the field form: a mesh of input-CRS positions
    mx, my = (a.ravel() for a in np.meshgrid(fx, fy))
    rc, wf = oracle.vector_matrix_field(src, dst, mx, my, fx.size, fy.size)
    assert rc == 1
    rc, gf = fb.mifi_get_vector_reproject_matrix_field(src, dst, mx, my, fx.size, fy.size)
    assert rc == fb.MIFI_OK
    _angles_close(gf, wf)
    # the values form: u/v rotated by that matrix
    rng = np.random.default_rng(case)
    u = rng.normal(0, 8, (2, ay.size, ax.size)).astype(np.float32)
    v = rng.normal(0, 8, (2, ay.size, ax.size)).astype(np.float32)
    rc, wu, wv = oracle.vector_reproject_values(src, dst, u, v, ax, ay, types[0], types[1], 2)
    rc2, gu, gv = fb.mifi_vector_reproject_values_f(0, src, dst, u, v, ax, ay, types[0], types[1], 2)
    assert rc == 1 and rc2 == fb.MIFI_OK
    speed = np.hypot(u, v).ravel()
    assert np.abs(np.hypot(gu, gv).ravel() - speed).max() <= 1e-5 * speed.max()
    assert np.abs(gu.ravel() - wu.ravel()).max() <= 1e-5 * speed.max() and np.abs(gv.ravel() - wv.ravel()).max() <= 1e-5 * speed.max()


def test_vector_matrix_points_and_grid(oracle):
    # the points form takes geographic points of the output CRS (the lat/lon-template path: a source CRS to lat/lon) and
    # differentiates in the input CRS over 100 m when that CRS is metric, over 1e-5 rad when it is in degrees
    rng = np.random.default_rng(9)
    lon, lat = rng.uniform(-60, 60, 300), rng.uniform(-10, 80, 300)
    for src, dst, metric in ((STERE_NAD, WGS84, 1), (ROT_SHIFT, WGS84, 0), (STERE_NAD, SRC_0_360, 1)):
        rc, want = oracle.vector_matrix_points(src, dst, metric, np.radians(lon), np.radians(lat))
        assert rc == 1
        rc, got = fb.mifi_get_vector_reproject_matrix_points(src, dst, metric, np.radians(lon), np.radians(lat))
        assert rc == fb.MIFI_OK
        _angles_close(got, want)
        _angles_close(fb.CachedVectorReprojection.fromPoints(fb.MIFI_VECTOR_KEEP_SIZE, src, dst, metric, lon, lat).getMatrix(), want)
    # a grid's own axes towards geographic directions (both against the WGS84 lat/lon CRS)
    xa, ya = np.linspace(-2e6, 2e6, 29), np.linspace(-3e6, 1e6, 21)
    mx, my = (a.ravel() for a in np.meshgrid(xa, ya))
    rc, want = oracle.vector_matrix_field(STERE_NAD, WGS84, mx, my, xa.size, ya.size)
    assert rc == 1
    _angles_close(fb.CachedVectorReprojection.fromGrid(fb.MIFI_VECTOR_KEEP_SIZE, STERE_NAD, xa, ya, False, True).getMatrix(), want)
    # and back from geographic directions: the axes go in as radians, so use a lat/lon grid (0..360, carrying a shift)
    lon_ax, lat_ax = np.arange(0.0, 360.0, 2.0), np.arange(-80.0, 80.1, 2.0)
    rc, want = oracle.vector_matrix(WGS84, SRC_0_360, np.radians(lon_ax), np.radians(lat_ax), 0, 0)
    assert rc == 1
    _angles_close(fb.CachedVectorReprojection.fromGrid(fb.MIFI_VECTOR_KEEP_SIZE, SRC_0_360, lon_ax, lat_ax, True, False).getMatrix(), want)


# ------------------------------------------------------------------------------------------------------ table producers
def _check_tables(oracle, method, ci, opx, opy, inX, inY, outX, outY, what):
    """positions within 4e-9 cells of the oracle's; gathers bit-exact on the device's own positions; every index that
    differs from the oracle's belongs to a position within 4e-9 cells of a cell (or half-cell) boundary"""
    gx, gy = ci.points()
    assert np.array_equal(np.isfinite(gx), np.isfinite(opx)) and np.array_equal(np.isfinite(gy), np.isfinite(opy)), what
    fin = np.isfinite(opx) & np.isfinite(opy)
    assert np.abs(gx[fin] - opx[fin]).max() <= 4e-9 and np.abs(gy[fin] - opy[fin]).max() <= 4e-9, what
    for g, o in ((gx[fin], opx[fin]), (gy[fin], opy[fin])):
        flip = np.floor(2 * g) != np.floor(2 * o)
        assert (np.abs(2 * o[flip] - np.round(2 * o[flip])) <= 8e-9).all(), what
    field = np.random.default_rng(5).normal(250, 30, (3, inY, inX)).astype(np.float32)
    got = ci.interpolateValues(field)
    assert_bit_equal(got, oracle.cached_interpolate(int(method), gx, gy, inX, inY, outX, outY, field), what,
                     nan_payload=(method == Method.NEAREST_NEIGHBOR))


LON_0_360 = np.arange(1440) * 0.25
LAT_DESC = 90 - np.arange(721) * 0.25


@pytest.mark.parametrize("method", [Method.NEAREST_NEIGHBOR, Method.BILINEAR, Method.BICUBIC])
def test_from_projection_with_shift(oracle, method):
    ax, ay = np.linspace(-3.5e6, 3.5e6, 140), np.linspace(-4e6, 2e6, 120)
    rc, x, y = oracle.project_axes(STERE_NAD, SRC_0_360, ax, ay)
    assert rc == 1
    px = oracle.points2position(x, np.radians(LON_0_360), 1)
    py = oracle.points2position(y, np.radians(LAT_DESC), 2)
    ci = fb.CachedInterpolation.fromProjection(method, STERE_NAD, ax, ay, False, False, SRC_0_360, LON_0_360, LAT_DESC, True)
    assert (x < 0).any()  # the shift returns (-180, 180]; points2position wraps that onto the 0..360 source
    _check_tables(oracle, method, ci, px, py, LON_0_360.size, LAT_DESC.size, ax.size, ay.size, f"fromProjection {method}")


@pytest.mark.parametrize("method", [Method.NEAREST_NEIGHBOR, Method.BILINEAR])
def test_from_template_with_shift(oracle, method):
    ny, nx = 30, 50
    jj, ii = np.meshgrid(np.arange(nx), np.arange(ny))
    tlon = (-40 + 1.6 * jj + 0.1 * ii + 0.3 * np.sin(ii / 5.0)).ravel()
    tlat = (30 + 1.4 * ii - 0.05 * jj + 0.2 * np.cos(jj / 7.0)).ravel()
    tlon[:5] = [-180.0, 180.0, 359.0, -0.01, 0.0]
    ci = fb.CachedInterpolation.fromTemplate(method, WGS84, tlon, tlat, nx, ny, SRC_0_360, LON_0_360, LAT_DESC, True)
    rc, x, y = oracle.project_values(WGS84, SRC_0_360, np.radians(tlon), np.radians(tlat))
    assert rc == 1 and (x < 0).any()
    px = oracle.points2position(x, np.radians(LON_0_360), 1)
    py = oracle.points2position(y, np.radians(LAT_DESC), 2)
    _check_tables(oracle, method, ci, px, py, LON_0_360.size, LAT_DESC.size, nx, ny, f"fromTemplate {method}")


def test_forward_from_coordinates_with_shift(oracle):
    rng = np.random.default_rng(3)
    ny, nx = 120, 80
    lat = 60 + np.linspace(0, 4, ny)[:, None] + np.linspace(0, 0.4, nx)[None, :] + rng.normal(0, 1e-3, (ny, nx))
    lon = 10 + np.linspace(0, 1, ny)[:, None] + np.linspace(0, 6, nx)[None, :]
    target = f"+proj=lcc +lat_1=50 +lat_2=70 +lat_0=60 +lon_0=15 {INTL7} +no_defs"
    ox, oy = np.arange(-200e3, 200e3 + 1, 5e3), np.arange(-350e3, 150e3 + 1, 5e3)
    rc, x, y = oracle.project_values(WGS84, target, np.radians(lon.ravel()), np.radians(lat.ravel()))
    assert rc == 1
    px, py = oracle.points2position(x, ox, 0), oracle.points2position(y, oy, 0)
    data = rng.normal(0, 1, (2, ny, nx)).astype(np.float32)
    cfi = fb.CachedForwardInterpolation.fromCoordinates(Method.FORWARD_MEAN, target, ox, oy, False, False, lon.ravel(), lat.ravel(), nx, ny)
    gx, gy = cfi.points()
    assert np.abs(gx - px).max() <= 4e-9 and np.abs(gy - py).max() <= 4e-9
    flips = (np.round(gx) != np.round(px)) | (np.round(gy) != np.round(py))
    assert (np.minimum(np.abs(px - np.floor(px) - 0.5), np.abs(py - np.floor(py) - 0.5))[flips] <= 4e-9).all()
    assert_bit_equal(cfi.interpolateValues(data), oracle.forward_interpolate(int(Method.FORWARD_MEAN), gx, gy, nx, ny, ox.size, oy.size, data),
                     "forward from coordinates")


# ------------------------------------------------------------------------------------------------------ Interpolator
@pytest.mark.parametrize("source", [STERE_NAD, f"+proj=lcc +lat_1=50 +lon_0=10 {INTL7} +no_defs", ROT_SHIFT,
                                    "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6378137 +b=6356752.3142 +towgs84=5,-9,12 +no_defs"])
def test_interpolator_lonlat_conversions_apply_no_shift(source):
    """the geographic CRS of convertFromLonLat / convertToLonLat keeps the source's earth tokens, datum included, so no
    shift happens: the results equal, bit for bit, those of the same source without its datum"""
    is_deg = "ob_tran" in source
    xs, ys = (np.linspace(-10, 10, 11), np.linspace(-8, 8, 9)) if is_deg else (np.linspace(-2e6, 2e6, 11), np.linspace(-2e6, 2e6, 9))
    with_datum = fb.Interpolator(source, xs, ys, is_deg)
    without = fb.Interpolator(ref.strip_datum(source), xs, ys, is_deg)
    lon, lat = np.linspace(-30, 40, 50), np.linspace(40, 85, 50)
    a, b = with_datum.convertFromLonLat(lon, lat), without.convertFromLonLat(lon, lat)
    assert all(np.array_equal(p.view(np.uint64), q.view(np.uint64)) for p, q in zip(a, b))
    a, b = with_datum.convertToLonLat(xs, ys[:1].repeat(xs.size)), without.convertToLonLat(xs, ys[:1].repeat(xs.size))
    assert all(np.array_equal(p.view(np.uint64), q.view(np.uint64)) for p, q in zip(a, b))
