"""The coordinate searches on the GPU (coord_nearestneighbor, coord_kdtree; `fimex_b200/csrc/coordnn_kernels.cu`) against the
independent reference `tests/coord_nn_reference.py`, through `CachedInterpolation.fromCoordinates` (the C ABI the reference's
call sites use).  Every target of every case is checked: unambiguous targets must name the reference's source, ambiguous ones
one of its candidates; where the reference calls a target unambiguous the restatement (`orc_coordnn` / `orc_coordkd`) must
agree too.  The designed edges are compared bit for bit with the stated tie rules.  `FIMEX_B200_CNNFUZZ_SEEDS` sets the number
of fuzz cases (default 60, half per method)."""
import os

import numpy as np
import pytest

from conftest import assert_bit_equal
import coord_nn_reference as R

pytestmark = pytest.mark.gpu

import fimex_b200 as fb  # noqa: E402
from fimex_b200 import Method  # noqa: E402

SEEDS = int(os.environ.get("FIMEX_B200_CNNFUZZ_SEEDS", "60"))
WGS84 = R.WGS84
MISS = {"nn": -1, "kd": -1000}


def _run(case):
    m = Method.COORD_NN if case["method"] == "nn" else Method.COORD_NN_KD
    ci = fb.CachedInterpolation.fromCoordinates(m, case["tcrs"], case["xa"], case["ya"], True, True, case["lon"], case["lat"], case["nx"],
                                                case["ny"], maxDistance=case["max_dist"])
    gx, gy = ci.points()
    return ci, gx, gy


def _table_in_use(ci, case, gx, gy, oracle, rng):
    """interpolateValues with the GPU's own indices, NaN payload included, against the restated gather"""
    nx, ny, ox, oy = case["nx"], case["ny"], case["xa"].size, case["ya"].size
    field = rng.normal(0, 1, (2, ny, nx)).astype(np.float32)
    field[rng.random(field.shape) < 0.05] = np.nan
    method = 3 if case["method"] == "nn" else 4
    assert_bit_equal(ci.interpolateValues(field), oracle.cached_interpolate(method, gx, gy, nx, ny, ox, oy, field), "table in use",
                     nan_payload=True)


def _check(case, oracle, exact_ties=False, with_oracle=True, rng=None):
    ci, gx, gy = _run(case)
    ref = R.reference_for(case, oracle, exact_ties=exact_ties)
    tx, ty, _ = R.case_targets(case, oracle)
    inside = np.abs(ty) < np.pi / 2  # at a pole every longitude of a latitude row is equidistant
    what = f"seed {case['seed']} {case['family']} {case['method']} {case['nx']}x{case['ny']} -> {gx.size} ({case['tcrs'][:14]})"
    n_amb = R.compare(ref, gx, gy, what, share_of=inside)
    if with_oracle:
        wx, wy, _ = R.oracle_for(case, oracle)
        # the restated scan prunes on |dlat|, which is no bound for a target beyond a pole (DESIGN section 2)
        sure = ~ref.amb & (np.abs(ty) <= np.pi / 2 if case["method"] == "nn" else True)
        bad = np.flatnonzero(sure & ((gx != wx) | (gy != wy)))
        assert bad.size == 0, f"{what}: {bad.size} targets differ from the restatement, first {bad[:5]}"
    _table_in_use(ci, case, gx, gy, oracle, rng or np.random.default_rng(case["seed"]))
    return ref, gx, gy, n_amb


def test_wgs84_target_projection_is_the_identity():
    """the search's targets are the mesh of the axes in radians: the latlong -> latlong step changes no bit, poles, date line
    and beyond included"""
    x = R.to_rad(np.array([-190.0, -180.0, -179.99, 0.0, 33.3, 180.0, 190.0, 359.5]))
    y = R.to_rad(np.array([-95.0, -90.0, -45.1, -0.0, 0.0, 12.7, 90.0, 95.0]))
    rc, px, py = fb.mifi_project_axes(WGS84, WGS84, x, y)
    assert rc == fb.MIFI_OK
    assert np.array_equal(px.view(np.uint64), np.tile(x, y.size).view(np.uint64))
    assert np.array_equal(py.view(np.uint64), np.repeat(y, x.size).view(np.uint64))


@pytest.mark.parametrize("seed", range(SEEDS))
def test_fuzz_against_reference(seed, oracle):
    case = R.make_case(seed, method="nn" if seed % 2 == 0 else "kd")
    _check(case, oracle)


@pytest.mark.parametrize("method", ["nn", "kd"])
def test_every_target_beyond_one_grid_stride(method, oracle):
    """more targets than the search's grid has warps (148 SMs x 64 blocks x 8 warps = 75 776), every one checked, on a
    1500 x 1500 curvilinear source"""
    case = R.make_case(1000 + (method == "kd"), family="curvilinear", method=method, max_src=1500 * 1500, max_tgt=1)
    rng = np.random.default_rng(5)
    nx = ny = 1500
    i = np.arange(nx)[None, :].astype(np.float64)
    j = np.arange(ny)[:, None].astype(np.float64)
    case.update(nx=nx, ny=ny, lon=(-20 + 0.02 * i + 0.005 * j + 0.1 * np.sin(j / 50)).ravel(),
                lat=(30 + 0.015 * j - 0.004 * i + 0 * i).ravel(), tcrs=WGS84, max_dist=30e3 if method == "kd" else 0.0)
    case["xa"] = -22 + 35 * np.arange(600) / 599 + rng.uniform(0, 0.01)
    case["ya"] = 24 + 32 * np.arange(505) / 504 + rng.uniform(0, 0.01)
    assert case["xa"].size * case["ya"].size > 300000
    ref, gx, gy, _ = _check(case, oracle, with_oracle=(method == "nn"))
    assert (ref.ix >= 0).sum() > 75776 and (ref.ix == MISS[method]).sum() > 1000


def _tiny(lon, lat, nx, ny, xa, ya, method, max_dist=0.0, seed=0):
    return dict(seed=seed, family="designed", method=method, nx=nx, ny=ny, lon=np.asarray(lon, np.float64), lat=np.asarray(lat, np.float64),
                tcrs=WGS84, xa=np.asarray(xa, np.float64), ya=np.asarray(ya, np.float64), max_dist=max_dist)


@pytest.mark.parametrize("method", ["nn", "kd"])
@pytest.mark.parametrize("first", ["+0", "-0"])
def test_signed_zero_latitude_tie(first, method, oracle):
    """two sources at exactly mirrored longitudes, one at latitude +0 and one at -0, and a target at (0, 0): an exact tie.
    coord_nn takes the one inserted first (equal latitudes in insertion order, -0 equal to +0); coord_kdtree the lowest
    position.  Both are ix = 0 whichever sign comes first."""
    lat = [0.0, -0.0] if first == "+0" else [-0.0, 0.0]
    case = _tiny([0.7, -0.7], lat, 2, 1, [0.0], [0.0], method, max_dist=500e3)
    ci, gx, gy = _run(case)
    assert (gx[0], gy[0]) == (0, 0), (first, method, gx, gy)
    ref = R.reference_for(case, oracle, exact_ties=True)
    assert not ref.amb[0] and (ref.ix[0], ref.iy[0]) == (0, 0)
    wx, wy, ties = R.oracle_for(case, oracle)
    assert (wx[0], wy[0]) == (0, 0) and ties == 1


@pytest.mark.parametrize("layout", ["x", "y"])
@pytest.mark.parametrize("mirror", [False, True])
def test_equal_latitude_ties_follow_insertion_order(layout, mirror, oracle):
    """sources at one latitude and exactly mirrored longitudes (cos h == cos -h).  A target below the row meets it scanning up:
    the first inserted wins; a target above meets it scanning down: the last inserted wins; a target on the row scans up.
    Insertion order is ix outer, iy inner, so the sources are laid out along x or along y.  A second pair at +-a latitude
    around a target on the equator is met scanning up first (+a) whatever the insertion order."""
    lon = [-0.9, 0.9] if not mirror else [0.9, -0.9]
    lat = [40.0, 40.0]
    nx, ny = (2, 1) if layout == "x" else (1, 2)
    for ya, want_first in (([38.5], True), ([41.5], False), ([40.0], True)):
        case = _tiny(lon, lat, nx, ny, [0.0], ya, "nn")
        ci, gx, gy = _run(case)
        want = (0, 0) if want_first else ((1, 0) if layout == "x" else (0, 1))
        assert (gx[0], gy[0]) == want, (layout, mirror, ya, gx, gy)
        ref = R.reference_for(case, oracle, exact_ties=True)
        wx, wy, _ = R.oracle_for(case, oracle)
        assert (ref.ix[0], ref.iy[0]) == want and (wx[0], wy[0]) == want
    for lat2 in ([3.0, -3.0], [-3.0, 3.0]):
        case = _tiny([10.0, 10.0], lat2, nx, ny, [10.0], [0.0], "nn")
        ci, gx, gy = _run(case)
        up = lat2.index(3.0)
        want = (up, 0) if layout == "x" else (0, up)
        assert (gx[0], gy[0]) == want
        wx, wy, _ = R.oracle_for(case, oracle)
        assert (wx[0], wy[0]) == want


@pytest.mark.parametrize("method", ["nn", "kd"])
def test_nan_source_coordinates_and_targets(method, oracle):
    """NaN in the longitude only and in the latitude only drops a source; targets placed exactly on the dropped points go to a
    neighbour; a NaN target matches nothing"""
    nx, ny = 23, 17
    lon = np.tile(5 + 0.37 * np.arange(nx), ny)
    lat = np.repeat(40 + 0.29 * np.arange(ny), nx)
    holes = [3 + 5 * nx, 11 + 9 * nx, 20 + 2 * nx]
    lon[holes[0]] = np.nan
    lat[holes[1]] = np.nan
    lon[holes[2]] = lat[holes[2]] = np.nan
    xa = np.concatenate([5 + 0.37 * np.array([3.0, 11.0, 20.0]) + 1e-3, [np.nan, 7.0]])
    ya = np.concatenate([40 + 0.29 * np.array([5.0, 9.0, 2.0]), [np.nan]])
    case = _tiny(lon, lat, nx, ny, xa, ya, method, max_dist=80e3)
    ref, gx, gy, _ = _check(case, oracle)
    nan_t = np.isnan(np.tile(xa, ya.size)) | np.isnan(np.repeat(ya, xa.size))
    assert (gx[nan_t] == MISS[method]).all() and (gy[nan_t] == MISS[method]).all()
    pos = gx[~nan_t] + gy[~nan_t] * nx
    assert not np.isin(pos[gx[~nan_t] >= 0], holes).any()


def test_whole_sphere_pole_rows(oracle):
    """a whole-sphere regular source with rows at +-90 degrees.  For a target at the pole every point of the pole row has
    cos_d == 1 exactly: the first of them in insertion order (ix = 0) wins.  All other targets against the reference."""
    lons = np.arange(0, 360, 2.5)
    lats = np.arange(90, -90.1, -2.5)
    lon, lat = np.tile(lons, lats.size), np.repeat(lats, lons.size)
    xa = np.array([-170.3, -35.0, 0.0, 61.1, 179.9])
    for ya, row in (([90.0], 0), ([-90.0], lats.size - 1)):
        case = _tiny(lon, lat, lons.size, lats.size, xa, ya, "nn")
        ci, gx, gy = _run(case)
        assert (gx == 0).all() and (gy == row).all(), (gx, gy)
        ref = R.reference_for(case, oracle, exact_ties=True)
        wx, wy, _ = R.oracle_for(case, oracle)
        assert (ref.ix == 0).all() and (ref.iy == row).all() and (wx == 0).all() and (wy == row).all()
    rng = np.random.default_rng(3)
    for method in ("nn", "kd"):
        case = _tiny(lon, lat, lons.size, lats.size, np.sort(rng.uniform(-180, 180, 300)), np.sort(rng.uniform(-88.0, 88.0, 200)), method,
                     max_dist=200e3, seed=3)
        _check(case, oracle)


@pytest.mark.parametrize("max_dist", [0.0, 1.0, 12742e3, 2e7])
def test_kd_distances(max_dist, oracle):
    """maxDistance derived from the axes (degrees times the earth radius), 1 m (only exact hits), and r >= 2 (the whole
    sphere: the window covers every latitude; at r == 2 an antipodal source is at the radius)"""
    case = R.make_case(77, family="curvilinear", method="kd", max_src=5000, max_tgt=5000)
    case["max_dist"] = max_dist
    case["tcrs"] = WGS84
    lon, lat = case["lon"], case["lat"]
    # targets on some sources (exact hits for 1 m) and on their antipodes
    k = np.flatnonzero(~np.isnan(lon) & ~np.isnan(lat))[:7]
    case["xa"] = np.concatenate([case["xa"], lon[k]])
    case["ya"] = np.concatenate([case["ya"], lat[k]])
    ref, gx, gy, _ = _check(case, oracle)
    if max_dist == 1.0:
        assert (gx >= 0).any()
    if max_dist >= 12742e3:
        assert (gx >= 0).mean() > 0.99


def test_kd_radius_is_strict(oracle):
    """a source whose squared chord equals r*r is outside (RadiusResultSet: dist < radius); one step more and it is inside.
    Target (0, 0), source (180, 0): q = (1, 0, 0), p = (-1, sin(pi), 0), so the chord squared is 4 + sin(pi)**2, which rounds
    to 4, and maxDistance = 12 742 km gives r = 2 exactly."""
    at = 12742e3
    above = float(np.nextafter(at, np.inf))
    assert at / R.EARTH_R == 2.0 and (above / R.EARTH_R) ** 2 > 4.0
    for md, want in ((at, -1000), (above, 0)):
        case = _tiny([180.0], [0.0], 1, 1, [0.0], [0.0], "kd", max_dist=md)
        wx, wy, _ = R.oracle_for(case, oracle)
        ci, gx, gy = _run(case)
        assert gx[0] == want and wx[0] == want, (md, gx, wx)
        # the reference leaves a chord this close to the radius to rounding and accepts either answer
        ref = R.reference_for(case, oracle)
        assert ref.amb[0] and (want, want if want < 0 else 0) in ref.cand[0]


def test_kd_latitude_window(oracle):
    """the kd search's latitude window: a source due south of the target at 59 degrees, chord 2 sin(29.5 deg) = 0.985 < r = 1
    (maxDistance 6371 km), lies beyond |dlat| = r but within the window 2 asin(r / 2) = 60 degrees; and a target at latitude 95
    is the point (85, lon + 180), where a source sits exactly"""
    for lon, lat, xa, ya, md in (([10.0, 100.0], [40.0, -30.0], [10.0], [-19.0], 6371e3), ([-170.0, 0.0], [85.0, 0.0], [10.0], [95.0], 100e3)):
        case = _tiny(lon, lat, 2, 1, xa, ya, "kd", max_dist=md)
        ci, gx, gy = _run(case)
        ref = R.reference_for(case, oracle)
        wx, wy, _ = R.oracle_for(case, oracle)
        assert (gx[0], gy[0]) == (0, 0) == (ref.ix[0], ref.iy[0]) == (wx[0], wy[0]) and not ref.amb[0], (ya, gx, gy)


def _switch_case(ns_x, ns_y, iso, method="nn"):
    """a dense 0.1-degree cluster of ns_x x ns_y points with the point at position `iso` moved 5 degrees away"""
    lon = np.tile(10 + 0.1 * np.arange(ns_x), ns_y)
    lat = np.repeat(50 + 0.1 * np.arange(ns_y), ns_x)
    lon[iso], lat[iso] = 10 + 0.1 * ns_x + 5.0, 45.0
    xa = 10 + 0.1 * ns_x + 0.05 + 0.25 * np.arange(12) + 0.0123
    ya = 50 + 0.1 * ns_y * np.arange(3) / 2 + 0.0071
    return _tiny(lon, lat, ns_x, ns_y, xa, ya, method)


def test_grid_distance_sampling_switch(oracle):
    """getGridDistance samples every point up to nx*ny = 1000 and 53 points k*(nx*ny/53) above.  An isolated point widens the
    ROI only when it is sampled: at 1000 always, at 1001 only at a multiple of 1001/53 = 18 (54 is, 55 is not)."""
    mapped = {}
    for name, (sx, sy, iso) in {"1000": (40, 25, 55), "1001_sampled": (77, 13, 54), "1001_skipped": (77, 13, 55)}.items():
        case = _switch_case(sx, sy, iso)
        ref, gx, gy, _ = _check(case, oracle)
        mapped[name] = int((gx >= 0).sum())
    assert mapped["1000"] > mapped["1001_skipped"] and mapped["1001_sampled"] > mapped["1001_skipped"], mapped


def test_single_valid_source_and_no_valid_sample(oracle):
    """one valid source: the ROI is 1.414 acos(-2), NaN, and every target gets (-1, -1), as in the reference.  No valid sample
    point among the 53 while other points are valid: acos(2), NaN, the same."""
    lon = np.full(12, np.nan)
    lat = np.full(12, np.nan)
    lon[5], lat[5] = 3.0, 4.0
    case = _tiny(lon, lat, 4, 3, [3.0, 3.1], [4.0], "nn")
    ci, gx, gy = _run(case)
    assert (gx == -1).all() and (gy == -1).all()
    # 1060 points: samples at k * 20; every one of them NaN, the rest a valid grid
    nx, ny = 53, 20
    lon = np.tile(0.5 * np.arange(nx), ny)
    lat = np.repeat(0.5 * np.arange(ny), nx)
    lon[np.arange(53) * (nx * ny // 53)] = np.nan
    case = _tiny(lon, lat, nx, ny, [3.1, 7.3], [2.2], "nn")
    ci, gx, gy = _run(case)
    assert (gx == -1).all() and (gy == -1).all()
    assert np.isnan(R.grid_roi(R.to_rad(lon), R.to_rad(lat), nx, ny)[0])
    wx, wy, _ = R.oracle_for(case, oracle)
    assert (wx == -1).all()
    assert_bit_equal(ci.interpolateValues(np.ones((1, ny, nx), np.float32)), np.full((1, 1, 2), np.nan, np.float32), "all undefined",
                     nan_payload=True)


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (41, 1), (5, 6), (31, 1), (1000, 1), (1001, 1), (7, 143)])
@pytest.mark.parametrize("method", ["nn", "kd"])
def test_sizes(shape, method, oracle):
    """1 x 1, 1-wide grids, fewer valid sources than a warp has lanes, nx*ny = 1000 and 1001"""
    nx, ny = shape
    rng = np.random.default_rng(nx * 7919 + ny)
    lon = (rng.uniform(-30, 30) + np.cumsum(rng.uniform(0.01, 0.3, nx * ny))).ravel()
    lat = (rng.uniform(-60, 60) + np.cumsum(rng.uniform(-0.2, 0.2, nx * ny))).ravel()
    xa = np.linspace(lon.min() - 3, lon.max() + 3, 40) + 0.0017
    ya = np.linspace(lat.min() - 3, lat.max() + 3, 30) + 0.0013
    case = _tiny(lon, lat, nx, ny, xa, ya, method, max_dist=0.0 if method == "nn" else 100e3, seed=nx * 10007 + ny)
    _check(case, oracle)


def test_typed_slice_and_interpolator(oracle):
    """getDataSlice on int16 with a fill value, and an Interpolator built from lon2d / lat2d with coord_nearestneighbor, go
    the same way as the restated gather on the GPU's own indices"""
    case = R.make_case(11, family="swath", method="nn", max_src=20000, max_tgt=3000)
    ci, gx, gy = _run(case)
    nx, ny, ox, oy = case["nx"], case["ny"], case["xa"].size, case["ya"].size
    rng = np.random.default_rng(11)
    packed = rng.integers(-3000, 3000, (3, ny, nx)).astype(np.int16)
    packed[rng.random(packed.shape) < 0.1] = -32767
    want = oracle.from_float(oracle.cached_interpolate(3, gx, gy, nx, ny, ox, oy, oracle.as_float(packed, -32767.0)), -32767.0, np.int16)
    got = ci.getDataSlice(packed, -32767.0)
    assert got.dtype == np.int16 and np.array_equal(got.ravel(), want.ravel())
    ip = fb.Interpolator(WGS84, np.arange(nx, dtype=np.float64), np.arange(ny, dtype=np.float64), False, lon2d=case["lon"], lat2d=case["lat"])
    ip.changeProjection(Method.COORD_NN, WGS84, case["xa"], case["ya"], "degrees_east", "degrees_north")
    px, py = ip.cachedInterpolation.points()
    assert np.array_equal(px, gx) and np.array_equal(py, gy)
    # getDataSlice ends in interpolationArray2Data: NaN, here the (-1, -1) targets, leaves as the float fill value
    field = rng.normal(0, 1, (2, ny, nx)).astype(np.float32)
    fill = fb.default_fill_value(np.float32)
    want = oracle.from_float(oracle.cached_interpolate(3, gx, gy, nx, ny, ox, oy, oracle.as_float(field, fill)), fill, np.float32)
    got = np.asarray(ip.getDataSlice(field))
    assert got.dtype == np.float32 and (gx < 0).any() and (got.ravel() == np.float32(fill)).any()
    assert_bit_equal(got.ravel(), want.ravel(), "Interpolator", nan_payload=True)
