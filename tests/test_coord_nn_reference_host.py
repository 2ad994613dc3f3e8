"""The independent reference for the coordinate searches (`tests/coord_nn_reference.py`) against the restatement
(`orc_coordnn`, `orc_coordkd`) on the CPU, and the reference's own known answers.  No GPU needed."""
import numpy as np
import pytest

import coord_nn_reference as R


def _designed(lon, lat, nx, ny, xa, ya, method, max_dist=0.0):
    return dict(seed=0, family="designed", method=method, nx=nx, ny=ny, lon=np.asarray(lon, np.float64), lat=np.asarray(lat, np.float64),
                tcrs=R.WGS84, xa=np.asarray(xa, np.float64), ya=np.asarray(ya, np.float64), max_dist=max_dist)


def test_longdouble_and_constants(oracle):
    """the reference needs more precision than fp64, and the library's degree -> radian factor and latlong targets"""
    assert np.finfo(np.longdouble).nmant >= 63  # x86-64 extended precision: a 64-bit mantissa
    assert R.DEG_TO_RAD == np.pi / 180
    x = R.to_rad(np.array([-190.0, -180.0, 0.0, 33.3, 180.0, 190.0, 359.5]))
    y = R.to_rad(np.array([-95.0, -90.0, -0.0, 0.0, 12.7, 90.0, 95.0]))
    rc, px, py = oracle.project_axes(R.WGS84, R.WGS84, x, y)
    assert rc == 1
    assert np.array_equal(px.view(np.uint64), np.tile(x, y.size).view(np.uint64))
    assert np.array_equal(py.view(np.uint64), np.repeat(y, x.size).view(np.uint64))


@pytest.mark.parametrize("block", range(10))
def test_restatement_against_reference(block, oracle):
    """200 seeded cases over every geometry family, both methods, latlong and rotated-pole targets"""
    for seed in range(block * 20, block * 20 + 20):
        case = R.make_case(seed, max_src=3000, max_tgt=3000)
        ref = R.reference_for(case, oracle)
        wx, wy, _ = R.oracle_for(case, oracle)
        tx, ty, _ = R.case_targets(case, oracle)
        inside = np.abs(ty) < np.pi / 2
        # the restated scan prunes on |dlat|, which is no bound for a target beyond a pole: compare those with the GPU only
        keep = inside | (np.abs(ty) == np.pi / 2) | (case["method"] == "kd")
        R.compare(ref, np.where(keep, wx, ref.ix), np.where(keep, wy, ref.iy), f"seed {seed} {case['family']} {case['method']}",
                  share_of=inside)


def test_kdtree_candidates_agree_with_brute_force(oracle, monkeypatch):
    """the cKDTree path (large cases) and the exhaustive path (small ones) give the same answers"""
    for seed in (3, 8, 19, 40, 41, 56):
        case = R.make_case(seed, max_src=3000, max_tgt=3000)
        a = R.reference_for(case, oracle)
        monkeypatch.setattr(R, "BRUTE_LIMIT", 0)
        b = R.reference_for(case, oracle)
        monkeypatch.undo()
        assert np.array_equal(a.ix, b.ix) and np.array_equal(a.iy, b.iy) and np.array_equal(a.amb, b.amb), seed


@pytest.mark.parametrize("method", ["nn", "kd"])
def test_target_on_a_source(method, oracle):
    lon = np.tile(10 + 0.5 * np.arange(6), 4)
    lat = np.repeat(60 + 0.3 * np.arange(4), 6)
    case = _designed(lon, lat, 6, 4, [11.5], [60.6], method, max_dist=1.0)
    ref = R.reference_for(case, oracle)
    wx, wy, _ = R.oracle_for(case, oracle)
    assert (ref.ix[0], ref.iy[0]) == (3, 2) == (wx[0], wy[0]) and not ref.amb[0]


@pytest.mark.parametrize("first", ["+0", "-0"])
def test_ties_both_directions(first, oracle):
    """exact ties: equal latitudes (-0 equal to +0) in insertion order scanning up, the last inserted scanning down, +a before -a
    around a target on the equator; coord_kdtree takes the lowest position"""
    lat = [0.0, -0.0] if first == "+0" else [-0.0, 0.0]
    for method in ("nn", "kd"):
        case = _designed([0.7, -0.7], lat, 2, 1, [0.0], [0.0], method, max_dist=500e3)
        ref = R.reference_for(case, oracle, exact_ties=True)
        wx, wy, ties = R.oracle_for(case, oracle)
        assert (ref.ix[0], wx[0]) == (0, 0) and not ref.amb[0] and ties == 1
        assert R.reference_for(case, oracle).amb[0]  # without the tie rule the reference does not decide
    for ya, want in (([38.5], 0), ([41.5], 1)):
        case = _designed([-0.9, 0.9], [40.0, 40.0], 2, 1, [0.0], ya, "nn")
        ref = R.reference_for(case, oracle, exact_ties=True)
        wx, wy, _ = R.oracle_for(case, oracle)
        assert ref.ix[0] == want == wx[0]
    case = _designed([10.0, 10.0], [-3.0, 3.0], 2, 1, [10.0], [0.0], "nn")
    assert R.reference_for(case, oracle, exact_ties=True).ix[0] == 1 == R.oracle_for(case, oracle)[0][0]


def test_one_valid_source_and_no_valid_sample(oracle):
    """one valid source: acos(-2) is NaN and every target gets (-1, -1).  All 53 samples NaN while other points are valid:
    acos(2), the same (the reference does not raise)."""
    lon = np.full(12, np.nan)
    lat = np.full(12, np.nan)
    lon[5], lat[5] = 3.0, 4.0
    case = _designed(lon, lat, 4, 3, [3.0, 3.1], [4.0], "nn")
    assert (R.reference_for(case, oracle).ix == -1).all() and (R.oracle_for(case, oracle)[0] == -1).all()
    nx, ny = 53, 20
    lon = np.tile(0.5 * np.arange(nx), ny)
    lat = np.repeat(0.5 * np.arange(ny), nx)
    lon[np.arange(53) * (nx * ny // 53)] = np.nan
    case = _designed(lon, lat, nx, ny, [3.1, 7.3], [2.2], "nn")
    assert np.isnan(R.grid_roi(R.to_rad(lon), R.to_rad(lat), nx, ny)[0])
    assert np.isnan(oracle.grid_distance(R.to_rad(lon), R.to_rad(lat), nx, ny))
    ref = R.reference_for(case, oracle)
    assert (ref.ix == -1).all() and not ref.amb.any() and (R.oracle_for(case, oracle)[0] == -1).all()


def test_sampling_switch_1000_1001(oracle):
    """an isolated point widens the ROI only when sampled: every point at nx*ny = 1000; at 1001 the points k*18"""
    mapped = {}
    for name, (sx, sy, iso) in {"1000": (40, 25, 55), "1001_sampled": (77, 13, 54), "1001_skipped": (77, 13, 55)}.items():
        lon = np.tile(10 + 0.1 * np.arange(sx), sy)
        lat = np.repeat(50 + 0.1 * np.arange(sy), sx)
        lon[iso], lat[iso] = 10 + 0.1 * sx + 5.0, 45.0
        xa = 10 + 0.1 * sx + 0.05 + 0.25 * np.arange(12) + 0.0123
        ya = 50 + 0.1 * sy * np.arange(3) / 2 + 0.0071
        case = _designed(lon, lat, sx, sy, xa, ya, "nn")
        ref = R.reference_for(case, oracle)
        wx, wy, _ = R.oracle_for(case, oracle)
        R.compare(ref, wx, wy, name)
        mapped[name] = int((ref.ix >= 0).sum())
    assert mapped["1000"] > mapped["1001_skipped"] and mapped["1001_sampled"] > mapped["1001_skipped"], mapped
    assert list(R.sample_positions(77, 13)[:4]) == [0, 18, 36, 54] and R.sample_positions(40, 25).size == 1000


def test_kd_radius_strict_and_whole_sphere(oracle):
    """chord squared exactly r*r is outside; r >= 2 reaches every source but one at exactly r = 2 on the antipode"""
    for md, want in ((12742e3, -1000), (float(np.nextafter(12742e3, np.inf)), 0)):
        case = _designed([180.0], [0.0], 1, 1, [0.0], [0.0], "kd", max_dist=md)
        ref = R.reference_for(case, oracle)
        assert R.oracle_for(case, oracle)[0][0] == want and ref.amb[0] and (want, want if want < 0 else 0) in ref.cand[0]
    rng = np.random.default_rng(9)
    lon, lat = rng.uniform(-180, 180, 200), rng.uniform(-80, 80, 200)
    case = _designed(lon, lat, 20, 10, np.linspace(-179, 179, 40), np.linspace(-85, 85, 30), "kd", max_dist=2e7)
    ref = R.reference_for(case, oracle)
    wx, wy, _ = R.oracle_for(case, oracle)
    R.compare(ref, wx, wy, "r > 2")
    assert (ref.ix >= 0).all()


def test_kd_latitude_window_known_answers(oracle):
    """a source beyond |dlat| = r but inside 2 asin(r / 2), and a target at latitude 95 on a source at (85, lon + 180)"""
    for lon, lat, ya, md in (([10.0, 100.0], [40.0, -30.0], [-19.0], 6371e3), ([-170.0, 0.0], [85.0, 0.0], [95.0], 100e3)):
        case = _designed(lon, lat, 2, 1, [10.0], ya, "kd", max_dist=md)
        ref = R.reference_for(case, oracle)
        wx, wy, _ = R.oracle_for(case, oracle)
        assert (ref.ix[0], ref.iy[0]) == (0, 0) == (wx[0], wy[0]) and not ref.amb[0]
