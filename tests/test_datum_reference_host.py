"""The datum-shift reference (tests/datum_reference.py) checked against known answers, and the CPU oracle's 3- and 7-parameter
datum shifts checked against the reference: random CRS pairs of all four projection families, the parser's handling of
+datum / +towgs84 / +ellps seen through the outputs, and the early exits that must leave a transform untouched."""
import numpy as np
import pytest

import datum_reference as ref
from datum_reference import Datum, figure, figure_of_ellps

ORACLE_BAR_DEG = 1e-11


# ---------------------------------------------------------------------------------------------------- the reference itself
@pytest.mark.parametrize("name", ["sphere", "WGS84", "bessel", "clrk66"])
def test_geodetic_ecef_round_trip(name):
    fig = figure_of_ellps(name)
    rng = np.random.default_rng(1)
    lat = np.concatenate([np.radians(rng.uniform(-90, 90, 4000)), np.radians([0.0, 90.0, -90.0, 89.9999999, -1e-12, 45.0])])
    lon = np.concatenate([np.radians(rng.uniform(-180, 180, 4000)), np.radians([0.0, 0.0, 0.0, 10.0, 180.0, -179.0])])
    lam, phi = ref.ecef_to_geodetic(fig, ref.geodetic_to_ecef(fig, lon, lat))
    assert np.abs(np.degrees(phi.astype(float) - lat)).max() <= 1e-13
    off_axis = np.abs(lat) < np.radians(89.99)
    dl = np.remainder(lam.astype(float) - lon + np.pi, 2 * np.pi) - np.pi
    assert np.abs(np.degrees(dl[off_axis]) * np.cos(lat[off_axis])).max() <= 1e-13
    assert (lam[np.abs(lat) == np.pi / 2] == 0).all()  # on the polar axis the longitude is 0


def test_sphere_known_answers():
    r1, r2 = figure(6371000.0), figure(6400000.0)
    rng = np.random.default_rng(2)
    lon, lat = np.radians(rng.uniform(-180, 180, 500)), np.radians(rng.uniform(-89, 89, 500))
    # sphere R1 -> sphere R2 with zero shifts: a radial move, the direction is kept
    lo, la = ref.shift(r1, Datum((0.0, 0.0, 0.0)), r2, Datum((0.0, 0.0, 0.0)), lon, lat)
    assert np.abs(la - lat).max() < 1e-14 and np.abs(np.remainder(lo - lon + np.pi, 2 * np.pi) - np.pi).max() < 1e-14
    # a pure translation (0, dy, 0) at (0, 0): lon = atan2(dy, R), lat = 0
    for dy in (1000.0, -2.5e5):
        lo, la = ref.shift(r1, Datum((0.0, dy, 0.0)), r1, Datum((0.0, 0.0, 0.0)), [0.0], [0.0])
        assert abs(lo[0] - np.arctan2(dy, 6371000.0)) < 1e-16 and la[0] == 0.0
    # a pure scale: the direction is kept
    lo, la = ref.shift(r1, Datum((0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 250.0)), r1, Datum((0.0, 0.0, 0.0)), lon, lat)
    assert np.abs(la - lat).max() < 1e-14 and np.abs(np.remainder(lo - lon + np.pi, 2 * np.pi) - np.pi).max() < 1e-14
    # a pure rz: the longitude moves by atan(rz); the small-angle matrix also stretches the equatorial plane by
    # sqrt(1 + rz^2), so tan(lat) shrinks by that factor
    rz = 7.5  # arc-seconds
    lo, la = ref.shift(r1, Datum((0.0, 0.0, 0.0, 0.0, 0.0, rz)), r1, Datum((0.0, 0.0, 0.0)), lon, lat)
    t = rz * np.pi / (180 * 3600)
    assert np.abs(np.remainder(lo - lon - np.arctan(t) + np.pi, 2 * np.pi) - np.pi).max() < 1e-14
    assert np.abs(la - np.arctan2(np.sin(lat), np.cos(lat) * np.sqrt(1 + t * t))).max() < 1e-14


def test_sphere_to_wgs84_is_the_geocentric_latitude_difference():
    """a zero shift from a sphere to WGS84 keeps each point's direction from the centre: the latitude becomes the geodetic
    latitude of a geocentric one.  Equator and poles stay; the change peaks near 45 degrees at about f = 1/298.26 rad (the
    textbook 11.5 arc-minutes)"""
    lat = np.radians(np.linspace(-90, 90, 18001))
    lon = np.zeros_like(lat)
    lo, la = ref.shift(figure(6371000.0), Datum((0.0, 0.0, 0.0)), figure_of_ellps("WGS84"), Datum((0.0, 0.0, 0.0)), lon, lat)
    d = np.degrees(la - lat)
    assert d[0] == 0 and d[-1] == 0 and abs(d[9000]) < 1e-15
    i = np.argmax(np.abs(d))
    assert 44.5 < abs(np.degrees(lat[i])) < 45.5
    assert abs(abs(d[i]) - np.degrees(1 / 298.257223563)) < 0.0015, d[i]


def test_proj_inverse_rotation_is_second_order():
    """R^T (PROJ's from-WGS84 step) against the exact inverse of R = I + W: the gap is W^2 (I + W)^-1 X, within theta^2 |X|"""
    rng = np.random.default_rng(3)
    for _ in range(20):
        rot = rng.uniform(-60, 60, 3)
        theta = np.linalg.norm(rot) * np.pi / (180 * 3600)
        r = ref.rotation(*rot).astype(np.float64)
        x = rng.normal(0, 6.4e6, (3, 50))
        gap = np.linalg.norm(r.T @ x - np.linalg.solve(r, x), axis=0)
        bound = theta**2 * np.linalg.norm(x, axis=0)
        assert (gap <= bound * (1 + 1e-6) + 1e-8).all()
        assert (gap > 0.01 * bound).any()  # second order, not zero: the two definitions really differ


# ---------------------------------------------------------------------------------------------------- the oracle against it
@pytest.mark.parametrize("seed", range(300))
def test_oracle_against_reference_fuzz(oracle, seed):
    src, dst, lon, lat = ref.fuzz_case(7000 + seed)
    sx, sy, glon, glat = ref.source_points(oracle.project_values, src, lon, lat)
    ref.check(oracle.project_values, src, dst, sx, sy, glon, glat, ORACLE_BAR_DEG, f"seed {seed}")


@pytest.mark.parametrize("case", range(3))
def test_oracle_edge_inputs(oracle, case):
    src, dst, lon, lat = ref.edge_cases()[case]
    rc, gx, gy = oracle.project_values(src.proj, dst.proj, np.radians(lon), np.radians(lat))
    assert rc == 1
    rlon, rlat = ref.shift(src.fig, src.datum, dst.fig, dst.datum, np.radians(lon), np.radians(lat))
    assert np.array_equal(np.isfinite(gx), np.isfinite(rlon)) and np.array_equal(np.isfinite(gy), np.isfinite(rlat))
    ok = np.isfinite(rlon)
    assert (np.abs(gx[ok]) <= np.pi).all()  # atan2: (-pi, pi] whatever the input range
    assert ref.arc_error_deg(oracle.project_values, dst, gx[ok], gy[ok], rlon[ok], rlat[ok]).max() <= ORACLE_BAR_DEG
    pole = ok & (np.abs(np.abs(rlat) - np.pi / 2) < 1e-15)
    assert (gx[pole] == 0).all() and (np.abs(gy[pole]) == np.pi / 2).all()


def test_parser_first_key_wins_and_datum_figures(oracle):
    ref.check_first_key_wins_and_datum_figures(oracle.project_values, ORACLE_BAR_DEG)


def test_datum_ellipsoid_shape_overrides_a_users_b(oracle):
    """`+a +b +datum=WGS84` is (a, WGS84's 1/f): modelling it from the user's +b instead misses the oracle by more than
    the bar, so the precedence the reference states is one the tests can tell apart"""
    lon, lat = ref.points(15)
    intl = ref.latlong_crs("+ellps=intl", figure_of_ellps("intl"), (-87.0, -98.0, -121.0))
    wrong = ref.Crs("+proj=latlong +a=6378137 +b=6356752.3142 +datum=WGS84 +no_defs", "", "", figure(6378137.0, b=6356752.3142),
                    Datum((0.0, 0.0, 0.0)), "ll")
    rc, gx, gy = oracle.project_values(wrong.proj, intl.proj, lon, lat)
    assert rc == 1
    rlon, rlat = ref.shift(wrong.fig, wrong.datum, intl.fig, intl.datum, lon, lat)
    assert np.nanmax(ref.arc_error_deg(oracle.project_values, intl, gx, gy, rlon, rlat)) > 10 * ORACLE_BAR_DEG


def test_parser_towgs84_forms(oracle):
    ref.check_towgs84_forms(oracle.project_values, ORACLE_BAR_DEG)


def test_parser_refuses_grid_shifts_and_unknown_datums(oracle):
    lon, lat = ref.points(13, 4)
    for bad in ("+proj=latlong +ellps=WGS84 +nadgrids=@null +no_defs", "+proj=latlong +datum=ED50 +no_defs",
                "+proj=stere +lat_0=90 +lon_0=0 +R=6371000 +nadgrids=ntv1_can.dat +no_defs"):
        assert oracle.project_values(bad, "+proj=latlong +datum=WGS84 +no_defs", lon, lat)[0] != 1, bad
        assert oracle.project_values("+proj=latlong +datum=WGS84 +no_defs", bad, lon, lat)[0] != 1, bad


@pytest.mark.parametrize("case", range(len(ref.IDENTITY)))
def test_oracle_identity_cases_are_bitwise_datum_free(oracle, case):
    src, dst = ref.IDENTITY[case]
    x, y = ref.identity_inputs(oracle.project_values, src)
    a = oracle.project_values(src, dst, x, y)
    b = oracle.project_values(ref.strip_datum(src), ref.strip_datum(dst), x, y)
    assert a[0] == b[0] == 1
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64)) and np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
