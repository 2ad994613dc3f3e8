"""Independent reference for the 3- and 7-parameter datum shift of the coordinate transforms (test infrastructure only).

Written from the geodesy, not from `oracle/pj_oracle.c` or `fimex_b200/csrc/proj.cuh`.  It does not parse proj strings:
the tests describe each CRS once, as a structured figure + datum, and build both the proj string and this module's
arguments from that description, so the parsers are checked too.

Geodesy (all arithmetic in `np.longdouble`):

  * Figure: semi-major axis `a` and squared eccentricity e^2 = f (2 - f) (from 1/f) or 1 - b^2/a^2 (from the minor axis);
    a sphere has e^2 = 0.  `ELLIPSOIDS` holds the defining constants of the `+ellps=` names the parser knows.
  * Geodetic -> ECEF at height 0: N = a / sqrt(1 - e^2 sin^2 phi), X = N cos phi cos lam, Y = N cos phi sin lam,
    Z = N (1 - e^2) sin phi.
  * To WGS84: the position-vector Helmert transform (EPSG method 9606) as a matrix product X' = T + (1 + s 1e-6) R X, with
    R = I + W the small-angle rotation, W = [[0, -rz, ry], [rz, 0, -rx], [-ry, rx, 0]], rx, ry, rz in arc-seconds.
  * From WGS84: PROJ 4's definition X = R^T (X' - T) / (1 + s 1e-6).  R^T is not R^-1: the two differ by
    W^2 (I + W)^-1, second order in the angles (bounded in tests/test_datum_reference_host.py).
  * ECEF -> geodetic: Heikkinen's closed form (1982; as in Zhu, IEEE AES 30 (1994) 957), polished by Newton steps on
    f(phi) = p sin phi - Z cos phi - e^2 N(phi) sin phi cos phi, the condition that (p, Z) lies on the normal at phi.

Conventions, as PROJ 4.9 behaves (pj_transform.c, pj_datum_set.c, geocent.c):

  * longitude = atan2(Y, X): after a shift it lies in (-pi, pi] whatever the input range;
  * on the polar axis (p / a < 1e-12) the longitude is 0;
  * |phi| in (pi/2, 1.001 pi/2) is clamped to +-pi/2; beyond that the point fails (HUGE_VAL, returned here as inf);
  * the shift uses the figure as given -- `a_orig`, `es_orig` -- also for ob_tran, which projects on a sphere;
  * early exits: no shift if either side has no datum, or if both datums compare equal (same kind, same a,
    |delta e^2| <= 5e-11, same parameters).  A zero 3-parameter shift on a figure with a = 6378137 and e^2 within 5e-11 of
    WGS84's counts as WGS84 (so `+datum=NAD83`, GRS80 + zero shift, equals `+datum=WGS84`).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

LD = np.longdouble
HALFPI = np.pi / 2  # the float64 value the clamp compares against
SEC2RAD = LD(np.pi) / LD(180 * 3600)

# +ellps= constants (PROJ's ellipsoid table): name -> (a, shape key, value)
ELLIPSOIDS = {
    "sphere": (6370997.0, "b", 6370997.0),
    "WGS84": (6378137.0, "rf", 298.257223563),
    "GRS80": (6378137.0, "rf", 298.257222101),
    "bessel": (6377397.155, "rf", 299.1528128),
    "intl": (6378388.0, "rf", 297.0),
    "clrk66": (6378206.4, "b", 6356583.8),
    "krass": (6378245.0, "rf", 298.3),
}

UNKNOWN, THREE, SEVEN, WGS84 = "unknown", "3param", "7param", "wgs84"


@dataclass(frozen=True)
class Figure:
    a: float
    es: float  # float64 value of e^2 (the longdouble value below is what the geodesy uses)
    es_ld: LD


def figure(a, rf=None, b=None) -> Figure:
    """sphere of radius a (neither rf nor b), or the ellipsoid of semi-major axis a and reciprocal flattening rf / minor axis b"""
    la = LD(a)
    if rf is not None:
        f = LD(1) / LD(rf)
        es = f * (LD(2) - f)
    elif b is not None:
        es = LD(1) - (LD(b) * LD(b)) / (la * la)
    else:
        es = LD(0)
    return Figure(float(a), float(es), es)


def figure_of_ellps(name) -> Figure:
    a, key, val = ELLIPSOIDS[name]
    return figure(a, **{key: val})


@dataclass(frozen=True)
class Datum:
    """None for a CRS without a datum; else the towgs84 values as written (m, arc-seconds, ppm), 3 or 7 of them"""
    towgs84: tuple | None

    def params(self):
        p = tuple(float(v) for v in self.towgs84) + (0.0,) * (7 - len(self.towgs84))
        return p[:7]


def datum_kind(fig: Figure, d: Datum) -> str:
    if d.towgs84 is None:
        return UNKNOWN
    p = d.params()
    if any(v != 0.0 for v in p[3:]):
        return SEVEN
    if p[:3] == (0.0, 0.0, 0.0) and fig.a == 6378137.0 and abs(fig.es - 0.006694379990) < 5e-11:
        return WGS84
    return THREE


def needs_shift(sfig: Figure, sd: Datum, dfig: Figure, dd: Datum) -> bool:
    ks, kd = datum_kind(sfig, sd), datum_kind(dfig, dd)
    if ks == UNKNOWN or kd == UNKNOWN:
        return False
    if ks == kd and sfig.a == dfig.a and abs(sfig.es - dfig.es) <= 5e-11:
        if ks == THREE and sd.params()[:3] == dd.params()[:3]:
            return False
        if ks == SEVEN and sd.params() == dd.params():
            return False
        if ks == WGS84:
            return False
    return sfig.a != dfig.a or sfig.es != dfig.es or ks in (THREE, SEVEN) or kd in (THREE, SEVEN)


def geodetic_to_ecef(fig: Figure, lon, lat):
    lam, phi = np.asarray(lon, dtype=LD), np.asarray(lat, dtype=LD)
    s, c = np.sin(phi), np.cos(phi)
    n = LD(fig.a) / np.sqrt(LD(1) - fig.es_ld * s * s)
    return np.stack([n * c * np.cos(lam), n * c * np.sin(lam), n * (LD(1) - fig.es_ld) * s])


def rotation(rx, ry, rz):
    """R = I + W for rotations in arc-seconds (position-vector convention)"""
    x, y, z = (LD(v) * SEC2RAD for v in (rx, ry, rz))
    one = LD(1)
    return np.array([[one, -z, y], [z, one, -x], [-y, x, one]], dtype=LD)


def helmert_to_wgs84(d: Datum, xyz):
    tx, ty, tz, rx, ry, rz, s = d.params()
    t = np.array([tx, ty, tz], dtype=LD).reshape(3, 1)
    m = LD(1) + LD(s) * LD(1e-6)
    return t + m * (rotation(rx, ry, rz) @ xyz)


def helmert_from_wgs84(d: Datum, xyz):
    """PROJ 4's definition of the inverse step: X = R^T (X' - T) / (1 + s 1e-6)"""
    tx, ty, tz, rx, ry, rz, s = d.params()
    t = np.array([tx, ty, tz], dtype=LD).reshape(3, 1)
    m = LD(1) + LD(s) * LD(1e-6)
    return (rotation(rx, ry, rz).T @ (xyz - t)) / m


def ecef_to_geodetic(fig: Figure, xyz, newton=3):
    """(lon, lat) in radians as longdouble; Heikkinen's closed form, then Newton on the normal condition"""
    X, Y, Z = (np.asarray(v, dtype=LD) for v in xyz)
    a, e2 = LD(fig.a), fig.es_ld
    b2 = a * a * (LD(1) - e2)
    p = np.sqrt(X * X + Y * Y)
    if e2 == 0:
        phi = np.arctan2(Z, p)
    else:
        b = np.sqrt(b2)
        ep2 = (a * a - b2) / b2
        F = LD(54) * b2 * Z * Z
        G = p * p + (LD(1) - e2) * Z * Z - e2 * (a * a - b2)
        c = e2 * e2 * F * p * p / (G * G * G)
        s = np.cbrt(LD(1) + c + np.sqrt(c * c + LD(2) * c))
        k = s + LD(1) + LD(1) / s
        P = F / (LD(3) * k * k * G * G)
        Q = np.sqrt(LD(1) + LD(2) * e2 * e2 * P)
        r0 = -(P * e2 * p) / (LD(1) + Q) + np.sqrt(np.maximum(
            LD(0.5) * a * a * (LD(1) + LD(1) / Q) - P * (LD(1) - e2) * Z * Z / (Q * (LD(1) + Q)) - LD(0.5) * P * p * p, LD(0)))
        V = np.sqrt((p - e2 * r0) ** 2 + (LD(1) - e2) * Z * Z)
        z0 = b2 * Z / (a * V)
        phi = np.arctan2(Z + ep2 * z0, p)
        for _ in range(newton):
            sp, cp = np.sin(phi), np.cos(phi)
            w = LD(1) - e2 * sp * sp
            n = a / np.sqrt(w)
            f = p * sp - Z * cp - e2 * n * sp * cp
            dn = n * e2 * sp * cp / w
            df = p * cp + Z * sp - e2 * (dn * sp * cp + n * (cp * cp - sp * sp))
            phi = phi - f / df
    lam = np.where(p / a < LD(1e-12), LD(0), np.arctan2(Y, X))
    return lam, phi


def shift(sfig: Figure, sd: Datum, dfig: Figure, dd: Datum, lon, lat):
    """geodetic (lon, lat) in radians on the source datum -> the destination datum, float64; failed points are inf.
    Without a shift (see `needs_shift`) the input comes back unchanged."""
    lon = np.array(lon, dtype=np.float64, copy=True)
    lat = np.array(lat, dtype=np.float64, copy=True)
    if not needs_shift(sfig, sd, dfig, dd):
        return lon, lat
    live = np.isfinite(lon) & np.isfinite(lat)
    clamp = live & (np.abs(lat) > HALFPI) & (np.abs(lat) < 1.001 * HALFPI)
    lat[clamp] = np.copysign(HALFPI, lat[clamp])
    bad = live & (np.abs(lat) > HALFPI)
    ok = live & ~bad
    xyz = geodetic_to_ecef(sfig, lon[ok], lat[ok])
    if datum_kind(sfig, sd) in (THREE, SEVEN):
        xyz = helmert_to_wgs84(sd, xyz)
    if datum_kind(dfig, dd) in (THREE, SEVEN):
        xyz = helmert_from_wgs84(dd, xyz)
    lam, phi = ecef_to_geodetic(dfig, xyz)
    lon[ok], lat[ok] = lam.astype(np.float64), phi.astype(np.float64)
    lon[bad] = lat[bad] = np.inf
    return lon, lat


# ---------------------------------------------------------------------------------------------------------------------
# Test cases: a CRS is described once (projection part, figure, datum) and both the proj string and the reference's
# arguments are built from that description.
# ---------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Crs:
    proj: str  # the full proj4 string
    plain: str  # the same CRS on the same figure with no datum (what the comparisons project through)
    geographic: str  # lat/long on the same figure with no datum
    fig: Figure
    datum: Datum
    family: str  # "ll", "rot" or "m"


def _fmt(v):
    return repr(float(v)).rstrip("0").rstrip(".") if float(v) != int(v) else str(int(v))


def towgs84_token(values):
    return "+towgs84=" + ",".join(_fmt(v) for v in values)


FIGURES = [  # (tokens, figure); the tokens name the figure and nothing else
    ("+R=6371000", figure(6371000.0)),
    ("+a=6378137 +b=6356752.3142", figure(6378137.0, b=6356752.3142)),
    ("+a=6377563.396 +rf=299.3249646", figure(6377563.396, rf=299.3249646)),
] + [(f"+ellps={n}", figure_of_ellps(n)) for n in ELLIPSOIDS]

REALISTIC = [(598.1, 73.7, 418.2, 0.202, 0.045, -2.455, 6.7), (446.448, -125.157, 542.06, 0.15, 0.247, 0.842, -20.489),
             (-87.0, -98.0, -121.0), (24.0, -123.0, -94.0), (-168.0, -60.0, 320.0), (23.92, -141.27, -80.9, 0.0, 0.35, 0.82, -0.12)]


def random_datum(rng):
    """(tokens, Datum) for a figure given by explicit tokens"""
    r = rng.integers(0, 9)
    if r == 0:
        return "", Datum(None)
    if r == 1:
        v = REALISTIC[rng.integers(0, len(REALISTIC))]
        return towgs84_token(v), Datum(tuple(v))
    if r == 2:  # realistic-sized 3-parameter
        v = tuple(np.round(rng.uniform(-600, 600, 3), 3))
        return towgs84_token(v), Datum(v)
    if r == 3:  # realistic-sized 7-parameter
        v = tuple(np.round(np.concatenate([rng.uniform(-600, 600, 3), rng.uniform(-3, 3, 3), rng.uniform(-12, 12, 1)]), 4))
        return towgs84_token(v), Datum(v)
    if r == 4:  # exaggerated
        v = tuple(np.round(np.concatenate([rng.uniform(-5e3, 5e3, 3), rng.uniform(-200, 200, 3), rng.uniform(-500, 500, 1)]), 3))
        return towgs84_token(v), Datum(v)
    if r == 5:  # zero shift (a WGS84 datum on a WGS84 / GRS80 figure, a 3-parameter datum on any other)
        return "+towgs84=0,0,0", Datum((0.0, 0.0, 0.0))
    if r == 6:  # seven values with zero rotations and scale: a 3-parameter shift
        v = tuple(np.round(rng.uniform(-300, 300, 3), 2)) + (0.0, 0.0, 0.0, 0.0)
        return towgs84_token(v), Datum(v)
    if r == 7:  # fewer than three values
        v = tuple(np.round(rng.uniform(-300, 300, int(rng.integers(1, 3))), 2))
        return towgs84_token(v), Datum(v)
    return "+datum=WGS84", Datum((0.0, 0.0, 0.0))  # after the figure's tokens: a zero 3-parameter shift on that figure


def figure_behind_datum(fig_t, fig, ellps):
    """(tokens, figure) that PROJ ends up with when `+datum=` appends `+ellps=<ellps>` behind the figure tokens `fig_t`.
    +R wins over everything and the first +ellps wins, but pj_ell_set reads the shape in the order es, e, rf, f, b
    after the ellipsoid's own +a and +rf / +b have been appended: the user's +a stays (first occurrence), while an
    ellipsoid's +rf overrides a user's +f or +b"""
    keys = [t.split("=")[0] for t in fig_t.split()]
    _, key, val = ELLIPSOIDS[ellps]
    if any(k in keys for k in ("+R", "+ellps", "+es", "+e", "+rf")) or key != "rf":
        return fig_t, fig
    a_tok = next(t for t in fig_t.split() if t.startswith("+a="))
    return f"{a_tok} +rf={_fmt(val)}", figure(fig.a, rf=val)


def random_crs(rng) -> Crs:
    """one of the four projection families with a random figure and datum"""
    d = rng.integers(0, 10)
    if d == 0:
        fig_t, fig, dat_t, dat = "", figure_of_ellps("WGS84"), "+datum=WGS84", Datum((0.0, 0.0, 0.0))
        plain_fig = "+ellps=WGS84"
    elif d == 1:
        fig_t, fig, dat_t, dat = "", figure_of_ellps("GRS80"), "+datum=NAD83", Datum((0.0, 0.0, 0.0))
        plain_fig = "+ellps=GRS80"
    else:
        fig_t, fig = FIGURES[rng.integers(0, len(FIGURES))]
        dat_t, dat = random_datum(rng)
        plain_fig = fig_t
        if dat_t == "+datum=WGS84":
            plain_fig, fig = figure_behind_datum(fig_t, fig, "WGS84")
    earth = " ".join(t for t in (fig_t, dat_t) if t)
    kind = rng.integers(0, 4)
    if kind == 0:
        head, fam = "+proj=latlong", "ll"
    elif kind == 1:
        head, fam = (f"+proj=ob_tran +o_proj=longlat +lon_0={rng.uniform(-180, 180):.4f} +o_lat_p={rng.uniform(5, 85):.4f} "
                     f"+o_lon_p={rng.choice([0, 0, 10.5, -170])}"), "rot"
    elif kind == 2:
        lat0 = rng.choice([90, -90, 60.0, 0.0, -37.5])
        ts = f"+lat_ts={rng.uniform(40, 80) * np.sign(lat0 if lat0 else 1):.3f}" if abs(lat0) == 90 and rng.random() < 0.7 else \
            f"+k={rng.uniform(0.9, 1.0):.5f}"
        head, fam = f"+proj=stere +lat_0={lat0} +lon_0={rng.uniform(-180, 180):.3f} {ts} +x_0={rng.choice([0, 7000, -2.5e5])}", "m"
    else:
        lat1 = rng.uniform(20, 70) * rng.choice([1, -1])
        lat2 = lat1 if rng.random() < 0.4 else lat1 + rng.uniform(-15, 15)
        head, fam = (f"+proj=lcc +lat_1={lat1:.3f} +lat_2={lat2:.3f} +lat_0={lat1 + rng.uniform(-5, 5):.3f} "
                     f"+lon_0={rng.uniform(-180, 180):.3f}"), "m"
    no_defs = " +no_defs" if rng.random() < 0.7 else ""
    return Crs(f"{head} {earth}{no_defs}", f"{head} {plain_fig} +no_defs", f"+proj=latlong {plain_fig} +no_defs", fig, dat, fam)



def fuzz_case(seed, n=600):
    """a random CRS pair and geographic points (radians) on the source figure, away from the poles"""
    rng = np.random.default_rng(seed)
    src, dst = random_crs(rng), random_crs(rng)
    lon = np.radians(rng.uniform(-179.5, 179.5, n))
    lat = np.radians(rng.uniform(-85.0, 85.0, n))
    return src, dst, lon, lat


def source_points(project, src: Crs, lon, lat):
    """(sx, sy): the points in src's own coordinates (no datum involved), and (glon, glat): their inverse through `project`,
    the geodetic input of the shift that the transform under test sees"""
    if src.family == "ll":
        return lon, lat, lon, lat
    rc, sx, sy = project(src.geographic, src.plain, lon, lat)
    assert rc == 1, src.plain
    ok = np.isfinite(sx) & np.isfinite(sy)
    sx, sy = sx[ok], sy[ok]
    rc, glon, glat = project(src.plain, src.geographic, sx, sy)
    assert rc == 1, src.plain
    return sx, sy, glon, glat


def arc_error_deg(project, dst: Crs, gx, gy, rlon, rlat):
    """per point distance in degrees of arc between a result (gx, gy) in dst's coordinates and the reference's geodetic
    (rlon, rlat) on dst's figure.  Lat/long: directly.  Otherwise in the geographic domain: dst's forward projection
    (through `project`, no datum) linearised at the reference point maps the coordinate difference back to (dlon, dlat).
    Where exactly one of the result and the (projected) reference is not finite the error is inf; where both are not,
    NaN."""
    got_ok = np.isfinite(gx) & np.isfinite(gy)
    if dst.family == "ll":
        dx = np.remainder(gx - rlon + np.pi, 2 * np.pi) - np.pi
        return _mask(np.degrees(np.hypot(dx * np.cos(rlat), gy - rlat)), got_ok, np.isfinite(rlon) & np.isfinite(rlat))
    wrap = dst.family == "rot"

    def d(u, v):
        r = u - v
        return np.remainder(r + np.pi, 2 * np.pi) - np.pi if wrap else r

    def fwd(lo, la):
        rc, x, y = project(dst.geographic, dst.plain, lo, la)
        assert rc == 1, dst.plain
        return x, y

    h = 1e-7
    fx, fy = fwd(rlon, rlat)
    xe, ye = fwd(rlon + h, rlat)
    xw, yw = fwd(rlon - h, rlat)
    xn, yn = fwd(rlon, rlat + h)
    xs, ys = fwd(rlon, rlat - h)
    j00, j01, j10, j11 = d(xe, xw) / (2 * h), d(xn, xs) / (2 * h), (ye - yw) / (2 * h), (yn - ys) / (2 * h)
    with np.errstate(invalid="ignore"):  # failed points: masked below
        ex, ey = d(gx, fx), gy - fy
        det = j00 * j11 - j01 * j10
        dlon = (j11 * ex - j01 * ey) / det
        dlat = (-j10 * ex + j00 * ey) / det
        out = np.degrees(np.hypot(dlon * np.cos(rlat), dlat))
    return _mask(out, got_ok, np.isfinite(fx) & np.isfinite(fy))


def _mask(err, got_ok, ref_ok):
    err = np.where(got_ok & ref_ok, err, np.nan)
    err[got_ok != ref_ok] = np.inf
    return err


def strip_datum(proj: str) -> str:
    return " ".join(t for t in proj.split() if t.split("=")[0] not in ("+datum", "+towgs84"))


# Edge inputs through lat/long sources that carry a shift: (source Crs, destination Crs, lon degrees, lat degrees)
def edge_cases():
    intl7 = (-87.0, -98.0, -121.0, 0.4, -0.3, 0.8, 1.5)
    src = Crs(f"+proj=latlong +ellps=intl {towgs84_token(intl7)} +no_defs", "+proj=latlong +ellps=intl +no_defs",
              "+proj=latlong +ellps=intl +no_defs", figure_of_ellps("intl"), Datum(intl7), "ll")
    wgs = Crs("+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs", "+proj=latlong +ellps=WGS84 +no_defs",
              "+proj=latlong +ellps=WGS84 +no_defs", figure_of_ellps("WGS84"), Datum((0.0, 0.0, 0.0)), "ll")
    clamp = 1.001 * 90.0
    lat = [90.0, -90.0, 90.0 + 1e-9, 90.03, clamp - 1e-7, -90.05, -(clamp - 1e-7),  # clamped to the pole
           clamp + 1e-7, 90.2, 135.0, -(clamp + 1e-7), -100.0,  # fail
           45.0, 45.0, 45.0, -30.0, 0.0, 0.0, 60.0]
    lon = [0.0, 77.0, 12.0, -45.0, 170.0, 10.0, -120.0,
           0.0, 5.0, 5.0, 0.0, 0.0,
           200.0, 359.9, -200.0, 180.0, -180.0, 180.0, -359.9]
    sph_z = Crs("+proj=latlong +R=6371000 +towgs84=0,0,120 +no_defs", "+proj=latlong +R=6371000 +no_defs",
                "+proj=latlong +R=6371000 +no_defs", figure(6371000.0), Datum((0.0, 0.0, 120.0)), "ll")
    sph_0 = Crs("+proj=latlong +R=6371000 +towgs84=0,0,0 +no_defs", "+proj=latlong +R=6371000 +no_defs",
                "+proj=latlong +R=6371000 +no_defs", figure(6371000.0), Datum((0.0, 0.0, 0.0)), "ll")
    return [(src, wgs, np.array(lon), np.array(lat)),
            (wgs, src, np.array(lon), np.array(lat)),
            (sph_z, sph_0, np.array([0.0, 33.0, -150.0, 10.0, 10.0]), np.array([90.0, -90.0, 90.0, 90.05, -90.05]))]


def latlong_crs(fig_tokens, fig, towgs84=None) -> Crs:
    tok = f" {towgs84_token(towgs84)}" if towgs84 is not None else ""
    plain = f"+proj=latlong {fig_tokens} +no_defs"
    return Crs(f"+proj=latlong {fig_tokens}{tok} +no_defs", plain, plain, fig, Datum(towgs84), "ll")


def check(project, src, dst, sx, sy, glon, glat, bar_deg, what=""):
    """`project`(src.proj, dst.proj, sx, sy) within `bar_deg` of arc of the reference shift of (glon, glat); returns the result"""
    rc, gx, gy = project(src.proj, dst.proj, sx, sy)
    assert rc == 1, (src.proj, dst.proj)
    rlon, rlat = shift(src.fig, src.datum, dst.fig, dst.datum, glon, glat)
    err = arc_error_deg(project, dst, gx, gy, rlon, rlat)
    differ = np.flatnonzero(np.isinf(err))
    assert differ.size == 0, (what, src.proj, dst.proj, "failure masks differ from the reference's at", differ[:5])
    worst = np.nanmax(err, initial=0.0)
    assert worst <= bar_deg, (what, src.proj, dst.proj, worst)
    return gx, gy


# transforms that must not shift: each equals, bit for bit, the same transform with the datum tokens removed
IDENTITY = [
    # WGS84 <-> NAD83: both are the WGS84 datum (GRS80 differs from WGS84 by 3.3e-11 in e^2, inside the 5e-11 of the comparison)
    ("+proj=stere +lat_0=90 +lon_0=-32 +lat_ts=60 +ellps=GRS80 +datum=NAD83", "+proj=lcc +lat_1=40 +lat_2=60 +lon_0=10 +datum=WGS84"),
    ("+proj=latlong +ellps=WGS84 +datum=WGS84 +no_defs", "+proj=latlong +ellps=GRS80 +datum=NAD83 +no_defs"),
    # identical +towgs84 on both sides
    ("+proj=latlong +ellps=intl +towgs84=-87,-98,-121 +no_defs", "+proj=stere +lat_0=50 +lon_0=5 +ellps=intl +towgs84=-87,-98,-121"),
    ("+proj=lcc +lat_1=50 +lon_0=10 +ellps=bessel +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7",
     "+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +ellps=bessel +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7"),
    # a datum on one side only
    ("+proj=latlong +ellps=bessel +towgs84=598.1,73.7,418.2,0.202,0.045,-2.455,6.7 +no_defs", "+proj=latlong +ellps=WGS84 +no_defs"),
    ("+proj=stere +lat_0=90 +lon_0=0 +R=6371000 +no_defs", "+proj=latlong +R=6371000 +towgs84=100,0,0 +no_defs"),
    ("+proj=latlong +a=6378137 +b=6356752.3142 +no_defs", "+proj=lcc +lat_1=40 +lat_2=60 +lon_0=10 +ellps=krass +towgs84=24,-123,-94"),
]


def identity_inputs(project, src):
    """geographic points carried into `src`'s coordinates without a datum"""
    rng = np.random.default_rng(14)
    lon, lat = np.radians(rng.uniform(-180, 180, 500)), np.radians(rng.uniform(-89, 89, 500))
    if not src.startswith("+proj=latlong"):
        g = "+proj=latlong " + " ".join(t for t in src.split() if t.split("=")[0] in ("+R", "+a", "+b", "+rf", "+ellps"))
        rc, lon, lat = project(g, strip_datum(src), lon, lat)
        assert rc == 1
        ok = np.isfinite(lon)
        lon, lat = lon[ok], lat[ok]
    return lon, lat


GEO = [("+R=6371000", figure(6371000.0)), ("+ellps=bessel", figure_of_ellps("bessel")), ("+ellps=krass", figure_of_ellps("krass")),
       ("+a=6378137 +b=6356752.3142", figure(6378137.0, b=6356752.3142))]


def points(seed, n=400):
    rng = np.random.default_rng(seed)
    return np.radians(rng.uniform(-180, 180, n)), np.radians(rng.uniform(-89, 89, n))


def check_first_key_wins_and_datum_figures(project, bar):
    """+ellps / +datum precedence, seen through the outputs"""
    lon, lat = points(11)
    wgs = latlong_crs("+ellps=WGS84", figure_of_ellps("WGS84"), (0.0, 0.0, 0.0))
    # +ellps=bessel +datum=WGS84: the datum's +ellps comes after the user's, so this is a zero 3-parameter shift on Bessel
    src = Crs("+proj=latlong +ellps=bessel +datum=WGS84 +no_defs", "", "", figure_of_ellps("bessel"), Datum((0.0, 0.0, 0.0)), "ll")
    check(project, src, wgs, lon, lat, lon, lat, bar, "bessel + datum=WGS84")
    rc, x, y = project(src.proj, wgs.proj, lon, lat)
    assert np.abs(y - lat).max() > 1e-6  # the figure changed: a real shift happened
    # +a +b +datum=WGS84: the user's +a is found first, but the shape is read as es, e, rf, f, b, so the +rf the datum's
    # ellipsoid appends overrides the user's +b; the figure is (a, WGS84's 1/f)
    intl = latlong_crs("+ellps=intl", figure_of_ellps("intl"), (-87.0, -98.0, -121.0))
    ab = Crs("+proj=latlong +a=6378137 +b=6356752.3142 +datum=WGS84 +no_defs", "", "",
             figure_behind_datum("+a=6378137 +b=6356752.3142", figure(6378137.0, b=6356752.3142), "WGS84")[1], Datum((0.0, 0.0, 0.0)), "ll")
    assert ab.fig == figure_of_ellps("WGS84")
    check(project, ab, intl, lon, lat, lon, lat, bar, "+a +b +datum=WGS84")
    check(project, intl, ab, lon, lat, lon, lat, bar, "to +a +b +datum=WGS84")
    # +datum=NAD83 alone is GRS80 (PROJ does not default +ellps when +datum is given), with and without +no_defs
    bessel7 = latlong_crs("+ellps=bessel", figure_of_ellps("bessel"), REALISTIC[0])
    for tail in (" +no_defs", ""):
        nad = Crs("+proj=latlong +datum=NAD83" + tail, "", "", figure_of_ellps("GRS80"), Datum((0.0, 0.0, 0.0)), "ll")
        check(project, nad, bessel7, lon, lat, lon, lat, bar, "NAD83" + tail)
        check(project, bessel7, nad, lon, lat, lon, lat, bar, "to NAD83" + tail)


def check_towgs84_forms(project, bar):
    """+towgs84 with 3, 7 and fewer values; arc-seconds and ppm"""
    lon, lat = points(12)
    for fig_t, fig in GEO:
        dst = latlong_crs("+ellps=intl", figure_of_ellps("intl"), (-87.0, -98.0, -121.0))
        # three values == seven with zero rotations and scale, bit for bit
        a = project(f"+proj=latlong {fig_t} +towgs84=1.5,-2,3 +no_defs", dst.proj, lon, lat)
        b = project(f"+proj=latlong {fig_t} +towgs84=1.5,-2,3,0,0,0,0 +no_defs", dst.proj, lon, lat)
        assert a[0] == b[0] == 1 and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        # fewer than three values: the missing ones are 0
        for vals in ((250.0,), (250.0, -40.0)):
            check(project, latlong_crs(fig_t, fig, vals), dst, lon, lat, lon, lat, bar, f"{fig_t} {vals}")
        # arc-seconds and ppm are converted: one rotation or a scale alone
        for vals in ((0, 0, 0, 3.0, 0, 0, 0), (0, 0, 0, 0, -2.0, 0, 0), (0, 0, 0, 0, 0, 4.0, 0), (0, 0, 0, 0, 0, 0, 40.0)):
            src = latlong_crs(fig_t, fig, tuple(float(v) for v in vals))
            check(project, src, dst, lon, lat, lon, lat, bar, f"{fig_t} {vals}")
            check(project, dst, src, lon, lat, lon, lat, bar, f"to {fig_t} {vals}")
