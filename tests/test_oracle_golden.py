"""Pin the oracle (oracle/mifi_oracle.c + oracle/pj_oracle.c):

  * against the reference's own known-answer tests, restated from
    /root/reference/test/testInterpolation.cc (line numbers in each test);
  * bit-for-bit against the golden vectors in tests/golden/, which were produced by the reference's own
    src/interpolation.c compiled unmodified (tests/golden/make_golden.py);
  * live against that compiled reference on fresh seeded inputs, when oracle/_ref/ exists.

CPU only.
"""
import numpy as np
import pytest

from conftest import assert_bit_equal
from oracle.oracle import (BICUBIC, BILINEAR, LATITUDE, LONGITUDE, NEAREST_NEIGHBOR, PROJ_AXIS)

EMEP = "+ellps=sphere +a=127.4 +e=0 +proj=stere +lat_0=90 +lon_0=-32 +lat_ts=60 +x_0=7 +y_0=109"
LATLONG = "+ellps=sphere +a=6370 +e=0 +proj=latlong"


# ---------------------------------------------------------------------------------------------------
# reference known answers
# ---------------------------------------------------------------------------------------------------
def test_points2position(oracle):
    # test/testInterpolation.cc:49-58
    got = oracle.points2position([-3.0, 5.0, 1.3, 2.0, 6.0], [1.0, 2, 3, 4, 5], PROJ_AXIS)
    assert np.allclose(got, [-4.0, 4.0, 0.3, 1.0, 5.0], atol=1e-10, rtol=0)


def test_points2position_reverse(oracle):
    # test/testInterpolation.cc:61-70
    got = oracle.points2position([-3.0, 5.0, 1.3, 2.0, 6.0], [5.0, 4, 3, 2, 1], PROJ_AXIS)
    assert np.allclose(got, [8.0, 0.0, 3.7, 3.0, -1.0], atol=1e-10, rtol=0)


def test_get_values_f(oracle):
    # test/testInterpolation.cc:73-80
    assert oracle.get_values(NEAREST_NEIGHBOR, [1.0, 2.0, 1.0, 2.0], 0.3, 0.3, 2, 2, 1)[0] == 1.0


def test_get_values_bilinear_f(oracle):
    # test/testInterpolation.cc:83-112
    f = np.array([1.0, 2.0, 2.0, 1 + np.sqrt(np.float32(2.0))], dtype=np.float32)
    g = lambda x, y: float(oracle.get_values(BILINEAR, f, x, y, 2, 2, 1)[0])
    assert abs(g(0.3, 0.0) - 1.3) < 1e-6
    assert abs(g(0.3, 0.0001) - 1.3) < 1e-4
    assert abs(g(0.0, 0.3) - 1.3) < 1e-6
    assert abs(g(0.0001, 0.3) - 1.3) < 1e-4
    assert not np.isnan(g(0, 0))
    assert not np.isnan(g(1, 1))
    for x, y in ((1.5, 0.5), (0.5, 1.5), (0.5, -0.5), (-0.5, 0.5)):
        assert np.isnan(g(x, y))


def test_get_values_bicubic_f(oracle):
    # test/testInterpolation.cc:115-155
    f = np.array([1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1], dtype=np.float32)
    ft = f.reshape(4, 4).T.copy().ravel()
    g = lambda a, x, y: float(oracle.get_values(BICUBIC, a, x, y, 4, 4, 1)[0])
    assert g(f, 1, 1) == pytest.approx(2.0, rel=1e-5)
    assert g(f, 1, 1.99999) == pytest.approx(2.0, rel=1e-5)
    assert g(f, 1, 1.5) == pytest.approx(2.125, rel=1e-5)
    assert g(f, 1.5, 1) == pytest.approx(2.0, rel=1e-5)
    assert g(ft, 1, 1) == pytest.approx(2.0, rel=1e-5)
    assert g(ft, 1.99999, 1) == pytest.approx(2.0, rel=1e-5)
    assert g(ft, 1.5, 1) == pytest.approx(2.125, rel=1e-5)
    assert g(ft, 1, 1.5) == pytest.approx(2.0, rel=1e-5)
    for x, y in ((0.5, 1), (1, 0.5), (2.5, 1), (1, 2.5)):
        assert np.isnan(g(f, x, y))


def test_project_axes_emep_pole(oracle):
    # test/testInterpolation.cc:265-278: all nine points lie north of 89 degrees
    rc, x, y = oracle.project_axes(EMEP, LATLONG, [6.0, 7, 8], [108.0, 109, 110])
    assert rc == 1
    assert np.all(np.degrees(y) > 89)
    # closed form (Snyder 21-1..4, sphere): the projection origin (7,109) is the pole itself
    assert np.degrees(y[4]) == pytest.approx(90.0, abs=1e-9)


def test_interpolate_f_emep(oracle, golden):
    # test/testInterpolation.cc:280-393: country map, cell (lon 9, lat 25) == 32 for NN, bilinear, bicubic
    g = golden("emep")
    assert g["infield"][50, 93] == 4.0  # :346
    for name, m in (("nn", NEAREST_NEIGHBOR), ("bilinear", BILINEAR), ("bicubic", BICUBIC)):
        rc, out = oracle.interpolate_f(m, EMEP, g["infield"], np.arange(170) + 1.0, np.arange(150) + 1.0, PROJ_AXIS, PROJ_AXIS, 1,
                                       LATLONG, g["lon"], g["lat"], LONGITUDE, LATITUDE)
        assert rc == 1
        assert abs(out[0, 25, 9] - 32) < 1e-6
        assert_bit_equal(out, g[name], f"emep {name} vs compiled reference")


def _rotate_setup(lon0_b):
    a = "+ellps=sphere +a=127.4 +e=0 +proj=stere +lat_0=90 +lon_0=0 +lat_ts=60"
    b = f"+ellps=sphere +a=127.4 +e=0 +proj=stere +lat_0=90 +lon_0={lon0_b} +lat_ts=60"
    ax = np.arange(5) - 2.0
    u = np.arange(25, dtype=np.float32)
    v = 25 - np.arange(25, dtype=np.float32)
    return a, b, ax, u, v


@pytest.mark.parametrize("lon0,tol", [(90, 1e-4), (180, 1e-5)])
def test_vector_reproject_rotate(oracle, lon0, tol):
    # test/testInterpolation.cc:396-453 (90 deg: u -> -v, v -> u) and :455-512 (180 deg: both negated)
    a, b, ax, u, v = _rotate_setup(lon0)
    _, uo = oracle.interpolate_f(NEAREST_NEIGHBOR, a, u, ax, ax, 0, 0, 1, b, ax, ax, 0, 0)
    _, vo = oracle.interpolate_f(NEAREST_NEIGHBOR, a, v, ax, ax, 0, 0, 1, b, ax, ax, 0, 0)
    rc, ur, vr = oracle.vector_reproject_values(a, b, uo, vo, ax, ax, 0, 0, 1)
    assert rc == 1
    uo, vo, ur, vr = uo.ravel(), vo.ravel(), ur.ravel(), vr.ravel()
    if lon0 == 90:
        assert np.all(np.abs(vo - ur) < tol)
        assert np.all(np.abs(uo + vr) < tol)
    else:
        assert np.all(np.abs(vo + vr) < tol)
        assert np.all(np.abs(uo + ur) < tol)


def test_vector_reproject_keep_size(oracle):
    # test/testInterpolation.cc:515-583: |(u,v)| is preserved
    ai = np.arange(4) + 6.0
    aj = np.arange(4) + 108.0
    lon = np.arange(4) * 60.0
    lat = np.arange(4) / 2.0 + 88.5
    u = np.arange(16, dtype=np.float32)
    v = -16 + np.arange(16, dtype=np.float32)
    _, uo = oracle.interpolate_f(NEAREST_NEIGHBOR, EMEP, u, ai, aj, 0, 0, 1, LATLONG, lon, lat, LONGITUDE, LATITUDE)
    _, vo = oracle.interpolate_f(NEAREST_NEIGHBOR, EMEP, v, ai, aj, 0, 0, 1, LATLONG, lon, lat, LONGITUDE, LATITUDE)
    rc, ur, vr = oracle.vector_reproject_values(EMEP, LATLONG, uo, vo, lon, lat, LONGITUDE, LATITUDE, 1)
    assert rc == 1
    ur, vr = ur.ravel(), vr.ravel()
    d = ur.astype(np.float64)**2 + vr.astype(np.float64)**2 - uo.ravel().astype(np.float64)**2 - vo.ravel().astype(np.float64)**2
    d = d[~np.isnan(d)]
    assert d.size > 0 and np.all(np.abs(d) < 1e-3)


def test_vector_reproject_directions(oracle):
    # test/testInterpolation.cc:586-654
    a = "+ellps=sphere +a=127.4 +e=0 +proj=stere +lat_0=90 +lon_0=0 +lat_ts=60"
    ax = (np.arange(5) - 2) * 1000.0
    xf, yf = np.meshgrid(ax, ax)
    rc, m = oracle.vector_matrix_field(a, LATLONG, xf.ravel(), yf.ravel(), 5, 5)
    assert rc == 1
    ang = oracle.vector_reproject_direction(m, np.zeros(25, dtype=np.float32), 5, 5, 1)
    close = lambda want, got: abs(got - want) <= 0.01 * max(abs(want), abs(got))
    assert close(315, ang[0 + 5 * 0]) and close(270, ang[0 + 5 * 2]) and close(225, ang[0 + 5 * 4])
    for j in (0, 1):
        o = ang[2 + 5 * j]
        o = o - 360 if o > 300 else o
        assert close(10, 10 + o)
    assert close(180, ang[2 + 5 * 3]) and close(180, ang[2 + 5 * 4])
    assert close(45, ang[4 + 5 * 0]) and close(90, ang[4 + 5 * 2]) and close(135, ang[4 + 5 * 4])


def test_string_to_method(oracle):
    # src/interpolation.c:66-101, incl. the forward_undef_min quirk (:97-98)
    assert oracle.string_to_method("bilinear") == BILINEAR
    assert oracle.string_to_method("nearestneighbor") == NEAREST_NEIGHBOR
    assert oracle.string_to_method("forward_mean") == 6
    assert oracle.string_to_method("forward_undef_min") == 9
    assert oracle.string_to_method("nope") == -1


# ---------------------------------------------------------------------------------------------------
# golden vectors produced by the compiled reference
# ---------------------------------------------------------------------------------------------------
def test_golden_kernels(oracle, golden):
    g = golden("kernels")
    field, px, py = g["field"], g["px"], g["py"]
    iz, iy, ix = field.shape
    for name, m in (("nn", NEAREST_NEIGHBOR), ("bilinear", BILINEAR), ("bicubic", BICUBIC)):
        got = np.stack([oracle.get_values(m, field, px[i], py[i], ix, iy, iz) for i in range(px.size)], axis=1)
        assert_bit_equal(got, g[name], f"{name} kernel")
    # the masked set is exactly the reference's out-of-bounds branch (interpolation.c:936)
    assert g["ub"].sum() > 0
    assert np.all(np.isnan(g["bilinear"][:, g["ub"]]))


def test_golden_points2position(oracle, golden):
    g = golden("points2position")
    for k in ("asc", "desc", "lon360", "lon180", "lon_regional", "lon_desc", "lat_desc", "nonuniform", "metric"):
        got = oracle.points2position(g[k + "_in"], g[k + "_axis"], int(g[k + "_type"]))
        want = g[k + "_out"]
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), k


def test_golden_vectors(oracle, golden):
    g = golden("vectors")
    for k in ("ll_rot", "ll_stere", "ll_lcc", "stere_ll", "rot_stere"):
        m = g[k + "_m"]
        u, v = g[k + "_u"], g[k + "_v"]
        oz, oy, ox = u.shape
        ur, vr = oracle.vector_reproject_by_matrix(m, u, v, ox, oy, oz)
        assert_bit_equal(ur.reshape(u.shape), g[k + "_ur"], k + " u")
        assert_bit_equal(vr.reshape(v.shape), g[k + "_vr"], k + " v")
        assert np.allclose(m[0::4]**2 + m[1::4]**2, 1.0, atol=1e-14)


# ---------------------------------------------------------------------------------------------------
# live against the compiled reference (only where oracle/_ref exists)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_oracle_equals_reference_kernels(oracle, reference, seed):
    rng = np.random.default_rng(seed)
    ix, iy, iz = int(rng.integers(2, 40)), int(rng.integers(2, 40)), int(rng.integers(1, 5))
    field = rng.normal(0, 100, (iz, iy, ix)).astype(np.float32)
    field[rng.random(field.shape) < 0.05] = np.nan
    px = rng.uniform(-2, ix + 1, 1500)
    py = rng.uniform(-2, iy + 1, 1500)
    px[:200] = np.round(px[:200] * 2) / 2  # integers and half-cells
    py[100:300] = np.round(py[100:300] * 2) / 2
    for m in (NEAREST_NEIGHBOR, BILINEAR, BICUBIC):
        for i in range(px.size):
            if m == BILINEAR and oracle.bilinear_is_ub(px[i], py[i], ix, iy):
                assert np.all(np.isnan(oracle.get_values(m, field, px[i], py[i], ix, iy, iz)))
                continue
            a = oracle.get_values(m, field, px[i], py[i], ix, iy, iz)
            b = reference.get_values(m, field, px[i], py[i], ix, iy, iz)
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (m, px[i], py[i])


def test_oracle_equals_reference_matrix(oracle, reference):
    src = "+proj=latlong +a=6371000 +e=0 +no_defs"
    for dst, xa, ya, xt, yt in (
        ("+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +R=6.371e+06 +no_defs", np.linspace(-10, 10, 11), np.linspace(-8, 8, 9),
         LONGITUDE, LATITUDE),
        ("+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0", np.linspace(-2e6, 2e6, 11), np.linspace(-2e6, 2e6, 9), 0, 0),
        ("+proj=lcc +lat_0=63 +lon_0=15 +lat_1=63 +lat_2=63 +no_defs +R=6.371e+06", np.linspace(-1e6, 1e6, 11), np.linspace(-2e6, 2e6, 9), 0, 0),
    ):
        rc1, m1 = oracle.vector_matrix(src, dst, xa, ya, xt, yt)
        rc2, m2 = reference.vector_matrix(src, dst, xa, ya, xt, yt)
        assert rc1 == rc2 == 1
        assert np.array_equal(m1.view(np.uint64), m2.view(np.uint64)), dst
    # lat/long target: bearing branch (interpolation.c:366-368, 408-412)
    rc1, m1 = oracle.vector_matrix("+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0", src, np.linspace(-30, 40, 9),
                                   np.linspace(50, 85, 7), LONGITUDE, LATITUDE)
    rc2, m2 = reference.vector_matrix("+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0", src, np.linspace(-30, 40, 9),
                                      np.linspace(50, 85, 7), LONGITUDE, LATITUDE)
    assert rc1 == rc2 == 1 and np.array_equal(m1.view(np.uint64), m2.view(np.uint64))
    xs = np.linspace(-1e6, 1e6, 13)
    rc1, m1 = oracle.vector_matrix_points(src, "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0", 1, xs, xs[::-1])
    rc2, m2 = reference.vector_matrix_points(src, "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0", 1, xs, xs[::-1])
    assert rc1 == rc2 == 1 and np.array_equal(m1.view(np.uint64), m2.view(np.uint64))


def test_oracle_cached_loop_equals_reference_kernels(oracle, reference):
    """orc_cached_interpolate (restated CachedInterpolation.cc:118-147) == the reference kernels point by point"""
    rng = np.random.default_rng(7)
    inX, inY, inZ, outX, outY = 19, 13, 4, 31, 11
    field = rng.normal(0, 1, (inZ, inY, inX)).astype(np.float32)
    field[rng.random(field.shape) < 0.05] = np.nan
    px = rng.uniform(0.2, inX - 1.2, outX * outY)  # interior + some strips, none in the UB corner
    py = rng.uniform(-0.4, inY - 0.6, outX * outY)
    for m in (NEAREST_NEIGHBOR, BILINEAR, BICUBIC):
        a = oracle.cached_interpolate(m, px, py, inX, inY, outX, outY, field, nthreads=3)
        b = reference.cached_interpolate(m, px, py, inX, inY, outX, outY, field)
        assert_bit_equal(a, b, f"cached loop method {m}")


# ---------------------------------------------------------------------------------------------------
# A2: the type / fill-value adapters either side of the gather (CDMInterpolator.cc:115-124)
# ---------------------------------------------------------------------------------------------------
def test_adapters_known_answers(oracle):
    """ScaleValue<float, OUT>(NaN, 1, 0, fill, 1, 0) (include/fimex/Utils.h:444-464) lives in a C++ template that cannot
    be compiled here (Boost): its restatement is pinned by the semantics the header spells out -- lround for integer
    targets (half away from zero), plain casts for floating point, NaN -> fill, '+ 0.' turning -0 into +0."""
    v = np.array([2.5, -2.5, 0.49999997, -0.5, 1e9, np.nan, -0.0, 3.4e38, 255.5, -1.0], dtype=np.float32)
    assert oracle.from_float(v[:6], -32767, np.int16).tolist() == [3, -3, 0, -1, np.int16(np.int32(1000000000)), -32767]
    assert oracle.from_float(v[:4], -127, np.int8).tolist() == [3, -3, 0, -1]
    assert oracle.from_float(v[[0, 5, 9]], 255, np.uint8).tolist() == [3, 255, 255]  # (unsigned char)(int)-1 == 255
    assert oracle.from_float(v[[0, 4, 5]], -2147483647, np.int32).tolist() == [3, 1000000000, -2147483647]
    f = oracle.from_float(v[[5, 6, 7]], 9.96921e36, np.float32)
    assert f[0] == np.float32(9.96921e36) and f[2] == np.float32(3.4e38)
    assert f[1] == 0 and not np.signbit(f[1])  # -0 + 0. == +0
    d = oracle.from_float(v[[0, 5]], 9.96921e36, np.float64)
    assert d[0] == 2.5 and d[1] == 9.96921e36
    # asFloat + mifi_bad2nanf: the fill value is compared after narrowing to float; a NaN fill value disables the pass
    s = np.array([-32767, 0, 5, 32767], dtype=np.int16)
    a = oracle.as_float(s, -32767)
    assert np.isnan(a[0]) and a[1:].tolist() == [0.0, 5.0, 32767.0]
    assert a.view(np.uint32)[0] == 0x7fc00000
    assert not np.isnan(oracle.as_float(s, np.nan)).any()
    big = np.array([2**53 + 1, -7], dtype=np.int64)
    assert oracle.as_float(big, 0).tolist() == [float(np.float32(2**53)), -7.0]
    dbl = np.array([9.9692099683868690e+36, 1.0000000001], dtype=np.float64)
    a = oracle.as_float(dbl, 9.9692099683868690e+36)
    assert np.isnan(a[0]) and a[1] == 1.0


def test_adapters_against_reference(oracle, reference):
    """mifi_bad2nanf / mifi_nanf2bad are part of the reference's src/interpolation.c (:1775-1793): the float forms of the
    restated adapters must agree with them bit for bit."""
    import ctypes as C
    rng = np.random.default_rng(77)
    v = rng.normal(0, 100, 5000).astype(np.float32)
    fill = np.float32(9.9692099683868690e+36)
    v[rng.integers(0, v.size, 200)] = fill
    v[rng.integers(0, v.size, 50)] = np.nan
    a = v.copy()
    f = reference.lib.mifi_bad2nanf
    f.restype = C.c_size_t
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_float]
    f(a.ctypes.data, a.ctypes.data + a.nbytes, fill)
    assert_bit_equal(oracle.as_float(v, float(fill)), a, "bad2nan", nan_payload=False)
    assert np.array_equal(np.isnan(a), np.isnan(v) | (v == fill))
    b = a.copy()
    g = reference.lib.mifi_nanf2bad
    g.restype = C.c_size_t
    g.argtypes = [C.c_void_p, C.c_void_p, C.c_float]
    g(b.ctypes.data, b.ctypes.data + b.nbytes, fill)
    assert_bit_equal(oracle.from_float(a, float(fill), np.float32), b, "nan2bad")


# ---------------------------------------------------------------------------------------------------
# coord_kdtree: the restated search against the reference's own nanoflann kd-tree
# ---------------------------------------------------------------------------------------------------
def test_coordkd_against_reference_nanoflann(oracle):
    """flannTranslatePointsToClosestInputCell (CDMInterpolator.cc:991-1062): the reference's vendored nanoflann header,
    compiled from where it lies behind the reference's call sequence (oracle/ref_kd_driver.cc), against the brute-force
    restatement.  A kd-tree only prunes: both must name the same nearest source point."""
    import ctypes as C
    import os
    from oracle import oracle as orc
    so = os.path.join(os.path.dirname(orc.REF_SO), "libkd_ref.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libkd_ref.so not built (no /root/reference on this machine)")
    lib = C.CDLL(so)
    rng = np.random.default_rng(42)
    nx, ny = 90, 61
    lon = np.radians(np.arange(nx) * 4.0)
    lat = np.radians(90 - np.arange(ny) * 3.0)
    lon2d, lat2d = oracle.lonlat_to_matrix(lon, lat)
    # (undefined source coordinates are a declared deviation: the reference leaves them in the cloud as NaN points, which
    # corrupts the tree's bounding boxes -- half of the targets lose their match; the restatement and the GPU skip them)
    tlon = rng.uniform(-np.pi, np.pi, 4000)
    tlat = rng.uniform(-np.pi / 2, np.pi / 2, 4000)
    for max_dist in (150e3, 400e3, 3000e3):
        wx, wy, ties = oracle.coordkd(tlon, tlat, lon2d, lat2d, nx, ny, max_dist)
        rx, ry = tlon.copy(), tlat.copy()
        dp = C.POINTER(C.c_double)
        lib.ref_coordkd.argtypes = [dp, dp, C.c_size_t, dp, dp, C.c_size_t, C.c_size_t, C.c_double]
        lib.ref_coordkd(rx.ctypes.data_as(dp), ry.ctypes.data_as(dp), rx.size, lon2d.ctypes.data_as(dp), lat2d.ctypes.data_as(dp), nx, ny,
                        max_dist)
        differ = int(((rx != wx) | (ry != wy)).sum())
        assert differ <= ties, (max_dist, differ, ties)  # equal distances (the pole row) are ordered by an unstable sort
        assert (wx == -1000).any() == (max_dist < 400e3)
    # getMaxDistanceOfInterest (:304-326): degrees are multiplied by the earth radius as given
    assert oracle.max_distance_of_interest([0, 0.5, 1.0], [10, 10.25], False) == 6371000 * 0.5
    assert oracle.max_distance_of_interest([0, 2500, 5000], [0, 1000], True) == 2500


# ---------------------------------------------------------------------------------------------------
# fill2d / creepfill2d: the restated sweeps against the compiled reference
# ---------------------------------------------------------------------------------------------------
def _holey_field(rng, shape, frac):
    ny, nx = shape[-2:]
    yy, xx = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    f = (280 + 10 * np.sin(xx / 7.0) * np.cos(yy / 5.0) + rng.normal(0, 0.5, shape)).astype(np.float32)
    f[rng.random(shape) < frac] = np.nan
    f[..., 3:9, 4:15] = np.nan  # a block hole, and holes on the border
    f[..., 0, :5] = np.nan
    f[..., -1, -3:] = np.nan
    f[..., 5:8, 0] = np.nan
    return f


@pytest.mark.parametrize("shape", [(3, 20, 31), (1, 2, 2), (2, 2, 9), (2, 9, 2), (1, 3, 3)])
def test_fill2d_and_creepfill2d_against_reference(oracle, reference, shape):
    """interpolation.c:1246-1537 compiled unmodified vs oracle/mifi_oracle.c, bit for bit, including the convergence exit,
    maxLoop < 5 (the size_t wrap of `maxLoop - 5`), degenerate 2-wide grids and levels with nothing to fill"""
    rng = np.random.default_rng(sum(shape))
    f = _holey_field(rng, shape, 0.1) if min(shape[-2:]) > 9 else rng.normal(5, 1, shape).astype(np.float32)
    if min(shape[-2:]) <= 9:
        f.reshape(-1)[::3] = np.nan
    for args in ((0.01, 1.6, 100), (1e-6, 1.0, 7), (0.5, 1.9, 3), (0.01, 1.6, 0)):
        got, n1 = oracle.fill2d(f, *args)
        want, n2 = oracle.fill2d(f, *args, lib=reference.lib, name="mifi_fill2d_f")
        assert n1 == n2
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), args
        assert not np.isnan(got).any()
    for repeat, weight, dv in ((20, 2, None), (3, 1, None), (5, 2, 0.0), (1, 3, -7.5), (0, 2, None)):
        got, n1 = oracle.creepfill2d(f, repeat, weight, dv)
        want, n2 = oracle.creepfill2d(f, repeat, weight, dv, lib=reference.lib, prefix="ref")
        assert n1 == n2
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (repeat, weight, dv)
    full = np.ones(shape, dtype=np.float32)
    assert np.array_equal(oracle.fill2d(full, 0.01, 1.6, 100)[0], full)
    allnan = np.full(shape, np.nan, dtype=np.float32)
    assert np.isnan(oracle.creepfill2d(allnan, 20, 2)[0]).all()


@pytest.mark.parametrize("nx,ny", [(799, 799), (800, 800), (1600, 1599), (1000, 1000), (1200, 900), (900, 1200), (2000, 2000), (30, 700),
                                   (700, 30)])
def test_fill2d_and_creepfill2d_against_reference_at_kernel_switch_shapes(oracle, reference, nx, ny):
    """the shapes at which tests/test_gpu_forward_fill_fuzz.py compares the device kernels with the restatement: the restatement
    against the compiled reference there too, one parameter set per process (a negative char weight for creepfillval2d)"""
    rng = np.random.default_rng(nx * 3 + ny)
    f = _holey_field(rng, (1, ny, nx), 0.1)
    got, n1 = oracle.fill2d(f, 0.01, 1.6, 100)
    want, n2 = oracle.fill2d(f, 0.01, 1.6, 100, lib=reference.lib, name="mifi_fill2d_f")
    assert n1 == n2 and np.array_equal(got.view(np.uint32), want.view(np.uint32))
    for repeat, weight, dv in ((20, 2, None), (5, 200, -3.5)):
        got, n1 = oracle.creepfill2d(f, repeat, weight, dv)
        want, n2 = oracle.creepfill2d(f, repeat, weight, dv, lib=reference.lib, prefix="ref")
        assert n1 == n2 and np.array_equal(got.view(np.uint32), want.view(np.uint32)), (repeat, weight, dv)
