"""An independent reference for the two coordinate searches, coord_nearestneighbor and coord_kdtree -- TEST INFRASTRUCTURE.

Both searches turn 2-D source longitude / latitude (radians) into a source index per target.  The kernels
(`fimex_b200/csrc/coordnn_kernels.cu`) and the restatement (`orc_coordnn` / `orc_coordkd` in `oracle/mifi_oracle.c`) share one
algorithm: a latitude-sorted array scanned around each target.  This module does not: it puts sources and targets on the unit
sphere and asks `scipy.spatial.cKDTree` (or, for small cases, an exhaustive search) for the nearest sources by chord length,
then decides among them in `numpy.longdouble` (64-bit mantissa on x86-64).  Chord length and great-circle distance order
points the same way (`cos_d = 1 - chord**2 / 2`), so the nearest sources by chord hold the winner of both searches.

The contract restated (DESIGN section 2):

* coord_nearestneighbor: the valid source (neither coordinate NaN) with the largest
  `cos_d = cos(lat_s) cos(lat_t) cos(lon_s - lon_t) + sin(lat_s) sin(lat_t)` among those with `cos_d > cos(roi)`, else (-1, -1).
  `roi = min(1.414 * acos(w), pi)` where w is the smallest, over the sample points of `getGridDistance`, of the largest `cos_d`
  from the sample to any other valid point.  Samples: every point when `nx*ny <= 1000`, else `k * (nx*ny / 53)` for k < 53;
  NaN samples are skipped.  No valid sample (or a single valid point) makes `roi` NaN, and every target gets (-1, -1).
  Exact ties: the candidate met first scanning up from `lower_bound(latitude)` and then down, equal latitudes (-0 equal to +0)
  in insertion order (`ix` outer, `iy` inner).
* coord_kdtree: `r = maxDist / 6371000` and `r2 = r * r` in fp64; the valid source with the smallest chord
  `d0*d0 + d1*d1 + d2*d2` of the unit vectors `(cos lat cos lon, cos lat sin lon, sin lat)` with chord < r2, else
  (-1000, -1000).  Exact ties: the lowest source position `ix + iy*nx`.

The error bound.  Both the kernels and the restatement start from the same fp64 radians (the degree -> radian product
`FB_DEG_TO_RAD * v` is one IEEE multiplication, done identically here by `to_rad`), so that rounding is common to all sides and
is not a term.  Let u = 2**-53.  The fp64 evaluation of the quantities above differs from the exact value of the same inputs by:

* `sin` / `cos` / `sincos`: at most 2 ulp in CUDA's fp64 library (CUDA Programming Guide, Mathematical Functions), at most 1 ulp
  in glibc; 2 ulp <= 4u relative.
* `lon_s - lon_t` is rounded once: relative u, which moves `cos` by at most `|sin(dlon)| * u * |dlon| <= u * |dlon|`.
* Products and sums: u relative each.  nvcc contracts `k_nn_search` and `k_grid_distance` into FMAs (no `--fmad=false`; those
  expressions use plain `*` / `+`); a contraction only drops roundings, so a bound that charges every operation covers it.
  `k_kd_search` uses `__dmul_rn` / `__dadd_rn` and is not contracted.

cos_d.  With `c = |cos lat_s cos lat_t cos dlon|` and `s = |sin lat_s sin lat_t|`: the first term carries 2 + 2 + 2 ulp-scale
factors of 4u (two latitude cosines, the longitude cosine) plus two products, the second two sines plus one product, and the sum
one rounding: `15u c + 10u s + u |dlon|` to first order.  The bound used is twice that, `eps_cd = 32u (c + s) + 2u |dlon|`
(the factor 2 covers second-order terms many times over).

chord.  Each unit-vector component carries two factors of 4u and a product: `9u` relative; each difference `d_i` then
`D_i = 9u (|q_i| + |p_i|) + u |d_i|`; the chord `sum(2 |d_i| D_i + D_i**2 + u d_i**2) + 2u * chord`; twice that is used.

Targets.  With the target CRS `+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs` the projection to the search's lat/long is the
identity, bit for bit (asserted by the tests on the CPU and on the GPU), so targets are the mesh of `to_rad(axis)`.  Other target
CRSs (rotated pole) are pinned to 1e-9 degree, `tests/test_gpu_fuzz.py::test_fuzz_projections_within_1e9_degree`; a target moved
by delta moves `cos_d` by at most `sin(d) * delta` and the chord by at most `delta` (so the chord squared by `2 chord delta +
delta**2`).  Callers pass `delta` for such targets.

ROI.  The sample's largest `cos_d` w carries `eps_cd`; `acos` turns that into `eps_cd / sqrt(1 - w**2)`, the factor 1.414 and
the fp64 `acos` / `cos` / products add a few u; `cos(roi)` moves by `sin(roi)` times the angle error.  A decision
`cos_d > cos(roi)` within the sum of both errors is ambiguous.

Ambiguity.  A target is flagged when its answer could go either way within these errors: when the runner-up candidate is within
`eps_1 + eps_2` of the best (exactly equal values included, unless the caller designed exact ties and asks for the tie rule), or when
the best is within the error of the ROI or radius threshold.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.spatial import cKDTree

LD = np.longdouble
U = 2.0 ** -53
DEG_TO_RAD = np.float64(".0174532925199432958")  # FB_DEG_TO_RAD (proj_api.h DEG_TO_RAD)
EARTH_R = 6371000.0  # MIFI_EARTH_RADIUS_M
PI = math.pi
DELTA_PROJ = 1e-9 * PI / 180  # the projections' pinned tolerance, 1e-9 degree, in radians
BRUTE_LIMIT = 10 ** 7  # sources x targets up to which the candidates come from an exhaustive search
K = 16


def to_rad(deg):
    """the library's degree -> radian conversion (`FB_DEG_TO_RAD * v`), bit for bit"""
    return DEG_TO_RAD * np.asarray(deg, dtype=np.float64)


def _unit(lon, lat):
    cl = np.cos(lat)
    return np.stack([cl * np.cos(lon), cl * np.sin(lon), np.sin(lat)], axis=-1)


def _unit_ld(lon, lat):
    lon, lat = np.asarray(lon, LD), np.asarray(lat, LD)
    cl = np.cos(lat)
    return np.stack([cl * np.cos(lon), cl * np.sin(lon), np.sin(lat)], axis=-1)


def cos_d_ld(slon, slat, tlon, tlat):
    slon, slat, tlon, tlat = (np.asarray(v, LD) for v in (slon, slat, tlon, tlat))
    return np.cos(slat) * np.cos(tlat) * np.cos(slon - tlon) + np.sin(slat) * np.sin(tlat)


def eps_cos_d(slon, slat, tlon, tlat, delta=0.0):
    c = np.abs(np.cos(slat) * np.cos(tlat) * np.cos(slon - tlon))
    s = np.abs(np.sin(slat) * np.sin(tlat))
    cd = np.clip(c * np.sign(np.cos(slon - tlon)) + np.sin(slat) * np.sin(tlat), -1, 1)
    return 32 * U * (c + s) + 2 * U * np.abs(slon - tlon) + delta * np.sqrt(1 - cd * cd) + 1e-300


def chord2_ld(slon, slat, tlon, tlat):
    d = _unit_ld(slon, slat) - _unit_ld(tlon, tlat)
    return (d * d).sum(axis=-1)


def eps_chord2(slon, slat, tlon, tlat, delta=0.0):
    p, q = _unit(slon, slat), _unit(tlon, tlat)
    d = q - p
    D = 9 * U * (np.abs(q) + np.abs(p)) + U * np.abs(d)
    c2 = (d * d).sum(axis=-1)
    e = (2 * np.abs(d) * D + D * D + U * d * d).sum(axis=-1) + 2 * U * c2
    ch = np.sqrt(c2)
    return 2 * e + 2 * ch * delta + delta * delta + 1e-300


def sample_positions(nx, ny):
    """getGridDistance's sample positions (CDMInterpolator.cc:1064-1125)"""
    ns = nx * ny
    if ns > 1000:
        return np.arange(53, dtype=np.int64) * (ns // 53)
    return np.arange(ns, dtype=np.int64)


def _nearest_candidates(src, tgt, k, exclude=None):
    """the nearest sources by chord for every target: (idx [n][k'] padded with -1, {row: idx} for rows widened to every source
    within 1e-9 of the best chord squared, where the k-th nearest is not clearly farther).  `exclude[i]`: a source index the
    row must not name (the sample itself in getGridDistance)."""
    n, m = len(tgt), len(src)
    if m == 0 or n == 0:
        return np.full((n, 1), -1, dtype=np.int64), {}
    kk = min(k + (exclude is not None), m)
    tree = None
    if n * m <= BRUTE_LIMIT:
        idx = np.empty((n, kk), dtype=np.int64)
        dist = np.empty((n, kk))
        step = max(1, BRUTE_LIMIT // (4 * m))
        for a in range(0, n, step):
            dd = ((tgt[a:a + step, None, :] - src[None, :, :]) ** 2).sum(-1)
            if exclude is not None:
                dd[np.arange(dd.shape[0]), exclude[a:a + step]] = np.inf
            part = np.argpartition(dd, kk - 1, axis=1)[:, :kk] if kk < m else np.broadcast_to(np.arange(m), dd.shape).copy()
            pd = np.take_along_axis(dd, part, 1)
            o = np.argsort(pd, axis=1, kind="stable")
            idx[a:a + step] = np.take_along_axis(part, o, 1)
            dist[a:a + step] = np.sqrt(np.take_along_axis(pd, o, 1))
    else:
        tree = cKDTree(src)
        dist, idx = tree.query(tgt, k=kk)
        dist, idx = dist.reshape(n, kk), idx.reshape(n, kk).astype(np.int64)
        if exclude is not None:
            dist = np.where(idx == exclude[:, None], np.inf, dist)
            o = np.argsort(dist, axis=1, kind="stable")
            idx, dist = np.take_along_axis(idx, o, 1), np.take_along_axis(dist, o, 1)
    idx = np.where(np.isfinite(dist), idx, -1)
    wide = {}
    if kk < m:
        last = np.where(np.isfinite(dist), dist, -1).max(axis=1)
        for i in np.flatnonzero(last ** 2 <= dist[:, 0] ** 2 + 1e-9):
            if tree is None:
                dd = ((src - tgt[i]) ** 2).sum(-1)
                ball = np.flatnonzero(dd <= dist[i, 0] ** 2 + 1e-9)
            else:
                ball = np.array(tree.query_ball_point(tgt[i], math.sqrt(dist[i, 0] ** 2 + 1e-9) + 1e-12), dtype=np.int64)
            if exclude is not None:
                ball = ball[ball != exclude[i]]
            wide[int(i)] = np.union1d(idx[i][idx[i] >= 0], ball)
    return idx, wide


class Result:
    """per target: ix, iy (the ideal answer, or the miss value), the ambiguity flag, and for ambiguous targets the set of
    (ix, iy) answers any of which is acceptable"""

    def __init__(self, ix, iy, amb, cand):
        self.ix, self.iy, self.amb, self.cand = ix, iy, amb, cand


def _valid(lon2d, lat2d):
    lon2d, lat2d = np.asarray(lon2d, np.float64).ravel(), np.asarray(lat2d, np.float64).ravel()
    return lon2d, lat2d, np.flatnonzero(~(np.isnan(lon2d) | np.isnan(lat2d)))


def grid_roi(lon2d, lat2d, nx, ny, k=K):
    """getGridDistance in longdouble: (roi or NaN, w, the error bound of w)"""
    lon2d, lat2d, valid = _valid(lon2d, lat2d)
    sp = sample_positions(nx, ny)
    sp = sp[~(np.isnan(lon2d[sp]) | np.isnan(lat2d[sp]))]
    if sp.size == 0 or valid.size < 2:
        return math.nan, math.nan, 0.0  # acos(2) (no valid sample) or acos(-2) (no other valid point)
    # the sample itself is excluded by position, not by distance: a duplicate point counts
    idx, wide = _nearest_candidates(_unit(lon2d[valid], lat2d[valid]), _unit(lon2d[sp], lat2d[sp]), k,
                                    exclude=np.searchsorted(valid, sp))
    best = np.empty(sp.size, dtype=LD)
    eps = np.empty(sp.size)
    for j in range(sp.size):
        c = valid[wide[j] if j in wide else idx[j][idx[j] >= 0]]
        cd = cos_d_ld(lon2d[c], lat2d[c], lon2d[sp[j]], lat2d[sp[j]])
        b = int(np.argmax(cd))
        best[j] = cd[b]
        eps[j] = float(eps_cos_d(lon2d[c[b]], lat2d[c[b]], lon2d[sp[j]], lat2d[sp[j]]))
    w = best.min()
    return min(1.414 * float(np.arccos(w)), PI), w, float(eps.max())


def _decide(c, q, e, thr, eps_thr, better, tie_key, exact_ties, nx, miss):
    """one block of targets: c [n][w] source positions (-1 pads), q their quantity (longdouble), e its error bound; `better`
    is +1 when larger q wins (cos_d) and -1 when smaller wins (chord).  Returns ix, iy, amb, cand (a dict row -> set)."""
    n, w = c.shape
    pad = c < 0
    s = np.where(pad, LD(-np.inf), better * q)  # larger s wins
    t = better * thr
    inside = (s > t) & ~pad
    near = (np.abs(s - t) <= e + eps_thr) & ~pad
    top = s.max(axis=1)
    is_top = (s == top[:, None]) & ~pad
    if exact_ties:
        key = np.where(is_top, tie_key, np.iinfo(np.int64).max)
        b = np.argmin(key, axis=1)
    else:
        b = np.argmax(s, axis=1)
    eb = np.take_along_axis(e, b[:, None], 1)
    close = ~pad & (s >= top[:, None] - (e + eb))
    close[np.arange(n), b] = False
    if exact_ties:
        close &= ~is_top
    hit = inside.any(axis=1)
    p = np.take_along_axis(c, b[:, None], 1)[:, 0]
    ix = np.where(hit, p % nx, miss)
    iy = np.where(hit, p // nx, miss)
    near_b = np.take_along_axis(near, b[:, None], 1)[:, 0]
    amb = np.where(hit, close.any(axis=1) | near_b, near.any(axis=1))
    cand = {}
    for i in np.flatnonzero(amb):
        if hit[i]:
            grp = close[i] | is_top[i]
            grp[b[i]] = True
            if near_b[i]:
                grp |= inside[i] | near[i]
        else:
            grp = near[i]
        cand[int(i)] = {(int(x % nx), int(x // nx)) for x in c[i][grp]}
        if not hit[i] or near_b[i]:
            cand[int(i)].add((miss, miss))
    return ix, iy, amb, cand


def _search(tlon, tlat, lon2d, lat2d, nx, ny, quantity, error, thr, eps_thr, better, tie_key_fn, exact_ties, miss, k, window=None):
    tlon, tlat = np.asarray(tlon, np.float64).ravel(), np.asarray(tlat, np.float64).ravel()
    lon2d, lat2d, valid = _valid(lon2d, lat2d)
    n = tlon.size
    ix = np.full(n, miss, dtype=np.int64)
    iy = np.full(n, miss, dtype=np.int64)
    amb = np.zeros(n, dtype=bool)
    cands = [None] * n
    ti = np.flatnonzero(~(np.isnan(tlon) | np.isnan(tlat)))  # a NaN target matches nothing
    if thr is None or valid.size == 0 or ti.size == 0:
        return Result(ix, iy, amb, cands)
    idx, wide = _nearest_candidates(_unit(lon2d[valid], lat2d[valid]), _unit(tlon[ti], tlat[ti]), k)
    blocks = [(np.arange(ti.size), idx)] + [(np.array([r]), row[None, :]) for r, row in wide.items()]
    for rows, ib in blocks:
        c = np.where(ib >= 0, valid[np.maximum(ib, 0)], -1)
        cc = np.maximum(c, 0)
        tl, tp = tlon[ti[rows]][:, None], tlat[ti[rows]][:, None]
        q = quantity(lon2d[cc], lat2d[cc], tl, tp)
        e = error(lon2d[cc], lat2d[cc], tl, tp)
        border = np.zeros(c.shape, dtype=bool)
        if window is not None:
            dl = np.abs(lat2d[cc] - tp)
            border = (np.abs(dl - window) <= 4 * U * (np.abs(tp) + window)) & (c >= 0)
            c_in = np.where(dl > window, -1, c)
        else:
            c_in = c
        bx, by, ba, bc = _decide(c_in, q, e, thr, eps_thr, better, tie_key_fn(cc, tp), exact_ties, nx, miss)
        t = ti[rows]
        ix[t], iy[t], amb[t] = bx, by, ba
        for i, v in bc.items():
            cands[t[i]] = v
        for i in np.flatnonzero(border.any(axis=1)):  # a candidate on the edge of the latitude window
            amb[t[i]] = True
            cands[t[i]] = {(int(x % nx), int(x // nx)) for x in c[i][c[i] >= 0]} | {(miss, miss)}
    return Result(ix, iy, amb, cands)


def coord_nn(tlon, tlat, lon2d, lat2d, nx, ny, delta=0.0, exact_ties=False, k=K):
    """the ideal coord_nearestneighbor answer per target, (-1, -1) for none.  `delta`: the targets' position tolerance (radians).
    `exact_ties`: candidates with exactly equal longdouble cos_d are resolved by the scan-rank rule instead of being flagged."""
    lon2d, lat2d, _ = _valid(lon2d, lat2d)
    roi, w, eps_w = grid_roi(lon2d, lat2d, nx, ny, k)
    thr = eps_thr = window = None
    if not math.isnan(roi):
        # the scan's latitude window |lat_s - lat_t| <= acos(cos(roi)) in fp64; implied by cos_d > cos(roi) for targets within
        # +-90 degrees, a restriction of its own for targets beyond the poles
        window = math.acos(math.cos(roi))
        thr = np.cos(LD(roi))
        # the ROI's angle error from the error of w (acos is steep near 1); near pi cos is flat, so whether the cap applies moves
        # the threshold by at most d_roi**2 / 2
        a0 = float(np.arccos(w))
        d_roi = 1.414 * max(abs(math.acos(max(float(w) - eps_w, -1.0)) - a0), abs(math.acos(min(float(w) + eps_w, 1.0)) - a0))
        d_roi += 8 * U * roi
        eps_thr = math.sin(roi) * d_roi + d_roi * d_roi / 2 + 8 * U
    seq = np.empty(lon2d.size, dtype=np.int64)  # insertion order: ix outer, iy inner
    seq[(np.arange(nx)[:, None] + np.arange(ny)[None, :] * nx).ravel()] = np.arange(lon2d.size)
    # scan rank: up from lower_bound(latitude) in (latitude, insertion) order, then down; -0 and +0 are equal latitudes
    rank_up = np.lexsort((seq, lat2d + 0.0))  # NaN latitudes sort last and are never candidates
    order_up = np.empty(lon2d.size, dtype=np.int64)
    order_up[rank_up] = np.arange(lon2d.size)

    def tie_key(cc, tp):
        up = lat2d[cc] >= tp
        return np.where(up, order_up[cc], 2 * lon2d.size - order_up[cc])

    return _search(tlon, tlat, lon2d, lat2d, nx, ny, lambda a, b, c, d: cos_d_ld(a, b, c, d),
                   lambda a, b, c, d: eps_cos_d(a, b, c, d, delta), thr, eps_thr, 1, tie_key, exact_ties, -1, k, window)


def max_distance_of_interest(xa, ya, is_metric):
    """getMaxDistanceOfInterest (CDMInterpolator.cc:304-326): the largest step of either axis, degrees times the earth radius
    as given"""
    factor = 1.0 if is_metric else EARTH_R
    m = 0.0
    for a in (np.asarray(xa, np.float64), np.asarray(ya, np.float64)):
        if a.size > 1:
            m = max(m, float((factor * np.abs(np.diff(a))).max()))
    return m


def coord_kd(tlon, tlat, lon2d, lat2d, nx, ny, max_dist_m, delta=0.0, exact_ties=False, k=K):
    """the ideal coord_kdtree answer per target, (-1000, -1000) for none"""
    r = np.float64(max_dist_m) / np.float64(EARTH_R)
    r2 = LD(r * r)  # both fp64 roundings are the kernel's own, so the threshold carries no error
    return _search(tlon, tlat, lon2d, lat2d, nx, ny, chord2_ld, lambda a, b, c, d: eps_chord2(a, b, c, d, delta), r2, 0.0, -1,
                   lambda cc, tp: np.broadcast_to(cc, cc.shape), exact_ties, -1000, k)


def compare(ref, gx, gy, what="", max_amb_share=0.01, check_share=True, share_of=None):
    """unambiguous targets identical, ambiguous ones among the reference's candidates, at most `max_amb_share` of the targets
    `share_of` (a mask; all by default) ambiguous; returns the number of ambiguous targets"""
    gx, gy = np.asarray(gx).ravel(), np.asarray(gy).ravel()
    sure = ~ref.amb
    bad = np.flatnonzero(sure & ((gx != ref.ix) | (gy != ref.iy)))
    assert bad.size == 0, f"{what}: {bad.size} unambiguous targets differ; first {bad[:5]}: got " \
                          f"{list(zip(gx[bad[:5]], gy[bad[:5]]))} want {list(zip(ref.ix[bad[:5]], ref.iy[bad[:5]]))}"
    for t in np.flatnonzero(ref.amb):
        assert (int(gx[t]), int(gy[t])) in ref.cand[t], f"{what}: target {t}: {(gx[t], gy[t])} not among {ref.cand[t]}"
    share_of = np.ones(ref.amb.size, dtype=bool) if share_of is None else share_of
    n_amb, n = int(ref.amb[share_of].sum()), int(share_of.sum())
    if check_share:
        assert n_amb <= max_amb_share * max(1, n), f"{what}: {n_amb} of {n} targets ambiguous"
    return n_amb


# ---------------------------------------------------------------------------------------------------
# seeded cases
# ---------------------------------------------------------------------------------------------------
WGS84 = "+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs"
ROTPOLE = "+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +R=6.371e+06 +no_defs"
FAMILIES = ("regular360", "regular180", "curvilinear", "swath", "polar", "dateline", "cluster")


def make_case(seed, family=None, max_src=40000, max_tgt=20000, method=None):
    """one seeded case: dict with family, nx, ny, lon2d / lat2d (degrees, [ny][nx] flattened), target CRS, target axes (degrees),
    method ('nn' or 'kd') and maxDistance (metres, 0 = derived)"""
    rng = np.random.default_rng(seed)
    family = family or FAMILIES[seed % len(FAMILIES)]
    method = method or ("nn" if seed % 2 == 0 else "kd")
    size = int(rng.choice([1, 2, 3, 5, 8, 20, 31, 40, 100, 200]))
    nx = int(np.clip(rng.integers(1, 3 * size + 2), 1, 2000))
    ny = int(np.clip(rng.integers(1, 3 * size + 2), 1, 2000))
    while nx * ny > max_src:
        nx, ny = max(1, nx // 2), max(1, ny // 2)
    i = np.arange(nx)[None, :].astype(np.float64)
    j = np.arange(ny)[:, None].astype(np.float64)
    if family in ("regular360", "regular180"):
        dl, dp = rng.uniform(0.05, 4.0), rng.uniform(0.05, 4.0)
        ny = min(ny, int(178 / dp) + 1)  # short of the poles: a pole row is equidistant from a polar target (its own test)
        j = j[:ny]
        l0 = 0.0 if family == "regular360" else -180.0
        lon = l0 + dl * i + 0 * j
        lat = rng.uniform(-89 + dp * (ny - 1), 89) - dp * j + 0 * i
        if rng.random() < 0.5:
            lat = lat[::-1]
    elif family == "curvilinear":
        a = rng.uniform(0, 2 * np.pi)
        s1, s2 = rng.uniform(0.02, 1.0, 2)
        lon = rng.uniform(-60, 60) + s1 * (i * np.cos(a) - j * np.sin(a)) + 0.3 * np.sin(j / 5.0)
        lat = 89.5 * np.tanh((rng.uniform(-50, 50) + s2 * (i * np.sin(a) + j * np.cos(a)) + 0.2 * np.cos(i / 7.0)) / 89.5)
    elif family == "swath":
        s = rng.uniform(0.01, 0.3)
        lon = rng.uniform(-180, 180) + s * i + 0.4 * s * j + 0.05 * (i - nx / 2) ** 2 * s / max(nx, 1)
        lat = 89.9 * np.tanh((rng.uniform(-70, 70) + s * j - 0.2 * s * i) / 89.9)
        lon, lat = lon.copy(), lat.copy()
        if ny > 2:
            lat[rng.integers(0, ny), :] = np.nan
        if nx > 2:
            lon[:, rng.integers(0, nx)] = np.nan
        holes = rng.random(lon.shape) < 0.03
        lon[holes & (rng.random(lon.shape) < 0.5)] = np.nan
        lat[holes & (rng.random(lon.shape) < 0.5)] = np.nan
    elif family == "polar":
        h = rng.uniform(5, 200) * 1e3
        x = (i - (nx - 1) / 2 + rng.uniform(-0.5, 0.5)) * h
        y = (j - (ny - 1) / 2 + rng.uniform(-0.5, 0.5)) * h + 0 * i
        rho = np.hypot(x, y)
        lat = 90 - np.degrees(2 * np.arctan(rho / (2 * 6371000.0)))
        lon = np.degrees(np.arctan2(x, -y)) + rng.uniform(-180, 180)
        if rng.random() < 0.5:
            lat = -lat
    elif family == "dateline":
        dl = rng.uniform(0.05, 2.0)
        lon = 180 - dl * (nx // 2) + dl * i + 0 * j
        if rng.random() < 0.5:
            lon = np.where(lon > 180, lon - 360, lon)
        lat = 89.5 * np.tanh((rng.uniform(-60, 60) + rng.uniform(0.05, 2.0) * j) / 89.5) + 0 * i
    else:  # cluster
        nx, ny = int(rng.integers(1, 6)), int(rng.integers(1, 6))
        i = np.arange(nx)[None, :].astype(np.float64)
        j = np.arange(ny)[:, None].astype(np.float64)
        c0, c1 = rng.uniform(-170, 170), rng.uniform(-80, 80)
        lon = c0 + rng.uniform(0.01, 0.5, (ny, nx)) * i
        lat = c1 + rng.uniform(0.01, 0.5, (ny, nx)) * j + 0 * i
    lon = np.ascontiguousarray(lon + 0 * j, dtype=np.float64).ravel()
    lat = np.ascontiguousarray(lat + 0 * i, dtype=np.float64).ravel()
    # targets
    tcrs = ROTPOLE if rng.random() < 0.3 else WGS84
    n_tgt = int(rng.choice([1, 7, 100, 1000, max_tgt]))
    ox = max(1, int(math.sqrt(n_tgt) * rng.uniform(0.5, 2.0)))
    oy = max(1, n_tgt // ox)
    if tcrs == WGS84:
        vlon, vlat = lon[~np.isnan(lon)], lat[~np.isnan(lat)]
        cx = float(vlon.mean()) if vlon.size else 0.0
        cy = float(vlat.mean()) if vlat.size else 0.0
        span = rng.uniform(0.5, 1.5) * max(1.0, float(np.ptp(vlon)) if vlon.size else 1.0)
        spany = rng.uniform(0.5, 1.5) * max(1.0, float(np.ptp(vlat)) if vlat.size else 1.0)
        if family == "cluster":
            span, spany = 60.0, 40.0
        xa = cx - span / 2 + span * np.arange(ox) / max(1, ox - 1) + rng.uniform(-0.01, 0.01)
        ya = np.clip(cy - spany / 2 + spany * np.arange(oy) / max(1, oy - 1), -100, 100) + rng.uniform(-0.01, 0.01)
        if rng.random() < 0.2:
            ya = np.concatenate([ya, [90.0, -90.0, 95.0]])  # at and beyond the poles
            xa = np.concatenate([xa, [180.0, -180.0, 190.0]])  # at and beyond the date line
    else:
        xa = rng.uniform(-180, 180) + np.arange(ox) * rng.uniform(0.05, 360.0 / ox)
        ya = rng.uniform(-80, 0) + np.arange(oy) * rng.uniform(0.05, 160.0 / oy)
    max_dist = 0.0
    if method == "kd":
        max_dist = float(rng.choice([0.0, 1.0, 50e3, 300e3, 3000e3, 12742e3, 2e7]))
    return dict(seed=seed, family=family, method=method, nx=nx, ny=ny, lon=lon, lat=lat, tcrs=tcrs, xa=np.asarray(xa, np.float64),
                ya=np.asarray(ya, np.float64), max_dist=max_dist)


def case_targets(case, oracle):
    """target lon / lat (radians) as the search sees them, and their position tolerance"""
    xr, yr = to_rad(case["xa"]), to_rad(case["ya"])
    if case["tcrs"] == WGS84:
        return np.tile(xr, yr.size), np.repeat(yr, xr.size), 0.0
    rc, tx, ty = oracle.project_axes(case["tcrs"], WGS84, xr, yr)
    assert rc == 1
    return tx, ty, DELTA_PROJ


def case_max_dist(case):
    return case["max_dist"] if case["max_dist"] > 0 else max_distance_of_interest(case["xa"], case["ya"], False)


def reference_for(case, oracle, exact_ties=False):
    tx, ty, delta = case_targets(case, oracle)
    lon, lat = to_rad(case["lon"]), to_rad(case["lat"])
    if case["method"] == "nn":
        return coord_nn(tx, ty, lon, lat, case["nx"], case["ny"], delta, exact_ties)
    return coord_kd(tx, ty, lon, lat, case["nx"], case["ny"], case_max_dist(case), delta, exact_ties)


def oracle_for(case, oracle):
    tx, ty, _ = case_targets(case, oracle)
    lon, lat = to_rad(case["lon"]), to_rad(case["lat"])
    if case["method"] == "nn":
        wx, wy, ties = oracle.coordnn(tx, ty, lon, lat, case["nx"], case["ny"])
    else:
        wx, wy, ties = oracle.coordkd(tx, ty, lon, lat, case["nx"], case["ny"], case_max_dist(case))
    return wx, wy, ties
