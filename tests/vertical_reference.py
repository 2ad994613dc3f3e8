"""An independent high-precision reference for the three vertical branches (pressure, height, depth) -- TEST INFRASTRUCTURE ONLY.

Written from the contract in DESIGN.md section 2, not from the C restatements (tests/vertical_*oracle.c): numpy ``longdouble``
(x87 extended, 64-bit significand) with the C library's ``logl`` / ``expl`` instead of the written-out fdlibm ``vlog`` / ``vexp``, the
published constants parsed from their decimal strings, the brackets found by counting over each column instead of a walk, and the
column, extrapolation and tie rules restated below.  :func:`ref_pressure`, :func:`ref_height` and :func:`ref_depth` return, per output
value, the ideal result, a derived error bound and an ambiguity flag with the candidate results; :func:`check` is the comparison rule.  :func:`draw_case` is the seeded case
generator that the CPU rehearsal (test_vertical_reference_host.py) and the GPU fuzz (test_gpu_vertical_fuzz.py) share.

Rules (DESIGN.md section 2), in the column's ascending coordinate (pressure p; altitude or height z; depth x = -z):

* a column whose end coordinates are equal or NaN is NaN; so is a height column whose surface level is NaN, and an ocean column with
  h NaN or <= 0 or a NaN eta.  A NaN level ends the walk of the height branch: every pair at or above it gives NaN;
* inside the range the bracket is the pair that holds the target, endpoints included; a target equal to an inner level takes the
  pair below it in walk order (height, depth; pressure on columns whose p increases with k) or above it (pressure on columns whose p
  decreases with k: the smallest k); outside, the end pair on that side (``extrapolate``) or NaN;
* ``w = (X - x_a) / (x_b - x_a)`` with x = p, ln p or ln ln p (pressure) or the coordinate itself, ``out = A + w (B - A)``, NaN when A
  or B is; nearest neighbour takes the level nearer in the search coordinate (p, z, x), on a tie the lower k (pressure) or the level
  earlier in walk order (height, depth).

The error bound.  u = 2^-53.  The kernel evaluates every coordinate in fp64, each operation rounded (|fl(a o b) - a o b| <= u |a o b|),
``vlog`` and ``vexp`` within 1 ulp <= 2u |result|, and the constants it forms from decimals (H = R*/(M g0), c_b = T_b/L_b,
e_b = -(R* L_b)/(g0 M), c = M/M_w - 1) within 4u relative (three decimal roundings of u/2 and two operations), H T_b within 6u.
Propagating these to first order through the formulas of DESIGN section 2, operation by operation, gives e_k >= |x_k(fp64) - x_k|
for every level coordinate and e_X for the target coordinate:

* pressure: q = ps s - shift: e_q = u |ps s| + u |q|; p = a + b q: e_p = |b| e_q + u |b q| + u |p| (0 for pressure levels); ln p:
  e_p / p + 2u |ln p|; ln ln p: e_ln / |ln p| + 2u |ln ln p|;
* standard atmosphere: r = ln(p/p_b): e_r = e_p/p + 1.5u + 2u |r|, then y = e r, exp(y), c (exp(y) - 1), h + ... each adding its
  rounding and constant error; where the fp64 p may fall in the other layer (|p - p_b| <= e_p + |p_b - fl(p_b)|) the difference
  of the two layers' altitudes is added;
* hypsometric: Tv = T (1 + c q) within (5u |c q| / (1 + c q) + 2u) Tv, each layer's H 0.5 (Tv + Tv') within 6u + that, ln of the
  pressure ratio within the two levels' e_p / p + u + 2u |ln|, and the K-level sum accumulates e_z_m = e_z_{m-1} + e_dz_m + u |z_m|;
* field: u |z|; height targets add u |z_s| + u |z - z_s|; ocean sigma, g1 and g2 the roundings of each operation of their formulas.

Every e is then multiplied by 1 + 2^-20, which covers the second-order terms (O(u^2) against O(u)).  The weight error follows from
those of its numerator N = X - x_a and denominator D = x_b - x_a: e_N = e_X + e_a + u |N|, e_D = e_a + e_b + u |D|,
e_w = (e_N + |w| e_D) / (|D| (1 - e_D/|D|)) (1 + u) + u |w|.  The fp64 result differs from A + w (B - A) by at most
E = |B - A| e_w (1 + 4u) + 2u |w| |B - A| + 2u |A + w (B - A)|, and rounding it to float32 adds at most 2^-24 (|r| + E).  The bound
is (E + 2^-24 (|r| + E)) (1 + 2^-8) + 2^-149: the last factor covers the reference's own longdouble rounding (2^-64 per operation
against the 2^-53 of the terms above), the last term float32's smallest step.

Ambiguity.  Two fp64 quantities whose ideal values differ by less than the sum of their bounds may compare either way.  A value is
ambiguous when a level's coordinate lies within e_X + e_k of the target (the bracket or the in-range decision could go either way;
both decisions are candidates), or when the two nearest-neighbour distances lie within their summed bounds of each other (both picks
are candidates).  A bound of exactly 0 is no ambiguity: the decision is exact.  Targets equal to the source levels of pressure-level
and depth-level sources are such exact hits (both sides compute the two coordinates from the same double), and their result is the
level's value exactly: bound 0.  The check requires levels farther apart than their bounds (asserted per case); columns that are not
monotone are outside the contract and never generated.

Not compared here: loglog with pressures <= 1 hPa (ln ln p is -inf or NaN; the GPU and the oracle agree on NaN / +-inf, pinned
separately), and NaN payloads (the oracle comparison pins those).
"""
from __future__ import annotations

import dataclasses

import numpy as np

LD = np.longdouble
U = 2.0 ** -53
SECOND_ORDER = 1.0 + 2.0 ** -20
REF_SLACK = 1.0 + 2.0 ** -8

LIN, LOG, LOGLOG, NN = 0, 1, 2, 3
METHOD_NAMES = {"linear": LIN, "log": LOG, "loglog": LOGLOG, "nearestneighbor": NN}

# US Standard Atmosphere 1976 / ICAO, as published (DESIGN.md section 2), parsed as decimals in extended precision
_HB = np.array([LD(v) for v in ("0", "11000", "20000", "32000", "47000", "51000", "71000")])
_TB = np.array([LD(v) for v in ("288.15", "216.65", "216.65", "228.65", "270.65", "270.65", "214.65")])
_LB = np.array([LD(v) for v in ("-6.5e-3", "0", "1e-3", "2.8e-3", "0", "-2.8e-3", "-2e-3")])
_PB = np.array([LD(v) for v in ("1013.25", "226.3206", "54.74889", "8.680187", "1.109063", "0.6693887", "0.03956420")])
_PB64 = np.array([1013.25, 226.3206, 54.74889, 8.680187, 1.109063, 0.6693887, 0.03956420])
_R, _M, _MW, _G0 = LD("8.31432"), LD("0.0289644"), LD("0.01801528"), LD("9.80665")
_H = _R / (_M * _G0)
_CQ = _M / _MW - 1


def _f(a):
    """longdouble -> float64 magnitudes for the error terms"""
    return np.abs(np.asarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------------- coordinates
def pressure_levels(kind, a, b, ptop, ps_scale, ps):
    """p [ncol][nk] (longdouble) and its bound: kind 0 pressure levels (a), 1 hybrid (a = ap, b), 2 sigma (b = sigma, ptop); ps [ncol]"""
    a = np.asarray(a, np.float64) if a is not None else None
    if kind == 0:
        p = np.broadcast_to(a.astype(LD)[None, :], (ps.size, a.size)).copy()
        return p, np.zeros(p.shape)
    bb = np.asarray(b, np.float64).astype(LD)[None, :]
    psd = ps.astype(np.float64).astype(LD)[:, None] * LD(ps_scale)
    shift = LD(ptop) if kind == 2 else LD(0)
    q = psd - shift
    aa = (np.full(bb.shape, ptop, np.float64) if kind == 2 else a[None, :]).astype(LD)
    p = aa + bb * q
    eq = U * _f(psd) + (U * _f(q) if kind == 2 else 0.0)
    ep = _f(bb) * eq + U * _f(bb * q) + U * _f(p)
    return p, ep * SECOND_ORDER


def _ln(x, ex):
    """ln x and its bound from that of x"""
    with np.errstate(divide="ignore", invalid="ignore"):
        lx = np.log(x)
        return lx, ex / _f(x) + 2 * U * _f(lx)


def _zstd_layer(p, ep, b):
    """the standard atmosphere's altitude of p in layer b (arrays) and its bound"""
    hb, pb, Lb, Tb = _HB[b], _PB[b], _LB[b], _TB[b]
    lapse = Lb != 0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.log(p / pb)
        er = ep / _f(p) + 1.5 * U + 2 * U * _f(r)
        e = np.where(lapse, -(_R * Lb) / (_G0 * _M), LD(0))
        c = np.where(lapse, Tb / np.where(lapse, Lb, LD(1)), _H * Tb)
        y = e * r
        ey = _f(e) * er + 5 * U * _f(y)
        E = np.exp(y)
        eE = _f(E) * ey + 2 * U * _f(E)
        cE = c * (E - 1)
        ecE = _f(c) * (eE + U * _f(E - 1)) + 5 * U * _f(cE)
        # L_b = 0: c = H T_b (6u), r2 = ln(p_b / p) = -r
        cr = c * (-r)
        ecr = _f(c) * er + 7 * U * _f(cr)
        dz = np.where(lapse, cE, cr)
        edz = np.where(lapse, ecE, ecr)
    z = hb + dz
    return z, edz + U * _f(z)


def standard_altitude(p, ep):
    """z of every p [m] (longdouble) and its bound: the last layer b with p <= p_b"""
    with np.errstate(invalid="ignore"):
        b = np.zeros(p.shape, dtype=np.int64)
        for lyr in range(1, 7):
            b = np.where(p <= _PB[lyr], lyr, b)
        z, ez = _zstd_layer(p, ep, b)
        # where the fp64 p may sit in the neighbouring layer, the two layers' altitudes differ by the rounding of the published p_b
        for lyr in range(1, 7):
            near = np.abs(np.asarray(p - _PB[lyr], np.float64)) <= ep + abs(float(_PB[lyr] - LD(_PB64[lyr]))) + U * _PB64[lyr]
            if near.any():
                other = np.where(b == lyr, lyr - 1, lyr)
                z2, ez2 = _zstd_layer(p, ep, other)
                ez = np.where(near, ez + np.maximum(ez2, 0) + _f(z2 - z), ez)
    return z, ez * SECOND_ORDER


def hypsometric_altitude(p, ep, up, psd, t, q, zadd):
    """the hypsometric sum upward from the surface: p, ep, t, q [ncol][nk] (q may be None); up [ncol]: level 0 is the surface;
    psd = ps ps_scale [ncol] (longdouble); zadd [ncol] (z_s or 0).  z [ncol][nk] in index order and its bound"""
    nk = p.shape[1]
    order = np.where(up[:, None], np.arange(nk)[None, :], nk - 1 - np.arange(nk)[None, :])
    pw = np.take_along_axis(p, order, 1)
    epw = np.take_along_axis(ep, order, 1)
    T = np.take_along_axis(t.astype(np.float64).astype(LD), order, 1)
    if q is not None:
        qq = np.take_along_axis(q.astype(np.float64).astype(LD), order, 1)
        cq = _CQ * qq
        tv = T * (1 + cq)
        with np.errstate(invalid="ignore", divide="ignore"):
            etv_rel = 5 * U * _f(cq) / _f(1 + cq) + 2 * U
    else:
        tv = T
        etv_rel = np.zeros(T.shape)
    with np.errstate(invalid="ignore", divide="ignore"):
        hterm = np.empty(tv.shape, dtype=LD)
        hterm[:, 0] = _H * tv[:, 0]
        hterm[:, 1:] = _H * (LD(0.5) * (tv[:, 1:] + tv[:, :-1]))
        eh_rel = np.empty(etv_rel.shape)
        eh_rel[:, 0] = 5 * U + etv_rel[:, 0]
        eh_rel[:, 1:] = 6 * U + np.maximum(etv_rel[:, 1:], etv_rel[:, :-1])
        prev = np.concatenate([psd[:, None], pw[:, :-1]], axis=1)
        eprev = np.concatenate([U * _f(psd)[:, None], epw[:, :-1]], axis=1)
        L = np.log(prev / pw)
        eL = eprev / _f(prev) + epw / _f(pw) + U + 2 * U * _f(L)
        dz = hterm * L
        edz = _f(hterm) * eL + _f(dz) * (eh_rel + U)
        zw = zadd[:, None] + np.cumsum(dz, axis=1)
        ezw = U * _f(zadd)[:, None] + np.cumsum(edz + U * _f(zw), axis=1)
    z = np.empty_like(zw)
    ez = np.empty_like(ezw)
    np.put_along_axis(z, order, zw, 1)
    np.put_along_axis(ez, order, ezw, 1)
    return z, ez * SECOND_ORDER


def ocean_depth(vcoord, s, Ck, depth_c, h, eta):
    """x = -z [ncol][nk] (longdouble) and its bound: vcoord 3 depth levels, 4 ocean sigma, 5 g1, 6 g2; h, eta [ncol] float64"""
    s = np.asarray(s, np.float64)
    if vcoord == 3:
        x = np.broadcast_to(s.astype(LD)[None, :], (h.size, s.size)).copy()
        return x, np.zeros(x.shape)
    hh = h.astype(LD)[:, None]
    e = eta.astype(LD)[:, None]
    sk = s.astype(LD)[None, :]
    with np.errstate(invalid="ignore", divide="ignore"):
        if vcoord == 4:
            eh = e + hh
            t = sk * eh
            z = e + t
            ez = _f(sk) * U * _f(eh) + U * _f(t) + U * _f(z)
        else:
            C = np.asarray(Ck, np.float64).astype(LD)[None, :]
            dcs = LD(depth_c) * sk
            if vcoord == 5:
                hd = hh - LD(depth_c)
                S = dcs + hd * C
                eS = U * _f(dcs) + _f(C) * U * _f(hd) + U * _f(hd * C) + U * _f(S)
                ratio = S / hh
                eone = eS / _f(hh) + U * _f(ratio) + U * _f(1 + ratio)
                t = e * (1 + ratio)
                z = S + t
                ez = eS + _f(e) * eone + U * _f(t) + U * _f(z)
            else:
                num = dcs + hh * C
                den = LD(depth_c) + hh
                S = num / den
                enum = U * _f(dcs) + U * _f(hh * C) + U * _f(num)
                eS = (enum + _f(S) * U * _f(den)) / _f(den) + U * _f(S)
                eh = e + hh
                t = eh * S
                z = e + t
                ez = _f(eh) * eS + _f(S) * U * _f(eh) + U * _f(t) + U * _f(z)
    return -z, ez * SECOND_ORDER


# ---------------------------------------------------------------------------------------------------------------- the rules
@dataclasses.dataclass
class Reference:
    """per output value [nt][np][nxy]: the ideal result (NaN where the contract gives NaN), its bound, the ideal weight (NaN where no
    pair is used or for nearest neighbour), the ambiguity flag, the candidate results [...][4] (NaN-padded) with their bounds and
    validity, and whether the value is an exact hit"""
    value: np.ndarray
    bound: np.ndarray
    weight: np.ndarray
    ambiguous: np.ndarray
    cand: np.ndarray
    cand_bound: np.ndarray
    cand_ok: np.ndarray
    exact: np.ndarray


def _interpolate(S, eS, W, eW, V, valid, T, eT, TW, eTW, method, extrapolate, tie_first, nn_tie_lower, direct):
    """the rules on columns in ascending search coordinate S [ncol][nk] (weights in W), values V [ncol][nk] float64, targets T [np].
    tie_first [ncol]: a target on an inner level takes the pair below it; nn_tie_lower [ncol]: a nearest-neighbour tie takes the
    lower level; direct: the coordinates are the inputs themselves (pressure and depth levels)"""
    ncol, nk = S.shape
    npt = T.size
    with np.errstate(invalid="ignore"):
        isn = np.isnan(np.asarray(S, np.float64)) | ~valid[:, None]
    mnan = np.where(isn.any(1), isn.argmax(1), nk)  # first NaN level (0 for invalid columns)
    Sv = np.where(isn, LD(np.inf), S)  # NaN levels sort above everything for the counts
    cnt_lt = np.empty((ncol, npt), np.int64)
    cnt_le = np.empty((ncol, npt), np.int64)
    step = max(1, int(2e6 // max(1, nk * npt)))
    for c0 in range(0, ncol, step):
        blk = Sv[c0:c0 + step, None, :]
        cnt_lt[c0:c0 + step] = (blk < T[None, :, None]).sum(2)
        cnt_le[c0:c0 + step] = (blk <= T[None, :, None]).sum(2)
    top = np.maximum(mnan - 1, 0)[:, None]
    S0 = S[:, :1]
    Stop = np.take_along_axis(S, top, 1)
    M = mnan[:, None]

    def decide(lt, le, below, above):
        """pair index, or -1 for NaN, from the counts and the out-of-range flags"""
        inner = np.where(tie_first[:, None], lt - 1, le - 1)
        pair = np.clip(inner, 0, np.maximum(M - 2, 0))
        pair = np.where(below, 0 if extrapolate else -1, pair)
        pair = np.where(above, np.where((M == nk) & extrapolate, nk - 2, -1), pair)
        pair = np.where(pair + 1 < M, pair, -1)
        return np.where(valid[:, None] & (M > 0), pair, -1)

    below = T[None, :] < S0
    above = T[None, :] > Stop
    pair0 = decide(cnt_lt, cnt_le, below, above)
    # a level that could compare either way with the target: only the ends and the two levels of the pair can be that close
    pc = np.clip(pair0, 0, nk - 2)
    near_k = np.full((ncol, npt), -1, np.int64)
    for kk in (np.zeros_like(pc), np.broadcast_to(top, pc.shape), pc, pc + 1):
        Sk = np.take_along_axis(S, kk, 1)
        tol = (eT[None, :] + np.take_along_axis(eS, kk, 1)) * REF_SLACK
        with np.errstate(invalid="ignore"):
            nr = (tol > 0) & (_f(Sk - T[None, :]) <= tol) & (kk < M) & valid[:, None]
        near_k = np.where(nr & (near_k < 0), kk, near_k)
    amb_pair = near_k >= 0
    kk = np.maximum(near_k, 0)
    # the decisions for a target just below and just above that level
    nan_pair = np.full_like(kk, -1)
    pair_lo = np.where(kk == 0, 0 if extrapolate else -1, kk - 1)
    pair_hi = np.where(kk == M - 1, np.where((M == nk) & extrapolate, nk - 2, nan_pair), kk)
    pair_lo, pair_hi = [np.where(valid[:, None] & (pr >= 0) & (pr + 1 < M), pr, -1) for pr in (pair_lo, pair_hi)]
    pairs = [pair0, np.where(amb_pair, pair_lo, pair0), np.where(amb_pair, pair_hi, pair0)]

    cand, cbound, cok, weights = [], [], [], None
    exact_all = np.zeros((ncol, npt), bool)
    for pi, pr in enumerate(pairs):
        use = pr >= 0
        pa = np.clip(pr, 0, nk - 2)
        pb = pa + 1
        A = np.take_along_axis(V, pa, 1)
        B = np.take_along_axis(V, pb, 1)
        Sa, Sb = np.take_along_axis(S, pa, 1), np.take_along_axis(S, pb, 1)
        eSa, eSb = np.take_along_axis(eS, pa, 1), np.take_along_axis(eS, pb, 1)
        hit_a = direct & (Sa == T[None, :])
        hit_b = direct & (Sb == T[None, :])
        if method == NN:
            with np.errstate(invalid="ignore"):
                da, db = _f(T[None, :] - Sa), _f(Sb - T[None, :])
                ea = eT[None, :] + eSa + U * da
                eb = eT[None, :] + eSb + U * db
                tol = (ea + eb) * REF_SLACK
                amb_nn = (tol > 0) & (np.abs(da - db) <= tol) & ~(hit_a | hit_b)
                # exact comparison of the ideal distances; a tie takes the lower level (nn_tie_lower) or the upper one
                dA, dB = np.abs(T[None, :] - Sa), np.abs(Sb - T[None, :])
                pick_b = np.where(nn_tie_lower[:, None], dB < dA, dB <= dA)
            for pick, extra in ((pick_b, None), (~pick_b, amb_nn)):
                val = np.where(pick, B, A)
                cand.append(np.where(use, val, np.nan))
                cbound.append(np.zeros((ncol, npt)))
                cok.append(np.ones((ncol, npt), bool) if extra is None else (extra & use))
            if pi == 0:
                weights = np.full((ncol, npt), np.nan)
                exact_all = use & (hit_a | hit_b)
            continue
        Wa, Wb = np.take_along_axis(W, pa, 1), np.take_along_axis(W, pb, 1)
        eWa, eWb = np.take_along_axis(eW, pa, 1), np.take_along_axis(eW, pb, 1)
        with np.errstate(invalid="ignore", divide="ignore"):
            N = TW[None, :] - Wa
            D = Wb - Wa
            w = np.where(D == 0, LD(0), N / D)
            r = A.astype(LD) + w * (B.astype(LD) - A.astype(LD))
            eN = eTW[None, :] + eWa + U * _f(N)
            eD = eWa + eWb + U * _f(D)
            absD = _f(D)
            ew = (eN + _f(w) * eD) / (absD * (1 - eD / absD)) * (1 + U) + U * _f(w)
            BA = np.abs(B - A)
            E = BA * ew * (1 + 4 * U) + 2 * U * _f(w) * BA + 2 * U * _f(r)
            bound = (E + 2.0 ** -24 * (_f(r) + E)) * REF_SLACK + 2.0 ** -149
        hit = use & (hit_a | hit_b)
        r64 = np.where(hit_a, A + 0 * B, np.where(hit_b, B + 0 * A, np.asarray(r, np.float64)))  # NaN if either is
        bound = np.where(hit, 0.0, bound)
        nan_val = np.isnan(A) | np.isnan(B)
        cand.append(np.where(use & ~nan_val, r64, np.nan))
        cbound.append(np.where(use & ~nan_val, bound, 0.0))
        cok.append(np.ones((ncol, npt), bool))
        if pi == 0:
            weights = np.where(use, np.asarray(w, np.float64), np.nan)
            exact_all = hit
    cand = np.stack(cand, -1)
    cbound = np.stack(cbound, -1)
    cok = np.stack(cok, -1)
    # candidates: the ideal decision first; then the alternative pairs (and, for nearest neighbour, each pair's other pick)
    cok[..., (2 if method == NN else 1):] &= amb_pair[..., None]
    ambiguous = cok[..., 1:].any(-1)
    return cand[..., 0], cbound[..., 0], weights, ambiguous, cand, cbound, cok, exact_all


def _ascending(x, ex, V, up):
    """reorder [ncol][nk] arrays so that the coordinate ascends (up [ncol]: it already does in k)"""
    nk = x.shape[1]
    order = np.where(up[:, None], np.arange(nk)[None, :], nk - 1 - np.arange(nk)[None, :])
    return [np.take_along_axis(a, order, 1) for a in (x, ex, V)]


def _finish(parts, nt, nxy):
    value, bound, weight, amb, cand, cb, cok, exact = parts
    npt = value.shape[1]

    def shape(a):  # [nt * nxy][np][...] -> [nt][np][nxy][...]
        return np.moveaxis(a.reshape((nt, nxy, npt) + a.shape[2:]), 1, 2)
    return Reference(*(shape(a) for a in (value, bound, weight, amb, cand, cb, cok, exact)))


def _columns(field):
    """[nt][nk][nxy] -> [nt * nxy][nk] float64"""
    nt, nk = field.shape[:2]
    return np.moveaxis(np.asarray(field, np.float32).reshape(nt, nk, -1), 1, 2).reshape(-1, nk).astype(np.float64)


def ref_pressure(method, kind, ap, b, levels, field, ps=None, ptop=0.0, ps_scale=1.0, extrapolate=True):
    """the pressure branch; arguments as vertical_oracle.vinterp"""
    nt, nk = field.shape[:2]
    nxy = int(np.prod(field.shape[2:]))
    V = _columns(field)
    psc = np.zeros(nt * nxy, np.float32) if ps is None else np.asarray(ps, np.float32).reshape(-1)
    p, ep = pressure_levels(kind, ap, b, ptop, ps_scale, psc)
    with np.errstate(invalid="ignore"):
        incr = p[:, 0] < p[:, -1]
        valid = incr | (p[:, 0] > p[:, -1])
    S, eS, Va = _ascending(p, ep, V, incr)
    P = np.asarray(levels, np.float64).astype(LD)
    eP = np.zeros(P.size)
    W, eW, TW, eTW = S, eS, P, eP
    if method in (LOG, LOGLOG):
        W, eW = _ln(S, eS)
        TW, eTW = _ln(P, eP)
        if method == LOGLOG:
            with np.errstate(invalid="ignore", divide="ignore"):
                W, eW = _ln(W, eW)
                TW, eTW = _ln(TW, eTW)
            assert np.all(np.asarray(P) > 1) and not np.any(valid[:, None] & (np.asarray(S, np.float64) <= 1)), \
                "loglog at pressures <= 1 is outside the compared contract"
    _separated(S, eS, valid)
    parts = _interpolate(S, eS, W, eW, Va, valid, P, eP, TW, eTW, method, extrapolate, tie_first=incr, nn_tie_lower=incr, direct=kind == 0)
    return _finish(parts, nt, nxy)


def _separated(S, eS, valid):
    """the case is inside the compared contract: every valid column strictly monotone, its levels farther apart than their bounds"""
    with np.errstate(invalid="ignore"):
        d = np.asarray(S[:, 1:] - S[:, :-1], np.float64)
        ok = ~(d <= (eS[:, 1:] + eS[:, :-1]) * REF_SLACK) | np.isnan(d)
    assert np.all(ok[valid]), "generated column not monotone beyond its error bound"


def ref_height(method, converter, target, kind, ap, b, levels, field, ps=None, t=None, q=None, z=None, zs=None, ptop=0.0, ps_scale=1.0,
               z_scale=1.0, zs_scale=1.0, extrapolate=True):
    """the height branch; arguments as vertical_height_oracle.vinterp_height (converter 0 standard, 1 hypsometric, 2 field; target
    0 altitude, 1 height)"""
    nt, nk = field.shape[:2]
    nxy = int(np.prod(field.shape[2:]))
    ncol = nt * nxy
    V = _columns(field)
    zsd = np.zeros(ncol, dtype=LD) if zs is None else np.tile(np.asarray(zs, np.float32).reshape(-1).astype(np.float64), nt).astype(LD) * LD(zs_scale)
    hyps = converter == 1
    if converter == 2:
        zc = _columns(z).astype(LD) * LD(z_scale)
        ez = U * _f(zc)
        with np.errstate(invalid="ignore"):
            up = zc[:, 0] < zc[:, -1]
            valid = up | (zc[:, 0] > zc[:, -1])
    else:
        psc = np.zeros(ncol, np.float32) if ps is None else np.asarray(ps, np.float32).reshape(-1)
        p, ep = pressure_levels(kind, ap, b, ptop, ps_scale, psc)
        with np.errstate(invalid="ignore"):
            up = p[:, 0] > p[:, -1]
            valid = up | (p[:, 0] < p[:, -1])
        if converter == 0:
            zc, ez = standard_altitude(p, ep)
        else:
            psd = psc.astype(np.float64).astype(LD) * LD(ps_scale)
            zadd = zsd if target == 0 else np.zeros(ncol, dtype=LD)
            zc, ez = hypsometric_altitude(p, ep, up, psd, _columns(t), None if q is None else _columns(q), zadd)
    if target == 1 and not hyps:
        zr = zc - zsd[:, None]
        ez = ez + U * _f(zsd)[:, None] + U * _f(zr)
        zc = zr
    S, eS, Va = _ascending(zc, ez, V, up)
    with np.errstate(invalid="ignore"):
        valid = valid & ~np.isnan(np.asarray(S[:, 0], np.float64))
    _separated(S, eS, valid)
    Z = np.asarray(levels, np.float64).astype(LD)
    eZ = np.zeros(Z.size)
    ones = np.ones(ncol, bool)
    parts = _interpolate(S, eS, S, eS, Va, valid, Z, eZ, Z, eZ, method, extrapolate, tie_first=ones, nn_tie_lower=ones, direct=False)
    return _finish(parts, nt, nxy)


def ref_depth(method, vcoord, s, Cs, levels, field, eta=None, depth=None, depth_c=0.0, extrapolate=True):
    """the depth branch; arguments as vertical_depth_oracle.vinterp_depth"""
    nt, nk = field.shape[:2]
    nxy = int(np.prod(field.shape[2:]))
    ncol = nt * nxy
    V = _columns(field)
    h = np.zeros(ncol) if depth is None else np.tile(np.asarray(depth, np.float32).reshape(-1).astype(np.float64), nt)
    e = np.zeros(ncol) if eta is None else np.asarray(eta, np.float32).reshape(-1).astype(np.float64)
    x, ex = ocean_depth(vcoord, s, Cs, depth_c, h, e)
    with np.errstate(invalid="ignore"):
        up = x[:, 0] < x[:, -1]
        valid = up | (x[:, 0] > x[:, -1])
        if vcoord != 3:
            valid &= (h > 0) & ~np.isnan(e)
    S, eS, Va = _ascending(x, ex, V, up)
    _separated(S, eS, valid)
    D = np.asarray(levels, np.float64).astype(LD)
    eD = np.zeros(D.size)
    ones = np.ones(ncol, bool)
    parts = _interpolate(S, eS, S, eS, Va, valid, D, eD, D, eD, method, extrapolate, tie_first=ones, nn_tie_lower=ones, direct=vcoord == 3)
    return _finish(parts, nt, nxy)


# ---------------------------------------------------------------------------------------------------------------- the comparison
def check(got, ref: Reference, what="", max_ambiguous=0.01):
    """the comparison rule: unambiguous values within the bound (exact hits exactly) with identical NaN masks; ambiguous ones equal
    to one of the candidates (NaN to a NaN candidate, a value within that candidate's bound); at most `max_ambiguous` of the values
    ambiguous.  Returns (largest error as a fraction of its bound, the ambiguous share)."""
    g = np.asarray(got, np.float32).reshape(ref.value.shape).astype(np.float64)
    amb = ref.ambiguous
    share = float(amb.mean()) if amb.size else 0.0
    assert share <= max_ambiguous, f"{what}: {share:.3%} of the values are ambiguous"
    un = ~amb
    gn, rn = np.isnan(g), np.isnan(ref.value)
    bad = un & (gn != rn)
    assert not bad.any(), f"{what}: NaN masks differ at {np.argwhere(bad)[:5].tolist()}: got {g[bad][:5]}, want {ref.value[bad][:5]}"
    fin = un & ~gn
    err = np.abs(g - ref.value)
    over = fin & (err > ref.bound)
    assert not over.any(), (f"{what}: {int(over.sum())} values beyond the bound, first at {np.argwhere(over)[:3].tolist()}: got {g[over][:3]}, "
                            f"want {ref.value[over][:3]} +- {ref.bound[over][:3]}")
    ex = un & ref.exact
    assert np.all((g[ex] == ref.value[ex]) | (np.isnan(g[ex]) & np.isnan(ref.value[ex]))), f"{what}: an exact hit is not exact"
    if amb.any():
        ga = g[amb][:, None]
        c, cb, ok = ref.cand[amb], ref.cand_bound[amb], ref.cand_ok[amb]
        match = ok & ((np.isnan(ga) & np.isnan(c)) | (np.abs(ga - c) <= cb))
        miss = ~match.any(1)
        assert not miss.any(), f"{what}: {int(miss.sum())} ambiguous values match no candidate: got {ga[miss][:3, 0]}, candidates {c[miss][:3]}"
    with np.errstate(invalid="ignore", divide="ignore"):
        frac = np.where(fin & (ref.bound > 0), err / np.where(ref.bound > 0, ref.bound, 1), 0.0)
    return float(frac.max()) if frac.size else 0.0, share


# ---------------------------------------------------------------------------------------------------------------- the cases
G0 = 9.80665
NK = (2, 3, 17, 137, 1024)
NP = (1, 2, 37, 1024)
NXY = (1, 31, 255, 256, 257, 517, 4099)
NAN_SHARES = (0.0, 0.01, 0.2)


@dataclasses.dataclass
class Case:
    """one seeded case: `handle()` builds the fimex_b200 interpolator, `kwargs` are the per-slice inputs of its calls (numpy), `oracle`
    and `reference` compute the C restatement's result and the reference of a field [nt][nk][nxy]"""
    what: str
    key: str
    method: str
    field: np.ndarray
    kwargs: dict
    handle: object
    oracle: object
    reference: object


def _hybrid_table(nk, rng, top=2e-5):
    """a seeded, monotone hybrid table (hPa) shaped like ECMWF's: near-geometric aloft, dense near the ground, b = 0 above eta = 0.2"""
    u = np.cumsum(rng.uniform(0.6, 1.4, nk))
    u = (u - u[0]) / (u[-1] - u[0]) if nk > 1 else u
    eta = np.exp(np.log(top) * (1 - u) ** 1.6)
    b = np.clip((eta - 0.2) / 0.8, 0, None)
    return 1013.25 * (eta - b), b


def _targets(rng, n, lo, hi, ends, on_levels=None):
    """n targets: uniform in [lo, hi], some beyond both ends, some on source levels, some duplicated"""
    lev = rng.uniform(lo, hi, n)
    if n >= 2:
        lev[rng.random(n) < 0.1] = ends[0]
        lev[rng.random(n) < 0.1] = ends[1]
    if on_levels is not None and n >= 2:
        pick = rng.random(n) < 0.2
        lev[pick] = rng.choice(on_levels, int(pick.sum()))
    if n >= 3:
        dup = rng.random(n) < 0.1
        lev[dup] = rng.choice(lev, int(dup.sum()))
    return lev


def _nan(a, rng, share):
    a = a.copy()
    a[rng.random(a.shape) < share] = np.nan
    return a


def draw_case(seed, budget=1_000_000, branch=None):
    """the seeded case `seed`: branch, converter or source coordinate, method, extrapolation, direction, nk, np, nxy, nt and NaN shares
    drawn at random; nxy is reduced until nt * nxy * nk * np <= budget (the reference's counts are that large)"""
    import vertical_depth_oracle as vdo
    import vertical_height_oracle as vho
    import vertical_oracle as vpo
    import fimex_b200.vertical as V

    rng = np.random.default_rng(seed)
    branch = branch or ["pressure", "height", "depth"][rng.integers(3)]
    nk, npt = int(rng.choice(NK)), int(rng.choice(NP))
    nt = int(rng.integers(1, 6))
    nxys = [n for n in NXY if nt * n * nk * npt <= budget] or [1]
    nxy = int(rng.choice(nxys))
    extrapolate = bool(rng.integers(2))
    down = bool(rng.integers(2))
    nan_share = float(rng.choice(NAN_SHARES))
    field = _nan(rng.normal(250, 30, (nt, nk, nxy)).astype(np.float32), rng, nan_share)
    what = f"seed {seed}: {branch} nt={nt} nk={nk} np={npt} nxy={nxy} extrapolate={extrapolate} down={down} nan={nan_share}"
    flip = (lambda a: a[::-1].copy()) if down else (lambda a: a)

    if branch == "pressure":
        method = ["linear", "log", "loglog", "nearestneighbor"][rng.integers(4)]
        kind = int(rng.integers(3))
        loglog = method == "loglog"
        ap, b = _hybrid_table(nk, rng, top=2e-3 if loglog else 2e-5)  # loglog: every pressure above 1 hPa
        ps_scale = float(rng.choice([1.0, 0.01]))
        ps = _nan(rng.uniform(480, 1040, (nt, nxy)).astype(np.float32), rng, nan_share / 4)
        if ps_scale != 1.0:
            ps = (ps.astype(np.float64) * 100).astype(np.float32)
        ptop = 0.0
        if kind == 0:
            p = flip(ap + b * 1013.25)
            name, terms, oap, ob = V.PRESSURE, {"p": p}, p, None
            on = p
        elif kind == 1:
            name, terms, oap, ob, on = V.HYBRID, {"ap": flip(ap), "b": flip(b)}, flip(ap), flip(b), None
        else:
            ptop = 5.0
            sigma = flip(np.linspace(0.0, 1.0, nk) ** 1.3)
            name, terms, oap, ob, on = V.SIGMA, {"sigma": sigma, "ptop": ptop}, None, sigma, None
        lo = 1.5 if loglog else 0.5
        levels = _targets(rng, npt, lo, 1100, (1.2 if loglog else 0.005, 1200.0), on)
        m = METHOD_NAMES[method]
        return Case(what + f" {method} kind={kind} ps_scale={ps_scale}", f"pressure {method} kind={kind}", method, field, {"ps": ps},
                    lambda: V.VerticalInterpolator(name, terms, method, levels, ps_scale=ps_scale, extrapolate=extrapolate),
                    lambda f: vpo.vinterp(m, kind, oap, ob, levels, f, ps=ps, ptop=ptop, ps_scale=ps_scale, extrapolate=extrapolate),
                    lambda f: ref_pressure(m, kind, oap, ob, levels, f, ps=ps, ptop=ptop, ps_scale=ps_scale, extrapolate=extrapolate))

    if branch == "height":
        method = ["linear", "nearestneighbor"][rng.integers(2)]
        converter = int(rng.integers(3))
        target = int(rng.integers(2))
        kind = int(rng.integers(1, 3)) if converter == 1 else int(rng.integers(3))
        ap, b = _hybrid_table(nk, rng)
        ptop = 0.0
        if kind == 0:
            oap, ob = ap + b * 1013.25, None
            name, terms = V.PRESSURE, {"p": flip(oap)}
        elif kind == 1:
            oap, ob = ap, b
            name, terms = V.HYBRID, {"ap": flip(ap), "b": flip(b)}
        else:
            ptop = 5.0
            oap, ob = None, np.linspace(0.0, 1.0, nk) ** 1.3
            name, terms = V.SIGMA, {"sigma": flip(ob), "ptop": ptop}
        oap = None if oap is None else flip(oap)
        ob = None if ob is None else flip(ob)
        ps = rng.uniform(480, 1040, (nt, nxy)).astype(np.float32)
        psd = ps.astype(np.float64)[:, None, :]
        p = (np.broadcast_to(oap[None, :, None], (nt, nk, nxy)) if kind == 0 else
             oap[None, :, None] + ob[None, :, None] * psd if kind == 1 else ptop + ob[None, :, None] * (psd - ptop))
        zstd = 44330.8 * (1 - (p / 1013.25) ** 0.190263)
        t = _nan((np.maximum(288.15 - 6.5e-3 * zstd, 210.0) + rng.normal(0, 1.5, p.shape)).astype(np.float32), rng, nan_share / 20)
        q = _nan((rng.uniform(0, 0.02, p.shape) * np.exp(-np.maximum(zstd, 0) / 2500)).astype(np.float32), rng, nan_share / 20)
        if rng.integers(2):
            q = None
        z = _nan((zstd * G0).astype(np.float32), rng, nan_share / 20)
        zs = _nan((rng.uniform(-50, 2500, nxy) * G0).astype(np.float32), rng, nan_share / 4)
        ps = _nan(ps, rng, nan_share / 4)
        hyps, fld = converter == 1, converter == 2
        needs_zs = (target == 1) != hyps
        kw = {"ps": ps if (hyps or (converter == 0 and kind != 0)) else None, "t": t if hyps else None, "q": q if hyps else None,
              "z": z if fld else None, "zs": zs if needs_zs else None}
        levels = _targets(rng, npt, -200 if target == 0 else -50, 16000, (-2000.0, 1e5))
        tname = ["altitude", "height"][target]
        cname = ["standard", "hypsometric", "field"][converter]
        m = METHOD_NAMES[method]
        args = dict(ptop=ptop, z_scale=1 / G0, zs_scale=1 / G0, extrapolate=extrapolate)
        return Case(what + f" {method} {cname} {tname} kind={kind} q={q is not None}", f"height {method} {cname} {tname}", method, field,
                    {k: v for k, v in kw.items() if v is not None},
                    lambda: V.HeightInterpolator(name, terms, method, levels, type=tname, converter=cname, z_scale=1 / G0, zs_scale=1 / G0,
                                                 extrapolate=extrapolate),
                    lambda f: vho.vinterp_height(m, converter, target, kind, oap, ob, levels, f, **kw, **args),
                    lambda f: ref_height(m, converter, target, kind, oap, ob, levels, f, **kw, **args))

    method = ["linear", "nearestneighbor"][rng.integers(2)]
    vcoord = int(rng.integers(3, 7))
    h = rng.uniform(5, 3000, nxy)
    land = rng.random(nxy) < 0.3
    h[land] = rng.choice([0.0, np.nan, -3.0], int(land.sum()))
    h = h.astype(np.float32)
    eta = _nan(rng.uniform(-1.5, 1.5, (nt, nxy)).astype(np.float32), rng, nan_share / 4) if rng.integers(2) else None
    Cs, dc = None, 0.0
    if vcoord == 3:
        s = np.concatenate([[0.0], np.cumsum(rng.uniform(0.5, 1.5, nk - 1))])
        s = flip(s / s[-1] * rng.uniform(2000, 3500))
        name, terms, on = V.DEPTH, {"depth": s}, s
    elif vcoord == 4:
        s = flip(np.linspace(-1, 0, nk + 1)[:-1] + 0.5 / nk)
        name, terms, on = V.OCEAN_SIGMA, {"sigma": s}, None
    else:
        s, Cs = vdo.roms_stretching(nk, theta_s=rng.uniform(3, 8), theta_b=rng.uniform(0.1, 3))
        s, Cs = flip(s), flip(Cs)
        # g1 is monotone in k only where h >= depth_c (ROMS requires depth_c <= the shallowest sea floor)
        dc = float(rng.uniform(0, 1) * (np.nanmin(h[h > 0]) if vcoord == 5 and (h > 0).any() else rng.uniform(5, 300)))
        name = V.OCEAN_S_G1 if vcoord == 5 else V.OCEAN_S_G2
        terms, on = {"s": s, "C": Cs, "depth_c": dc}, None
    levels = _targets(rng, npt, -5, 3600, (-20.0, 5000.0), on)
    ocean = vcoord != 3
    kw = {"eta": eta if ocean else None, "depth": h if ocean else None}
    m = METHOD_NAMES[method]
    return Case(what + f" {method} vcoord={vcoord} eta={eta is not None}", f"depth {method} vcoord={vcoord}", method, field,
                {k: v for k, v in kw.items() if v is not None},
                lambda: V.DepthInterpolator(name, terms, method, levels, extrapolate=extrapolate),
                lambda f: vdo.vinterp_depth(m, vcoord, s, Cs, levels, f, eta=kw["eta"], depth=kw["depth"], depth_c=dc, extrapolate=extrapolate),
                lambda f: ref_depth(m, vcoord, s, Cs, levels, f, eta=kw["eta"], depth=kw["depth"], depth_c=dc, extrapolate=extrapolate))


def contraction_targets(n=8):
    """(levels, A, B, targets): pressure levels [100, 103] hPa with the values A, B, and n targets for which linear interpolation
    rounded as the contract says, fl(A + fl(w (B - A))), and contracted into one FMA, fl(A + w (B - A)), give different float32
    results.  Found by scanning, near float32 rounding midpoints m, the targets P whose weight w = (P - 100) / 3 puts A + w (B - A)
    closest to m (exact rational arithmetic for the FMA)."""
    from fractions import Fraction
    A, B = np.float32(250.0), np.float32(251.2345678)
    d = float(B) - float(A)  # exact
    found = []
    for j in range(0, 60000, 7):
        P0 = 100 + 3 * (250 + (j + 0.5) * 2.0 ** -16 - 250) / d
        for k in range(-150, 150):
            P = P0 + k * 2.0 ** -46  # ulp(P) on [64, 128)
            w = (P - 100.0) / 3.0
            if np.float32(float(A) + w * d) != np.float32(float(Fraction(float(A)) + Fraction(w) * Fraction(d))):
                found.append(P)
        if len(found) >= n:
            return np.array([100.0, 103.0]), A, B, np.array(found[:n])
    raise AssertionError("no targets found")
