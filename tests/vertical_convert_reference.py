"""An independent high-precision reference for the vertical interpolator's data conversions (theta2T, omega2vwind, add4Dpressure) --
TEST INFRASTRUCTURE ONLY.

Written from the contract in DESIGN.md section 2, not from the C restatement (tests/vertical_convert_oracle.c): numpy ``longdouble``
(x87 extended, 64-bit significand), ``powl`` for (p / p0)^kappa instead of the written-out fdlibm ``vlog`` / ``vexp``, p_k formed in
longdouble, and the constants parsed from their decimal strings (kappa = 2/7, p0 = 1000 hPa, R* = 8.31432, M = 0.0289644,
g0 = 9.80665).  :func:`reference` returns, per value, the ideal result and an error bound; :func:`check` is the comparison rule;
:func:`draw_case` is the seeded case generator that the CPU rehearsal (test_vertical_convert_host.py) and the GPU fuzz
(test_gpu_vertical_convert.py) share.

The error bound.  u = 2^-53.  The kernel evaluates every operation in fp64, each rounded (|fl(a o b) - a o b| <= u |a o b|), ``vlog``
and ``vexp`` within 1 ulp <= 2u |result|, and reads the inputs as float (exact in fp64).  Operation by operation, to first order:

* p_k: psd = ps s within u |psd|; hybrid p = a + b psd: e_p = u |p| + 2u |b psd|; sigma q = psd - ptop within u |psd| + u |q|,
  p = ptop + b q: e_p = u |p| + |b| (2u |q| + u |psd|); pressure levels: e_p = 0 (p_k is the level as given);
* theta2T: r = p / p0 within the relative error d_r = u + e_p / |p|; L = vlog(r) within 2u |L| + d_r of ln(p / p0); kappa = fl(2/7)
  within u relative, m = kappa L within kappa (4u |L| + d_r); exp(m) within 2u relative plus the error of m; theta exp(m) adds u:
  the fp64 result lies within E = |T| (3u + kappa (4u |L| + d_r)) of the ideal T;
* omega2vwind: H = R* / (M g0) from three decimal constants (within u/2 each) and two operations: within 5u relative; H T,
  omega (H T), 100 p and the division one u each, and 100 p carries e_p / |p|: E = |w| (9u + e_p / |p|);
* add4Dpressure: E = e_p.

Every E is multiplied by 1 + 2^-20 (second-order terms).  Rounding the fp64 result to float32 adds at most half a float32 step at
|ideal| + E; the reference's own longdouble rounding (2^-64 per operation) is covered by the factor 1 + 2^-8 on the whole bound, and
2^-149 (float32's smallest step) is added.  A NaN input (theta, omega, T or ps) gives NaN and must give NaN; pressures p_k <= 0 are
outside this comparison (pinned GPU == restatement only) and never generated.
"""
from __future__ import annotations

import dataclasses

import numpy as np

import vertical_reference as vr

LD = np.longdouble
U = 2.0 ** -53
SECOND_ORDER = 1.0 + 2.0 ** -20
REF_SLACK = 1.0 + 2.0 ** -8

THETA2T, OMEGA2VWIND, PRESSURE = 0, 1, 2  # FB200_VCONV_*
OPS = {"theta2T": THETA2T, "omega2vwind": OMEGA2VWIND, "add4Dpressure": PRESSURE}
VCOORD_PRESSURE, VCOORD_HYBRID, VCOORD_SIGMA = 0, 1, 2

_KAPPA = LD(2) / LD(7)
_P0 = LD("1000")
_R, _M, _G0 = LD("8.31432"), LD("0.0289644"), LD("9.80665")
_KAPPA64 = 2.0 / 7.0


@dataclasses.dataclass
class Reference:
    ideal: np.ndarray  # longdouble [nt][nk][nxy]
    bound: np.ndarray  # float64, |float32 result - ideal| <= bound


def pressure(kind, a, b, ptop, ps_scale, ps, nk, nt, nxy):
    """(p_k in longdouble, its fp64 error bound e_p), both [nt][nk][nxy]"""
    if kind == VCOORD_PRESSURE:
        p = np.broadcast_to(np.asarray(a, dtype=LD).reshape(1, nk, 1), (nt, nk, nxy))
        return p, np.zeros(p.shape)
    psd = (np.asarray(ps, dtype=np.float32).astype(LD) * LD(ps_scale)).reshape(nt, 1, nxy)
    bb = np.asarray(b, dtype=LD).reshape(1, nk, 1)
    if kind == VCOORD_HYBRID:
        p = np.asarray(a, dtype=LD).reshape(1, nk, 1) + bb * psd
        e = U * np.abs(p) + 2 * U * np.abs(bb * psd)
    else:
        q = psd - LD(ptop)
        p = LD(ptop) + bb * q
        e = U * np.abs(p) + np.abs(bb) * (2 * U * np.abs(q) + U * np.abs(psd))
    return p, e.astype(np.float64) * SECOND_ORDER


def reference(op, kind, a, b, nk, field=None, ps=None, t=None, ptop=0.0, ps_scale=1.0, nt=None, nxy=None) -> Reference:
    """the ideal values [nt][nk][nxy] and their bounds; the shapes as vertical_convert_oracle.vconvert takes them"""
    if field is not None:
        x = np.asarray(field, dtype=np.float32)
        nt = x.shape[0]
        nxy = x.size // (nt * nk)
        x = x.reshape(nt, nk, nxy).astype(LD)
    elif ps is not None:
        nt = np.asarray(ps).shape[0]
        nxy = np.asarray(ps).size // nt
    p, ep = pressure(kind, a, b, ptop, ps_scale, ps, nk, nt, nxy)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        rel_p = ep / np.abs(p.astype(np.float64))
        if op == THETA2T:
            ideal = x * np.power(p / _P0, _KAPPA)  # powl
            L = np.abs(np.log((p / _P0).astype(np.float64)))
            E = np.abs(ideal.astype(np.float64)) * (3 * U + _KAPPA64 * (4 * U * L + U + rel_p))
        elif op == OMEGA2VWIND:
            T = np.asarray(t, dtype=np.float32).reshape(nt, nk, nxy).astype(LD)
            ideal = -(x * _R * T) / (_M * _G0 * LD(100) * p)
            E = np.abs(ideal.astype(np.float64)) * (9 * U + rel_p)
        else:
            ideal = np.array(p, dtype=LD)
            E = ep
        E = E * SECOND_ORDER
        mag = np.abs(ideal.astype(np.float64)) + E
        half_step = 0.5 * np.spacing(np.minimum(mag, np.finfo(np.float32).max).astype(np.float32)).astype(np.float64)
    return Reference(ideal=ideal, bound=(E + half_step) * REF_SLACK + 2.0 ** -149)


def check(got, ref: Reference, what=""):
    """every value within its bound, NaN exactly where the ideal is NaN; returns the largest error / bound"""
    g = np.asarray(got, dtype=np.float32).reshape(ref.ideal.shape)
    nan_i, nan_g = np.isnan(ref.ideal), np.isnan(g)
    bad = np.flatnonzero((nan_i != nan_g).ravel())
    assert bad.size == 0, f"{what}: NaN masks differ at {bad[:5]}: {g.ravel()[bad[:5]]} vs {ref.ideal.ravel()[bad[:5]]}"
    ok = ~nan_i
    err = np.abs(g[ok].astype(LD) - ref.ideal[ok]).astype(np.float64)
    ratio = err / ref.bound[ok]
    worst = float(ratio.max()) if ratio.size else 0.0
    if worst > 1.0:
        i = int(np.argmax(ratio))
        raise AssertionError(f"{what}: error {err[i]:.3e} exceeds the bound {ref.bound[ok][i]:.3e} (x{worst:.3f}); got {g[ok][i]!r}, "
                             f"ideal {ref.ideal[ok][i]!r}")
    return worst


# ------------------------------------------------------------------------------------------------------------ the seeded cases
@dataclasses.dataclass
class Case:
    op: int
    kind: int
    a: np.ndarray
    b: np.ndarray
    nk: int
    ptop: float
    ps_scale: float
    field: np.ndarray
    ps: np.ndarray
    t: np.ndarray

    def args(self):
        return dict(ptop=self.ptop, ps_scale=self.ps_scale)


def _nan(a, rng, share):
    if a is not None and share:
        a[rng.random(a.shape) < share] = np.nan
    return a


def draw_case(seed, budget=200_000, op=None, kind=None) -> Case:
    """one seeded case: every op x source coordinate; 1 to 137 levels; ps in hPa or Pa (ps_scale 0.01); a few NaN inputs"""
    rng = np.random.default_rng(seed)
    op = int(rng.integers(0, 3)) if op is None else op
    kind = int(rng.integers(0, 3)) if kind is None else kind
    nk = int(rng.choice([1, 2, 3, 17, 60, 137]))
    nxy = int(rng.choice([1, 31, 255, 257, 1031]))
    nt = max(1, min(int(rng.integers(1, 5)), budget // (nk * nxy)))
    ptop, pa = 0.0, rng.random() < 0.5
    ps_scale = 0.01 if pa else 1.0
    if kind == VCOORD_PRESSURE:
        a, b = np.sort(rng.uniform(1, 1100, nk))[::-1 if rng.random() < 0.5 else 1].copy(), None
    elif kind == VCOORD_HYBRID:
        a, b = vr._hybrid_table(max(nk, 2), rng)
        a, b = a[:nk].copy(), b[:nk].copy()
    else:
        a, b, ptop = None, np.sort(rng.uniform(0.0, 1.0, nk)), float(rng.uniform(0, 50))
    ps = None
    if kind != VCOORD_PRESSURE:
        ps = rng.uniform(480, 1060, (nt, nxy)).astype(np.float32)
        ps = (ps * 100).astype(np.float32) if pa else ps
        ps = _nan(ps, rng, rng.choice([0.0, 0.02]))
    shape = (nt, nk, nxy)
    field = t = None
    if op == THETA2T:
        field = rng.uniform(180, 1500, shape).astype(np.float32)
    elif op == OMEGA2VWIND:
        field = rng.normal(0, 1.5, shape).astype(np.float32)
        t = rng.uniform(180, 320, shape).astype(np.float32)
    share = rng.choice([0.0, 0.01])
    return Case(op, kind, a, b, nk, ptop, ps_scale, _nan(field, rng, share), ps, _nan(t, rng, share))
