"""The independent reference of the vertical branches (tests/vertical_reference.py) against the C restatements on the CPU, and the
argument checks of the Python layer's device path (no GPU needed).

The restatements are bit-identical to the kernels (tests/test_gpu_vertical*.py), so the seeded cases, the reference and its derived
bound are validated here, on every branch, converter, source coordinate and method, before the GPU fuzz
(test_gpu_vertical_fuzz.py) runs the same cases against the kernels.  ``FIMEX_B200_VREF_SEEDS`` sets the number of seeds (default 200;
more: a one-off soak run)."""
import os

import numpy as np
import pytest

import vertical_oracle as vpo
import vertical_reference as vr

SEEDS = int(os.environ.get("FIMEX_B200_VREF_SEEDS", "200"))


def test_reference_agrees_with_the_restatements():
    """every seeded case: the restatement within the reference's bound (exact hits exactly), NaN masks identical, ambiguous values
    on a candidate and at most 1 % of them; together the seeds cover every branch x converter / source coordinate x method"""
    seen, worst, worst_share, exact = set(), 0.0, 0.0, 0
    for seed in range(SEEDS):
        case = vr.draw_case(seed)
        ref = case.reference(case.field)
        frac, share = vr.check(case.oracle(case.field), ref, case.what)
        worst, worst_share, exact = max(worst, frac), max(worst_share, share), exact + int(ref.exact.sum())
        seen.add(case.key)
    print(f"{SEEDS} seeds: largest error {worst:.3f} of the bound, largest ambiguous share {worst_share:.4%}, {exact} exact hits")
    assert exact > 0
    if SEEDS >= 200:
        want = {f"pressure {m} kind={k}" for m in vr.METHOD_NAMES for k in range(3)}
        want |= {f"height {m} {c} {t}" for m in ("linear", "nearestneighbor") for c in ("standard", "hypsometric", "field")
                 for t in ("altitude", "height")}
        want |= {f"depth {m} vcoord={v}" for m in ("linear", "nearestneighbor") for v in range(3, 7)}
        missing = want - seen
        assert not missing, f"the seeds miss {sorted(missing)}"


def test_reference_sees_a_wrong_bracket_and_a_wrong_weight():
    """the bound is tight enough that the results of a neighbouring bracket, and of targets moved by 2^-20 of their value, fail"""
    rng = np.random.default_rng(4)
    p = np.array([1000.0, 925.0, 850.0, 700.0, 500.0, 300.0])
    field = rng.normal(250, 30, (1, p.size, 64)).astype(np.float32)
    levels = np.array([990.0, 880.0, 600.0, 400.0])
    ref = vr.ref_pressure(vr.LOG, 0, p, None, levels, field)
    good = vpo.vinterp(vr.LOG, 0, p, None, levels, field)
    vr.check(good, ref, "restatement")
    shifted = vpo.vinterp(vr.LOG, 0, p, None, levels * (1 + 2.0 ** -20), field)
    with pytest.raises(AssertionError):
        vr.check(shifted, ref, "targets moved by 2^-20")
    wrong = vpo.vinterp(vr.LOG, 0, p, None, levels, np.concatenate([field[:, 1:], field[:, -1:]], 1))
    with pytest.raises(AssertionError):
        vr.check(wrong, ref, "the bracket one level up")


def test_targets_on_levels_are_exact_hits():
    """pressure and depth levels: a target equal to a level is that level's value, bit for bit, with either neighbour NaN or not"""
    rng = np.random.default_rng(8)
    p = np.array([1000.0, 925.0, 850.0, 700.0, 500.0, 300.0, 100.0])
    field = rng.normal(250, 30, (2, p.size, 40)).astype(np.float32)
    for method in (vr.LIN, vr.LOG, vr.LOGLOG, vr.NN):
        for levels in (p, p[::-1].copy()):
            ref = vr.ref_pressure(method, 0, levels, None, p, field)
            assert ref.exact.all() and (ref.bound == 0).all()
            # the level's own value (the other level of the pair is finite here)
            np.testing.assert_array_equal(ref.value, field[:, [list(levels).index(x) for x in p], :])
            vr.check(vpo.vinterp(method, 0, levels, None, p, field), ref, f"method {method}")


def test_loglog_at_and_below_one_hpa_is_nan_or_infinite():
    """loglog is ln ln p: ln ln 1 = -inf and ln ln p is NaN below 1 hPa.  A pair with a level at or below 1 hPa gives NaN; a target of
    exactly 1 hPa extrapolated from levels above 1 hPa gives -+inf (w = -inf).  The reference does not compare these; the GPU is
    pinned to the restatement on them (test_gpu_vertical_fuzz.py)."""
    field = np.array([[[200.0], [220.0], [260.0], [280.0]]], np.float32)
    era5_top = np.array([0.01, 0.5, 2.0, 10.0])
    out = vpo.vinterp(vr.LOGLOG, 0, era5_top, None, [0.3, 1.0, 1.5, 5.0], field)[0, :, 0]
    assert np.isnan(out[:3]).all() and np.isfinite(out[3])
    above = np.array([1.5, 2.0, 10.0, 50.0])
    out = vpo.vinterp(vr.LOGLOG, 0, above, None, [1.0, 1.2], field)[0, :, 0]
    assert out[0] == -np.inf and np.isfinite(out[1])  # 200 + (-inf) * (220 - 200)
    assert np.isnan(vpo.vinterp(vr.LOGLOG, 0, above, None, [1.0], field, extrapolate=False)[0, 0, 0])
    with pytest.raises(AssertionError, match="outside the compared contract"):
        vr.ref_pressure(vr.LOGLOG, 0, era5_top, None, [1.5, 5.0], field)


# ---------------------------------------------------------------------------------------------- the device path's argument checks
class _Recorder:
    """stands in for the C library: every function returns MIFI_OK and records its call"""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append(name)
            return 1
        return fn


def _fake_cuda(t):
    """a CPU tensor that reports itself as a CUDA tensor: the device path's checks run without a GPU (its address is never used
    because every call here must be refused)"""
    import torch

    class FakeCuda(torch.Tensor):
        @property
        def is_cuda(self):
            return True
    return torch.Tensor._make_subclass(FakeCuda, t)


@pytest.fixture
def recorder(monkeypatch):
    import fimex_b200.vertical as V
    rec = _Recorder()
    monkeypatch.setattr(V, "load", lambda: rec)
    return rec


def _bad(torch, n):
    """per-column inputs the C ABI would misread: on the host, float64, float16; each holds the right number of values"""
    return {"cpu": torch.zeros(n, dtype=torch.float32), "float64": _fake_cuda(torch.zeros(n, dtype=torch.float64)),
            "float16": _fake_cuda(torch.zeros(n, dtype=torch.float16))}


def test_device_path_refuses_ps_it_would_misread(recorder):
    """VerticalInterpolator's device calls take ps only as a float32 CUDA tensor: a host tensor would hand the kernel a host
    pointer, a float64 or float16 one would be read as float32; the C function is never called"""
    torch = pytest.importorskip("torch")
    import fimex_b200 as fb
    from fimex_b200.vertical import HYBRID, VerticalInterpolator
    vi = VerticalInterpolator(HYBRID, {"ap": np.array([0.0, 10.0, 100.0]), "b": np.array([1.0, 0.5, 0.0])}, "log", [500.0, 850.0])
    field = _fake_cuda(torch.zeros((2, 3, 5), dtype=torch.float32))
    recorder.calls.clear()
    for what, ps in _bad(torch, 10).items():
        with pytest.raises(fb.FimexB200Error, match="ps must be a float32 CUDA tensor"):
            vi.interpolateValues(field, ps.reshape(2, 5))
        with pytest.raises(fb.FimexB200Error, match="ps must be a float32 CUDA tensor"):
            vi.getDataSlice(field, ps.reshape(2, 5))
    with pytest.raises(fb.FimexB200Error):
        vi.interpolateValues(field, np.zeros((2, 5), np.float32))
    assert recorder.calls == []
    vi._h = None


def test_device_path_refuses_columns_it_would_misread(recorder):
    """the same for every per-column input of the height and depth calls (ps, t, q, z, zs; eta and the sea-floor depth)"""
    torch = pytest.importorskip("torch")
    import fimex_b200 as fb
    from fimex_b200.vertical import DepthInterpolator, HYBRID, HeightInterpolator, OCEAN_S_G2
    nt, nk, nxy = 2, 3, 5
    terms = {"ap": np.array([0.0, 10.0, 100.0]), "b": np.array([1.0, 0.5, 0.0])}
    field = _fake_cuda(torch.zeros((nt, nk, nxy), dtype=torch.float32))
    ok_level = _fake_cuda(torch.zeros(nt * nxy, dtype=torch.float32))
    ok_column = _fake_cuda(torch.zeros(nt * nk * nxy, dtype=torch.float32))
    ok_zs = _fake_cuda(torch.zeros(nxy, dtype=torch.float32))
    hyps = HeightInterpolator(HYBRID, terms, "linear", [10.0, 100.0], type="altitude", converter="hypsometric")
    fld = HeightInterpolator(HYBRID, terms, "linear", [10.0, 100.0], type="height", converter="field")
    dep = DepthInterpolator(OCEAN_S_G2, {"s": np.array([-0.9, -0.5, -0.1]), "C": np.array([-0.8, -0.4, -0.05]), "depth_c": 10.0}, "linear",
                            [1.0, 50.0])
    good = {hyps: {"ps": ok_level, "t": ok_column, "q": ok_column, "zs": ok_zs}, fld: {"z": ok_column, "zs": ok_zs},
            dep: {"eta": ok_level, "depth": ok_zs}}
    recorder.calls.clear()
    for h, kw in good.items():
        for name, a in kw.items():
            for what, bad in _bad(torch, a.numel()).items():
                args = dict(kw, **{name: bad})
                for call in (h.interpolateValues, h.getDataSlice):
                    with pytest.raises(fb.FimexB200Error, match=f"{name} must be a float32 CUDA tensor"):
                        call(field, **args)
    assert recorder.calls == []
    for h in good:
        h._h = None


def test_targets_on_computed_levels_are_ambiguous():
    """a target equal to a hybrid level as fp64 computes it lies within that level's bound: the bracket (and, without extrapolation at
    the column's end, the in-range decision) could go either way, so the value is ambiguous and the restatement gives one of the
    candidates"""
    rng = np.random.default_rng(12)
    ap, b = vr._hybrid_table(30, rng)
    ps = np.array([[987.6543]], np.float32)
    field = rng.normal(250, 30, (1, 30, 1)).astype(np.float32)
    field[0, 10, 0] = np.nan
    p64 = ap + b * np.float64(ps[0, 0])  # as the kernel forms p_k
    levels = p64[[3, 9, 11, 17, 29]]
    for method in (vr.LIN, vr.LOG, vr.NN):
        for extrapolate in (True, False):
            ref = vr.ref_pressure(method, 1, ap, b, levels, field, ps=ps, extrapolate=extrapolate)
            assert ref.ambiguous.all()
            vr.check(vpo.vinterp(method, 1, ap, b, levels, field, ps=ps, extrapolate=extrapolate), ref, f"method {method}", max_ambiguous=1.0)


def test_restatement_rounds_without_contraction():
    """targets whose result changes when the two-level formula is contracted into an FMA: the restatement gives the uncontracted
    float32 value (the GPU is pinned to it on the same targets, test_gpu_vertical_fuzz.py)"""
    levels, A, B, targets = vr.contraction_targets()
    field = np.array([[[A], [B]]], np.float32)
    got = vpo.vinterp(vr.LIN, 0, levels, None, targets, field)[0, :, 0]
    w = (targets - 100.0) / 3.0
    np.testing.assert_array_equal(got, (float(A) + w * (float(B) - float(A))).astype(np.float32))
