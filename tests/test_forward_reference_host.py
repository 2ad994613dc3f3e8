"""CPU checks of forward interpolation's restatement (oracle/mifi_oracle.c) against tests/forward_reference.py, which is written
independently from the reference's per-cell definitions and calls the C++ library's own std::nth_element for the median.
No GPU needed."""
import itertools

import numpy as np
import pytest

import forward_reference as fr

NAN = np.float32(np.nan)
SYMBOLS = np.array([np.nan, -0.0, 0.0, 1.0, 2.0], dtype=np.float32)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("n", range(1, 9))
def test_introselect_every_permutation_of_small_multisets(oracle, n):
    """every ordering of every multiset of n <= 8 elements drawn from {NaN, -0, +0, 1, 2} -- that is, every word of length n --
    rearranged exactly as std::nth_element(v, v + n/2, v + n) rearranges it, element for element"""
    words = np.array(list(itertools.product(range(SYMBOLS.size), repeat=n)), dtype=np.int64)
    rows = SYMBOLS[words]
    for r in range(rows.shape[0]):
        got = oracle.nth_element(rows[r], n // 2)
        want = fr.nth_element(rows[r], n // 2)
        assert np.array_equal(_bits(got), _bits(want)), (rows[r], got, want)


def test_introselect_random_buckets(oracle):
    """10^4 buckets of up to 200 values with ties, NaN (both signs, several payloads), signed zeros, sorted and reversed runs"""
    rng = np.random.default_rng(2024)
    nans = np.array([0x7FC00000, 0xFFC00000, 0x7FC00001], dtype=np.uint32).view(np.float32)
    for case in range(10_000):
        n = int(rng.integers(1, 201))
        pool = np.concatenate([nans, np.array([-0.0, 0.0, 1.0, 2.0, -3.0], dtype=np.float32),
                               rng.normal(0, 2, int(rng.integers(1, 40))).astype(np.float32)])
        p = rng.random(pool.size) ** rng.uniform(0.2, 4.0)
        v = rng.choice(pool, n, p=p / p.sum())
        if case % 7 == 0:
            v = np.sort(v)
        elif case % 7 == 1:
            v = np.sort(v)[::-1].copy()
        nth = n // 2 if case % 3 else int(rng.integers(0, n))
        got, want = oracle.nth_element(v, nth), fr.nth_element(v, nth)
        assert np.array_equal(_bits(got), _bits(want)), (case, v, nth)


def test_median_known_answers(oracle):
    """std::nth_element picks NaN from {NaN, 3, 1, 2} and +0 from {-0, +0, +0, -0, 1}; a sort would pick 2, and the first
    equal element in input order would be 3 and -0"""
    a = np.array([np.nan, 3, 1, 2], dtype=np.float32)
    b = np.array([-0.0, 0.0, 0.0, -0.0, 1.0], dtype=np.float32)
    assert np.isnan(fr.nth_element(a, 2)[2]) and np.isnan(oracle.nth_element(a, 2)[2])
    assert _bits(fr.nth_element(b, 2)[2]) == 0 and _bits(oracle.nth_element(b, 2)[2]) == 0
    # the same through forward interpolation: every point in cell (0, 0) of a 2 x 1 grid
    for method, v, is_nan in ((fr.FORWARD_UNDEF_MEDIAN, a, True), (fr.FORWARD_MEDIAN, b, False)):
        px = np.zeros(v.size)
        want = fr.forward(method, px, px, 2, 1, v[None])
        got = oracle.forward_interpolate(method, px, px, v.size, 1, 2, 1, v[None])
        fr.assert_forward_equal(got, want, method, "known answer")
        assert np.isnan(got[0, 0, 0]) if is_nan else _bits(got[0, 0, 0]) == 0
    # forward_median drops the NaN: median of {3, 1, 2}
    assert oracle.forward_interpolate(fr.FORWARD_MEDIAN, np.zeros(4), np.zeros(4), 4, 1, 1, 1, a[None])[0, 0, 0] == 2


def test_round_and_clamp_against_oracle(oracle):
    pos = np.array([0.49999999999999994, 0.5, -0.5, -0.49999999999999994, 1.5, 2.5, 3.4999999999999996, 3.5, 4.5, 4.50000001, -0.0,
                    1e12, -1e12, 3e9, 2147483647.0, np.nan, np.inf, -np.inf, 4503599627370497.0])
    assert np.array_equal(fr.round_and_clamp(pos, 4), oracle.round_and_clamp(pos, 4))
    assert list(fr.round_and_clamp(pos[:10], 4)) == [0, 1, -1, 0, 2, 3, 3, 4, -1, -1]


@pytest.mark.parametrize("seed", range(200))
def test_oracle_forward_against_reference(oracle, seed):
    """orc_forward_interpolate == forward_reference.py, bit for bit; NaN payloads may differ only for sum and mean"""
    c = fr.make_case(seed)
    want = fr.forward(c["method"], c["px"], c["py"], c["outX"], c["outY"], c["data"])
    got = oracle.forward_interpolate(c["method"], c["px"], c["py"], c["inX"], c["inY"], c["outX"], c["outY"], c["data"])
    fr.assert_forward_equal(got, want, c["method"], f"seed {seed}")


def test_generator_covers_every_method_and_edge():
    cases = [fr.make_case(s) for s in range(200)]
    assert {c["method"] for c in cases} == set(fr.METHODS)
    cells = [c["outX"] * c["outY"] for c in cases]
    assert min(cells) < 4 and any(n >= 4 and n & (n - 1) == 0 for n in cells)
    assert any((c["px"] == -7.0).all() for c in cases)
    assert any(np.isnan(c["data"]).mean() > 0.2 for c in cases)
