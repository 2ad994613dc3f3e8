"""Host side of the merger on the GPU (fimex_b200/merger.py): the --merge.smoothing parser, and the numpy restatement of the linear
border smoothing (linear_border_smoothing, the reference tests/test_gpu_merge.py holds the kernel to) against an independent
per-cell loop written from the rule in DESIGN.md section 2 -- no GPU needed."""
import math

import numpy as np
import pytest

from fimex_b200.capi import FimexB200Error
from fimex_b200.merger import linear_border_smoothing, parse_smoothing


@pytest.mark.parametrize("spec,want", [("LINEAR(5,2)", (5, 2)), ("LINEAR(1,0)", (1, 0)), ("LINEAR(10,3)", (10, 3)), (" LINEAR( 12 , 0 ) ", (12, 0))])
def test_parse_smoothing_accepts(spec, want):
    assert parse_smoothing(spec) == want


@pytest.mark.parametrize("spec", ["LINEAR(0,2)", "LINEAR(5,-1)", "LINEAR(-5,2)", "LINEAR(5)", "LINEAR(5,2,1)", "LINEAR(2.5,1)", "LINEAR(5,2)x",
                                  "linear(5,2)", "COSINE(5,2)", "LINEAR", "", None, 5])
def test_parse_smoothing_refuses(spec):
    with pytest.raises(FimexB200Error):
        parse_smoothing(spec)


def scalar_smoothing(inner, outer, t, b, use_outer):
    """the rule cell by cell, in Python floats (fp64, no contraction)"""
    vi, vo = np.asarray(inner, dtype=np.float64), np.asarray(outer, dtype=np.float64)
    ny, nx = vi.shape[-2:]
    xmin1, xmax1, xmax2 = b, b + t, nx - b
    xmin2 = xmax2 - t
    ymin1, ymax1, ymax2 = b, b + t, ny - b
    ymin2 = ymax2 - t
    out = np.empty(vi.shape)
    for idx in np.ndindex(vi.shape[:-2]):
        for y in range(ny):
            for x in range(nx):
                dx = xmax1 - x if x < xmax1 else (x - xmin2 if x >= xmin2 else 0)
                dy = ymax1 - y if y < ymax1 else (y - ymin2 if y >= ymin2 else 0)
                alpha = min(max(math.sqrt(float(dx * dx + dy * dy)) / t, 0.0), 1.0)
                outside = x < xmin1 or x >= xmax2 or y < ymin1 or y >= ymax2
                inside = xmax1 <= x < xmin2 and ymax1 <= y < ymin2
                a, o = float(vi[idx + (y, x)]), float(vo[idx + (y, x)])
                if outside:
                    m = o
                elif inside:
                    m = a
                else:
                    d = o - a
                    m = o if d == 0 else a + alpha * d
                if math.isnan(o):
                    m = a
                if math.isnan(a):
                    m = o if use_outer else math.nan
                out[idx + (y, x)] = m
    return out


def fields(rng, shape):
    vi = rng.uniform(-50, 50, shape)
    vo = rng.uniform(-50, 50, shape)
    vi[rng.random(shape) < 0.1] = np.nan
    vo[rng.random(shape) < 0.1] = np.nan
    same = rng.random(shape) < 0.05  # vo - vi == 0: the outer value itself
    vo[same] = vi[same]
    return vi, vo


@pytest.mark.parametrize("use_outer", [True, False])
@pytest.mark.parametrize("t,b", [(1, 0), (5, 2), (10, 3)])
@pytest.mark.parametrize("shape", [(1, 1), (7, 2), (2, 7), (3, 11, 13), (19, 23), (30, 40), (2, 41, 37)])
def test_linear_border_smoothing_matches_the_rule(shape, t, b, use_outer):
    rng = np.random.default_rng(hash((shape, t, b, use_outer)) % 2**32)
    vi, vo = fields(rng, shape)
    got = linear_border_smoothing(vi, vo, t, b, use_outer)
    want = scalar_smoothing(vi, vo, t, b, use_outer)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(got.view(np.int64)[~np.isnan(got)], want.view(np.int64)[~np.isnan(want)])


def test_degenerate_grids_follow_the_formulas():
    # nx < 2 (b + t): the ramps of both edges overlap, there is no interior, and the blend still follows the per-cell rule
    vi, vo = np.full((4, 9), 10.0), np.full((4, 9), 20.0)
    got = linear_border_smoothing(vi, vo, 5, 2)
    assert not (got == 10.0).any()  # no interior cell
    assert np.array_equal(got, scalar_smoothing(vi, vo, 5, 2, True))
    # 1 x 1 with no border: x = 0 < xmax1 = t, the cell is in the ramp with alpha = 1 (sqrt(2) t / t clipped)
    assert linear_border_smoothing(np.array([[1.0]]), np.array([[3.0]]), 1, 0)[0, 0] == 3.0
