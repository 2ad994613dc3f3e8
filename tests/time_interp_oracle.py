"""The restatement of time interpolation (DESIGN.md section 2, "time interpolation") -- TEST INFRASTRUCTURE ONLY (tests/ and
profiles/tools/time_interp_time.py).

It is built from pieces pinned elsewhere: the bracket rule of orc_vinterp_pressure (the smallest k with t_k <= tau <= t_k+1, the end
pair outside the range when extrapolating), the two-level step vertical_oracle.vint_values(LIN, ...) (orc_vint_value, pinned
against the reference's mifi_get_values_linear_f), and the typed adapters Oracle.as_float / from_float.
"""
from __future__ import annotations

import numpy as np

import vertical_oracle as vo


def time_map(times, new_times, extrapolate=True):
    """(ia, ib, w) per target: a linear scan for the smallest bracket, as orc_vinterp_pressure walks its levels"""
    t = np.asarray(times, dtype=np.float64)
    ia, ib, w = [], [], []
    for tau in np.asarray(new_times, dtype=np.float64).ravel():
        k = -1
        if tau < t[0] or tau > t[-1]:
            if extrapolate:
                k = 0 if tau < t[0] else t.size - 2
        else:
            for i in range(t.size - 1):
                if t[i] <= tau <= t[i + 1]:
                    k = i
                    break
        ia.append(k)
        ib.append(-1 if k < 0 else k + 1)
        w.append(0.0 if k < 0 else float((tau - t[k]) / (t[k + 1] - t[k])))
    return np.array(ia), np.array(ib), np.array(w)


def step(oracle, times, tau, k, a, b, bad, out_dtype):
    """one target step of bracket k (-1: none) from the raw slices a, b: as_float -> vint_values(LIN) -> from_float"""
    a = np.asarray(a)
    if k < 0:
        f = np.full(a.shape, np.nan, dtype=np.float32)
    else:
        fa, fb = oracle.as_float(a, bad).ravel(), oracle.as_float(np.asarray(b), bad).ravel()
        f = vo.vint_values(vo.LIN, fa, fb, float(times[k]), float(times[k + 1]), float(tau)).reshape(a.shape)
    return oracle.from_float(f, bad, out_dtype)


def stack(oracle, times, new_times, data, bad, out_dtype, extrapolate=True):
    """data [nt][...] -> [nt_new][...]"""
    ia, _, _ = time_map(times, new_times, extrapolate)
    data = np.asarray(data)
    out = np.empty((len(ia),) + data.shape[1:], dtype=np.dtype(out_dtype))
    for j, k in enumerate(ia):
        out[j] = step(oracle, times, new_times[j], k, data[max(k, 0)], data[max(k, 0) + 1], bad, out_dtype)
    return out
