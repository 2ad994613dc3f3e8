"""Vertical interpolation to height and altitude levels at ERA5 size: 1440 x 721 columns, 24 steps x 137 model levels.  Prints one JSON
line (and appends it to --out).

Two workloads:
* hypsometric: t and q integrated from the surface -> 15 heights above ground (10 m ... 5 km);
* standard: the standard-atmosphere altitude of each level's pressure -> flight levels FL050 ... FL450 (pressure altitudes, FL x 30.48 m).

The hybrid table is SYNTHETIC (seeded, monotone, shaped like ECMWF's L137; the real table is not in the repository), ps is one seeded
field with lows down to about 500 hPa, and t, q follow a standard lapse rate with seeded noise; ps, t and q are the same at every step,
the field differs.  Per workload: ms per step (CUDA events around the device call over all 24 steps, warmed up; the inputs, 13.7 GB
per 3-D field, are far larger than L2), values/s, algorithmic bytes 4 * nxy * nt * (P + K_field + n_aux * K_walk + 1) + 4 * nxy, with
K_field = the distinct field levels a column reads (its brackets), K_walk = the levels its walk reaches, n_aux = 2 (t, q) or 0, counted
here from the same inputs; the fraction of the HBM peak bench.py uses; the host-buffer call's end-to-end rate (pinned host arrays, 4
steps, copies inside the timed region) and the CPU oracle on all cores for one step, checked bit for bit against the GPU.

    python profiles/tools/vertical_height_time.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vertical_time import NK, NT, NX, NY, gpu_info, hybrid_table, surface_pressure  # noqa: E402

HEIGHTS = np.array([10, 20, 50, 100, 150, 200, 250, 300, 500, 750, 1000, 1500, 2000, 3000, 5000], dtype=np.float64)
FLIGHT_LEVELS = np.arange(50, 451, 10) * 30.48  # FL050 ... FL450 in metres
NT_HOST = 4
M = 0.0289644
HYPS = 8.31432 / (0.0289644 * 9.80665)  # R* / (M g0)


def column_inputs(torch, ap, b, ps, dev):
    """t [K] and q [kg/kg] of one step, [NK][nxy], seeded; and the column pressures [hPa]"""
    p = torch.from_numpy(ap).to(dev)[:, None] + torch.from_numpy(b).to(dev)[:, None] * ps.double()[None, :]
    z = 44330.8 * (1 - (p / 1013.25) ** 0.190263)
    g = torch.Generator(device=dev).manual_seed(11)
    t = torch.clamp(288.15 - 6.5e-3 * z, min=216.65) + torch.randn(p.shape, device=dev, generator=g, dtype=torch.float64)
    q = 0.015 * torch.exp(-torch.clamp(z, min=0) / 2500) * torch.rand(p.shape, device=dev, generator=g, dtype=torch.float64)
    return t.float(), q.float(), p


def levels_read(torch, zc, targets):
    """(K_field, K_walk) per column of a coordinate zc [NK][nxy] that rises with the walk index (the surface first)"""
    P = torch.sort(torch.as_tensor(targets, device=zc.device, dtype=torch.float64)).values
    nk = zc.shape[0]
    j = torch.ones((P.numel(), zc.shape[1]), dtype=torch.int64, device=zc.device)
    for m in range(1, nk - 1):
        j += (zc[m][None, :] < P[:, None]).to(torch.int64)
    ks = torch.sort(torch.cat([j - 1, j]), dim=0).values
    k_field = 1 + (torch.diff(ks, dim=0) != 0).sum(dim=0)
    return k_field.double(), (j[-1] + 1).double()


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vertical_height_time.py needs a GPU")
    import fimex_b200 as fb
    from bench import peaks
    import vertical_height_oracle as vo

    rng = np.random.default_rng(20261020)
    ap, b = hybrid_table(NK, rng)
    ps = surface_pressure(rng)
    nxy = NX * NY
    dev = torch.device("cuda:0")
    psd1 = torch.from_numpy(ps).to(dev)
    t1, q1, p = column_inputs(torch, ap, b, psd1, dev)
    # the walk's coordinate for the byte count (surface = k = NK - 1: reverse to walk order)
    pw, tv = p.flip(0), (t1.double() * (1 + (M / 0.01801528 - 1) * q1.double())).flip(0)
    zh = torch.empty_like(pw)
    zh[0] = HYPS * tv[0] * torch.log(psd1.double() / pw[0])
    for m in range(1, NK):
        zh[m] = zh[m - 1] + HYPS * 0.5 * (tv[m] + tv[m - 1]) * torch.log(pw[m - 1] / pw[m])
    zstd = torch.empty_like(pw)
    for m in range(NK):  # the standard converter's two lowest layers, enough for FL450 (only the counts are needed)
        zstd[m] = 44330.8 * (1 - (pw[m] / 1013.25) ** 0.190263)
        hi = pw[m] < 226.3206
        zstd[m][hi] = 11000.0 + HYPS * 216.65 * torch.log(226.3206 / pw[m][hi])
    peak, peak_src = peaks()
    info_before = gpu_info()
    g = torch.Generator(device=dev).manual_seed(7)
    field = torch.randn((NT, NK, nxy), device=dev, generator=g) * 30 + 250
    psd = psd1.repeat(NT, 1)
    t = t1.repeat(NT, 1, 1)
    q = q1.repeat(NT, 1, 1)
    result = {"workload": f"{NX}x{NY} x {NT} steps x {NK} levels (synthetic L137-like hybrid table)", "peak_gbs": peak, "peak_source": peak_src,
              "runs": {}}
    lib = fb.load()
    runs = {"hypsometric_15_heights": ("hypsometric", "height", HEIGHTS, zh, 2),
            "standard_flight_levels": ("standard", "altitude", FLIGHT_LEVELS, zstd, 0)}
    for key, (conv, target, levels, zc, n_aux) in runs.items():
        k_field, k_walk = levels_read(torch, zc, levels)
        P = levels.size
        alg_bytes = 4 * nxy * NT * (P + float(k_field.mean()) + n_aux * float(k_walk.mean()) + 1) + 4 * nxy
        hi = fb.HeightInterpolator("atmosphere_hybrid_sigma_pressure_coordinate", {"ap": ap, "b": b}, "linear", levels, type=target, converter=conv)
        out = torch.empty((NT, P, nxy), device=dev)
        cols, keep = hi._columns(NT, nxy, True, psd, t, q, None, None)
        call = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values_columns_device(  # noqa: E731
            hi._h, fb.capi.ptr(field), fb.vertical.C.byref(cols), nxy, NT, fb.capi.ptr(out), fb.cached._stream_ptr(None)))
        for _ in range(2):
            call()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / NT)
        ms = float(np.median(times))
        gbs = alg_bytes / NT / (ms * 1e-3) / 1e9
        result["runs"][key] = {"targets": P, "k_field_mean": float(k_field.mean()), "k_walk_mean": float(k_walk.mean()),
                               "k_walk_max": int(k_walk.max()), "algorithmic_bytes_per_step": alg_bytes / NT, "ms_per_step": ms,
                               "ms_per_step_min": float(min(times)), "values_per_s": nxy * P / (ms * 1e-3), "hbm_gbs": gbs, "roofline_frac": gbs / peak}
        hi.close()
    info_after = gpu_info()

    # host-buffer call (hypsometric heights), pinned host arrays, NT_HOST steps in one call
    hi = fb.HeightInterpolator("atmosphere_hybrid_sigma_pressure_coordinate", {"ap": ap, "b": b}, "linear", HEIGHTS, converter="hypsometric")
    h_field = field[:NT_HOST].cpu().pin_memory()
    h_t, h_q, h_ps = t[:NT_HOST].cpu().pin_memory(), q[:NT_HOST].cpu().pin_memory(), psd[:NT_HOST].cpu().pin_memory()
    h_out = torch.empty((NT_HOST, HEIGHTS.size, nxy), pin_memory=True)
    hcols, hkeep = hi._columns(NT_HOST, nxy, False, h_ps.numpy(), h_t.numpy(), h_q.numpy(), None, None)
    hcall = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values_columns(hi._h, fb.capi.ptr(h_field), fb.vertical.C.byref(hcols), nxy,  # noqa: E731
                                                                               NT_HOST, fb.capi.ptr(h_out)))
    hcall()
    ht = []
    for _ in range(3):
        t0 = time.perf_counter()
        hcall()
        ht.append(time.perf_counter() - t0)
    h_ms = float(np.median(ht)) * 1e3 / NT_HOST
    pcie_bytes = 4 * nxy * (3 * NK + 1 + HEIGHTS.size)
    result["host_call_hypsometric"] = {"steps": NT_HOST, "ms_per_step": h_ms, "values_per_s": nxy * HEIGHTS.size / (h_ms * 1e-3),
                                       "pcie_gbs": pcie_bytes / (h_ms * 1e-3) / 1e9}

    # CPU oracle on all cores, one step, and the check that the GPU's step is bit-identical to it
    t0 = time.perf_counter()
    want = vo.vinterp_height(vo.LIN, vo.HYPSOMETRIC, vo.HEIGHT, vo.VCOORD_HYBRID, ap, b, HEIGHTS, h_field[:1].numpy(), ps=h_ps[:1].numpy(),
                             t=h_t[:1].numpy(), q=h_q[:1].numpy())
    cpu_s = time.perf_counter() - t0
    result["cpu_oracle_hypsometric"] = {"ms_per_step": cpu_s * 1e3, "threads": os.cpu_count(),
                                        "gpu_step_bit_identical": bool(h_out[:1].numpy().tobytes() == want.tobytes())}
    result["gpu"] = {"before": info_before, "after": info_after}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
