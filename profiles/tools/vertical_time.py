"""Vertical interpolation to pressure levels at ERA5 size: 1440 x 721 columns, 24 steps x 137 model levels -> the 37 ERA5 pressure
levels, per method.  Prints one JSON line (and appends it to --out).

The hybrid table is SYNTHETIC (seeded, monotone, shaped like ECMWF's L137: near-geometric spacing aloft, dense near the ground; the
real table is not in the repository).  ps is one seeded field, the same at every step: about 1013 hPa with lows down to about 500 hPa.
Per method: ms per step (CUDA events around the device call over all 24 steps, warmed up; the inputs, 3.4 GB, are far larger than
L2), values/s, algorithmic bytes 4 * nxy * nt * (P + K_read + 1) with K_read = the distinct input levels a column reads (counted
here on the host from the same ps field), the fraction of the HBM peak bench.py uses, the host-buffer call's end-to-end rate (pinned
host arrays, copies inside the timed region), and the CPU oracle on all cores for one step.

    python profiles/tools/vertical_time.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

NX, NY, NT, NK = 1440, 721, 24, 137
ERA5_LEVELS = np.array([1, 2, 3, 5, 7, 10, 20, 30, 50, 70, 100, 125, 150, 175, 200, 225, 250, 300, 350, 400, 450, 500, 550, 600, 650, 700,
                        750, 775, 800, 825, 850, 875, 900, 925, 950, 975, 1000], dtype=np.float64)


def hybrid_table(nk, rng):
    u = np.cumsum(rng.uniform(0.6, 1.4, nk))
    u = (u - u[0]) / (u[-1] - u[0])
    eta = np.exp(np.log(2e-5) * (1 - u) ** 1.6)
    b = np.clip((eta - 0.2) / 0.8, 0, None)
    return 1013.25 * (eta - b), b


def surface_pressure(rng):
    y, x = np.mgrid[0:NY, 0:NX]
    ps = 1013.0 + rng.normal(0, 8, (NY, NX))
    for _ in range(40):  # "mountains": lows down to about 500 hPa
        cx, cy, r, depth = rng.uniform(0, NX), rng.uniform(0, NY), rng.uniform(5, 60), rng.uniform(100, 510)
        ps -= depth * np.exp(-((x - cx) ** 2 + (y - cy) ** 2) / (2 * r * r))
    return np.maximum(ps, 480.0).astype(np.float32).ravel()


def levels_read(ap, b, ps):
    """distinct input levels per column (the kernel reads levels k and k + 1 of every bracket, extrapolation on)"""
    psd = ps.astype(np.float64)
    P = np.sort(ERA5_LEVELS)[:, None]
    j = np.ones((P.size, psd.size), dtype=np.int16)
    for k in range(1, ap.size - 1):
        j += (ap[k] + b[k] * psd)[None, :] < P  # p_k increases with k here
    ks = np.sort(np.concatenate([j - 1, j]), axis=0)
    return 1 + (np.diff(ks, axis=0) != 0).sum(axis=0)


def gpu_info():
    q = "name,clocks.sm,clocks.max.sm,power.limit"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, sm, smax, pl = [s.strip() for s in out.split(",")]
        return {"name": name, "sm_mhz": float(sm), "sm_max_mhz": float(smax), "power_limit_w": float(pl)}
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vertical_time.py needs a GPU")
    import fimex_b200 as fb
    from bench import peaks
    import vertical_oracle as vo

    rng = np.random.default_rng(20261020)
    ap, b = hybrid_table(NK, rng)
    ps = surface_pressure(rng)
    nxy = NX * NY
    kread = levels_read(ap, b, ps)
    P = ERA5_LEVELS.size
    alg_bytes = 4 * nxy * NT * (P + float(kread.mean()) + 1)
    peak, peak_src = peaks()
    info_before = gpu_info()

    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(7)
    field = torch.randn((NT, NK, nxy), device=dev, generator=g) * 30 + 250
    psd = torch.from_numpy(np.tile(ps, (NT, 1))).to(dev)
    out = torch.empty((NT, P, nxy), device=dev)
    result = {"workload": f"{NX}x{NY} x {NT} steps x {NK} levels (synthetic L137-like hybrid table) -> {P} ERA5 pressure levels",
              "k_read_mean": float(kread.mean()), "k_read_max": int(kread.max()), "algorithmic_bytes_per_step": alg_bytes / NT,
              "peak_gbs": peak, "peak_source": peak_src, "methods": {}}
    lib = fb.load()
    for method in ("linear", "log", "loglog", "nearestneighbor"):
        vi = fb.VerticalInterpolator("atmosphere_hybrid_sigma_pressure_coordinate", {"ap": ap, "b": b}, method, ERA5_LEVELS)
        call = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values_device(vi._h, fb.capi.ptr(field), fb.capi.ptr(psd), nxy, NT,  # noqa: E731
                                                                                  fb.capi.ptr(out), fb.cached._stream_ptr(None)))
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
        result["methods"][method] = {"ms_per_step": ms, "ms_per_step_min": float(min(times)), "values_per_s": nxy * P / (ms * 1e-3),
                                     "hbm_gbs": gbs, "roofline_frac": gbs / peak}
        vi.close()
    info_after = gpu_info()

    # host-buffer call (log), pinned host arrays, all 24 steps in one call
    vi = fb.VerticalInterpolator("atmosphere_hybrid_sigma_pressure_coordinate", {"ap": ap, "b": b}, "log", ERA5_LEVELS)
    h_field = torch.empty((NT, NK, nxy), pin_memory=True)
    h_field.copy_(field.cpu())
    h_ps = torch.from_numpy(np.tile(ps, (NT, 1))).pin_memory()
    h_out = torch.empty((NT, P, nxy), pin_memory=True)
    hcall = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values(vi._h, fb.capi.ptr(h_field), fb.capi.ptr(h_ps), nxy, NT,  # noqa: E731
                                                                       fb.capi.ptr(h_out)))
    hcall()
    ht = []
    for _ in range(3):
        t0 = time.perf_counter()
        hcall()
        ht.append(time.perf_counter() - t0)
    h_ms = float(np.median(ht)) * 1e3 / NT
    pcie_bytes = 4 * nxy * (NK + 1 + P)
    result["host_call_log"] = {"ms_per_step": h_ms, "values_per_s": nxy * P / (h_ms * 1e-3), "pcie_gbs": pcie_bytes / (h_ms * 1e-3) / 1e9}

    # CPU oracle on all cores, one step (log), and the check that the GPU's step is bit-identical to it
    f0 = h_field[:1].numpy()
    t0 = time.perf_counter()
    want = vo.vinterp(vo.LOG, vo.VCOORD_HYBRID, ap, b, ERA5_LEVELS, f0, ps=ps[None])
    cpu_s = time.perf_counter() - t0
    result["cpu_oracle_log"] = {"ms_per_step": cpu_s * 1e3, "threads": os.cpu_count(), "gpu_step_bit_identical": bool(h_out[:1].numpy().tobytes() == want.tobytes())}
    result["gpu"] = {"before": info_before, "after": info_after}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
