"""Vertical interpolation to depth levels at the size of a coastal ocean forecast: 2600 x 900 columns (about 30 % land), 24 steps x 35
ocean_s_coordinate_g2 levels -> 16 depths (0, 3, 10, ... 3000 m).  Prints one JSON line (and appends it to --out).

The ocean is SYNTHETIC and seeded (tests/vertical_depth_oracle.py, synthetic_ocean): a smooth relief whose lowest 30 % is land (h = 0,
eta NaN), the sea floor from 5 to 3000 m, a sea surface height of up to about 1.5 m; the levels are ROMS's Vstretching = 4 (theta_s = 7,
theta_b = 2) with depth_c = 250 m.  h and eta are the same at every step, the field differs.  Reported: ms per step (CUDA events around
the device call over all 24 steps, warmed up; the field, 7.9 GB, is far larger than L2), values/s, algorithmic bytes
4 * (nxy * nt * P + n_sea * nt * (K_field + 1) + nxy), K_field = the distinct field levels a sea column reads (its brackets), the 1 its
eta, counted here from the same inputs; land columns read nothing but h and write P NaN.  The fraction of the HBM peak bench.py uses;
the host-buffer call's end-to-end rate, timed once after a warm-up (pinned host arrays, 4 steps, copies inside the timed region), and
the CPU oracle on all cores for one step, checked bit for bit against the GPU.

    python profiles/tools/vertical_depth_time.py [--out FILE] [--reps 5]
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

from vertical_height_time import levels_read  # noqa: E402
from vertical_time import gpu_info  # noqa: E402

NX, NY, NT, NK = 2600, 900, 24, 35
DEPTH_C = 250.0
NT_HOST = 4


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vertical_depth_time.py needs a GPU")
    import fimex_b200 as fb
    from bench import peaks
    import vertical_depth_oracle as vo

    rng = np.random.default_rng(20261020)
    s, Cs = vo.roms_stretching(NK)
    h, eta = vo.synthetic_ocean(NX, NY, rng)
    levels = vo.DEPTHS16
    P = levels.size
    nxy = NX * NY
    dev = torch.device("cuda:0")
    d_h1, d_eta1 = torch.from_numpy(h).to(dev), torch.from_numpy(eta).to(dev)
    # the walk's coordinate x = -z of the sea columns for the byte count (the sea floor is k = 0: reverse to walk order)
    sea = d_h1 > 0
    hs, es = d_h1[sea].double(), d_eta1[sea].double()
    S = (DEPTH_C * torch.from_numpy(s).to(dev)[:, None] + hs[None, :] * torch.from_numpy(Cs).to(dev)[:, None]) / (DEPTH_C + hs[None, :])
    xw = -(es[None, :] + (es + hs)[None, :] * S).flip(0)
    k_field, _ = levels_read(torch, xw, levels)
    n_sea = int(sea.sum())
    alg_bytes = 4 * (nxy * NT * P + n_sea * NT * (float(k_field.mean()) + 1) + nxy)
    del S, xw

    peak, peak_src = peaks()
    info_before = gpu_info()
    g = torch.Generator(device=dev).manual_seed(7)
    field = torch.randn((NT, NK, nxy), device=dev, generator=g) * 5 + 10
    d_eta = d_eta1.repeat(NT, 1)
    di = fb.DepthInterpolator("ocean_s_coordinate_g2", {"s": s, "C": Cs, "depth_c": DEPTH_C}, "linear", levels)
    out = torch.empty((NT, P, nxy), device=dev)
    lib = fb.load()
    cols, keep = di._columns(NT, nxy, True, d_eta, d_h1)
    call = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values_columns_device(  # noqa: E731
        di._h, fb.capi.ptr(field), fb.vertical.C.byref(cols), nxy, NT, fb.capi.ptr(out), fb.cached._stream_ptr(None)))
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
    info_after = gpu_info()
    result = {"workload": f"{NX}x{NY} x {NT} steps x {NK} ocean_s_coordinate_g2 levels (synthetic ROMS-like, Vstretching 4, depth_c {DEPTH_C} m)"
                          f" -> {P} depths", "peak_gbs": peak, "peak_source": peak_src,
              "land_share": 1 - n_sea / nxy, "targets": P, "k_field_mean_sea": float(k_field.mean()), "k_field_max": int(k_field.max()),
              "algorithmic_bytes_per_step": alg_bytes / NT, "ms_per_step": ms, "ms_per_step_min": float(min(times)),
              "values_per_s": nxy * P / (ms * 1e-3), "hbm_gbs": gbs, "roofline_frac": gbs / peak}

    # host-buffer call, pinned host arrays, NT_HOST steps in one call: one warm-up, one timed call
    h_field = field[:NT_HOST].cpu().pin_memory()
    h_eta = d_eta[:NT_HOST].cpu().pin_memory()
    h_h = d_h1.cpu().pin_memory()
    h_out = torch.empty((NT_HOST, P, nxy), pin_memory=True)
    hcols, hkeep = di._columns(NT_HOST, nxy, False, h_eta.numpy(), h_h.numpy())
    hcall = lambda: fb.capi.check(lib.fb200_vinterp_interpolate_values_columns(di._h, fb.capi.ptr(h_field), fb.vertical.C.byref(hcols), nxy,  # noqa: E731
                                                                               NT_HOST, fb.capi.ptr(h_out)))
    hcall()
    t0 = time.perf_counter()
    hcall()
    h_ms = (time.perf_counter() - t0) * 1e3 / NT_HOST
    pcie_bytes = 4 * nxy * (NK + 1 + P) + 4 * nxy / NT_HOST
    result["host_call"] = {"steps": NT_HOST, "ms_per_step": h_ms, "values_per_s": nxy * P / (h_ms * 1e-3), "pcie_gbs": pcie_bytes / (h_ms * 1e-3) / 1e9}

    # CPU oracle on all cores, one step, and the check that the GPU's step is bit-identical to it
    t0 = time.perf_counter()
    want = vo.vinterp_depth(vo.LIN, vo.OCEAN_S_G2, s, Cs, levels, h_field[:1].numpy(), eta=h_eta[:1].numpy(), depth=h, depth_c=DEPTH_C)
    cpu_s = time.perf_counter() - t0
    result["cpu_oracle"] = {"ms_per_step": cpu_s * 1e3, "threads": os.cpu_count(),
                            "gpu_step_bit_identical": bool(h_out[:1].numpy().tobytes() == want.tobytes())}
    result["gpu"] = {"before": info_before, "after": info_after}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
