"""The vertical interpolator's data conversions at ERA5 size: 1440 x 721 columns, 24 steps x 137 model levels (synthetic L137-like
hybrid table and ps, as vertical_time.py), each of theta2T, omega2vwind and add4Dpressure.  Prints one JSON line (and appends it to
--out).

Per op: ms per step (CUDA events around the device call over all 24 steps, warmed up; each field is 13.7 GB, far larger than L2),
algorithmic bytes 4 * nxy * nt * (2 nk + 1) for theta2T, (3 nk + 1) for omega2vwind and (nk + 1) for the pressure field, and the
fraction of the HBM peak bench.py uses.  Then the host-buffer call (theta2T, pinned host arrays, 4 steps, copies inside the timed
region), and the CPU restatement on all cores for one step, checked bit for bit against the GPU's step.  The card's name and power
limit are read in the same run.

    python profiles/tools/vertical_convert_time.py [--out FILE] [--reps 5]
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

HOST_STEPS = 4


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vertical_convert_time.py needs a GPU")
    import fimex_b200 as fb
    from fimex_b200.vertical import HYBRID, PressureConversion, _Columns
    from bench import peaks
    import vertical_convert_oracle as vc
    import ctypes as C

    rng = np.random.default_rng(20261020)
    ap, b = hybrid_table(NK, rng)
    ps = surface_pressure(rng)
    nxy = NX * NY
    peak, peak_src = peaks()
    info_before = gpu_info()

    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(7)
    field = torch.rand((NT, NK, nxy), device=dev, generator=g) * 1300 + 200
    temp = torch.rand((NT, NK, nxy), device=dev, generator=g) * 140 + 180
    psd = torch.from_numpy(np.tile(ps, (NT, 1))).to(dev)
    out = torch.empty((NT, NK, nxy), device=dev)
    levels = 4 * nxy * NT
    alg = {"theta2T": levels * (2 * NK + 1), "omega2vwind": levels * (3 * NK + 1), "add4Dpressure": levels * (NK + 1)}
    result = {"workload": f"{NX}x{NY} x {NT} steps x {NK} levels (synthetic L137-like hybrid table)", "peak_gbs": peak, "peak_source": peak_src,
              "ops": {}}
    lib = fb.load()
    cols = _Columns()
    cols.ps = fb.capi.ptr(psd).value
    cols.t = fb.capi.ptr(temp).value
    for op in ("theta2T", "omega2vwind", "add4Dpressure"):
        pc = PressureConversion(HYBRID, {"ap": ap, "b": b}, op)
        call = lambda: fb.capi.check(lib.fb200_vconvert_values_device(pc._h, fb.capi.ptr(field), C.byref(cols), nxy, NT,  # noqa: E731
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
        gbs = alg[op] / NT / (ms * 1e-3) / 1e9
        result["ops"][op] = {"ms_per_step": ms, "ms_per_step_min": float(min(times)), "values_per_s": nxy * NK / (ms * 1e-3),
                             "algorithmic_bytes_per_step": alg[op] / NT, "hbm_gbs": gbs, "roofline_frac": gbs / peak}
        pc.close()
    info_after = gpu_info()
    del temp, out

    # host-buffer call (theta2T), pinned host arrays, HOST_STEPS steps in one call
    pc = PressureConversion(HYBRID, {"ap": ap, "b": b}, "theta2T")
    h_field = torch.empty((HOST_STEPS, NK, nxy), pin_memory=True)
    h_field.copy_(field[:HOST_STEPS].cpu())
    h_ps = torch.from_numpy(np.tile(ps, (HOST_STEPS, 1))).pin_memory()
    h_out = torch.empty((HOST_STEPS, NK, nxy), pin_memory=True)
    hcols = _Columns()
    hcols.ps = fb.capi.ptr(h_ps).value
    hcall = lambda: fb.capi.check(lib.fb200_vconvert_values(pc._h, fb.capi.ptr(h_field), C.byref(hcols), nxy, HOST_STEPS,  # noqa: E731
                                                            fb.capi.ptr(h_out)))
    hcall()
    ht = []
    for _ in range(3):
        t0 = time.perf_counter()
        hcall()
        ht.append(time.perf_counter() - t0)
    h_ms = float(np.median(ht)) * 1e3 / HOST_STEPS
    pcie_bytes = 4 * nxy * (2 * NK + 1)
    result["host_call_theta2T"] = {"steps": HOST_STEPS, "ms_per_step": h_ms, "pcie_gbs": pcie_bytes / (h_ms * 1e-3) / 1e9}

    # the CPU restatement on all cores, one step (theta2T), and the check that the GPU's step is bit-identical to it
    f0 = h_field[:1].numpy()
    t0 = time.perf_counter()
    want = vc.vconvert(vc.THETA2T, vc.VCOORD_HYBRID, ap, b, NK, field=f0, ps=ps[None])
    cpu_s = time.perf_counter() - t0
    result["cpu_restatement_theta2T"] = {"ms_per_step": cpu_s * 1e3, "threads": os.cpu_count(),
                                         "gpu_step_bit_identical": bool(h_out[:1].numpy().tobytes() == want.tobytes())}
    result["gpu"] = {"before": info_before, "after": info_after}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
