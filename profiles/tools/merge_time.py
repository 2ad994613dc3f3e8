"""The merger at regional-model size: an equidistant 0.025 degree inner grid of 1200 x 1000 inside a 0.1 degree outer grid of 700 x 500,
merged on the inner grid extended over the outer one (setTargetGridFromInner: 2800 x 2000), bilinear, LINEAR(5,2), 64 levels; float32
-> float32 and int16 -> int16 (with a fill value).  Prints one JSON line (and appends it to --out).

Per type:
  * the device call (fb200_merge_get_data_slice_device) timed with CUDA events over --reps warmed repetitions, every stack larger
    than L2;
  * each stage's device time, from the kernel records of one torch.profiler run of a further call (crop, the three gathers, the
    smoothing, the overlay), in a pass of its own;
  * the bytes the chain moves -- each stage reading its inputs and writing its output once -- and the minimum any merge moves (inner
    and outer read once, the merged slice written once), each over the call time and as a fraction of the device-to-device copy
    bandwidth measured in the same run;
  * float32 only: the host-buffer call (pageable numpy arrays) against the chain this library ran before it had the merge call,
    rebuilt here: three Interpolator.getDataSlice calls on float64 copies, the numpy blend and np.where; outputs compared.
The card's name and power limit are read in the same run.

    python profiles/tools/merge_time.py [--out FILE] [--reps 5] [--levels 64]
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vertical_time import gpu_info  # noqa: E402

PROJ = "+proj=latlong +a=6371000 +e=0 +no_defs"
X_OUTER, Y_OUTER = -40.0 + 0.1 * np.arange(700), 70.0 - 0.1 * np.arange(500)
X_INNER, Y_INNER = -20.0 + 0.025 * np.arange(1200), 60.0 - 0.025 * np.arange(1000)
STAGES = {"k_crop_as_float": "crop", "k_border_smooth_linear": "smooth", "k_merge_overlay": "overlay"}


def stage_of(name):
    for k, v in STAGES.items():
        if k in name:
            return v
    return "gathers_and_other"


def old_chain(m, vi, vo):
    """the slice path before the merge call: three gathers on float64 host arrays, blend and overlay in numpy"""
    import fimex_b200 as fb
    nan = float("nan")
    vi, vo = np.asarray(vi, dtype=np.float64), np.asarray(vo, dtype=np.float64)
    on_inner = m._outer_to_inner.getDataSlice(vo, bad_value=nan)
    smooth = fb.linear_border_smoothing(vi, on_inner, m.transitionWidth, m.borderWidth, m.useOuterIfInnerUndefined)
    top = m._inner_to_target.getDataSlice(smooth, bad_value=nan)
    base = m._outer_to_target.getDataSlice(vo, bad_value=nan)
    return np.where(np.isnan(top), base, top)


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    ap_.add_argument("--levels", type=int, default=64)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("merge_time.py needs a GPU")
    import fimex_b200 as fb
    from fimex_b200.cached import _stream_ptr

    info_before = gpu_info()
    nz = args.levels
    dev = torch.device("cuda:0")
    m = fb.Merger(PROJ, X_INNER, Y_INNER, PROJ, X_OUTER, Y_OUTER, True)
    m.setTargetGridFromInner()
    mh = m._merge_handle()
    hs = {"outer_to_inner": m._outer_to_inner.cachedInterpolation, "inner_to_target": m._inner_to_target.cachedInterpolation,
          "outer_to_target": m._outer_to_target.cachedInterpolation}
    I, O = X_INNER.size * Y_INNER.size, X_OUTER.size * Y_OUTER.size
    T = hs["inner_to_target"].getOutX() * hs["inner_to_target"].getOutY()
    win = {k: h.getInX() * h.getInY() for k, h in hs.items()}
    lib = fb.load()
    g = torch.Generator(device=dev).manual_seed(3)

    # device-to-device copy bandwidth of this card, same run: 4 GB read + 4 GB written per copy
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    for _ in range(2):
        b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 5 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()

    result = {"workload": f"inner {X_INNER.size}x{Y_INNER.size} at 0.025 deg in outer {X_OUTER.size}x{Y_OUTER.size} at 0.1 deg -> target "
                          f"{hs['inner_to_target'].getOutX()}x{hs['inner_to_target'].getOutY()} (setTargetGridFromInner), bilinear, "
                          f"LINEAR({m.transitionWidth},{m.borderWidth}), {nz} levels",
              "windows": win, "copy_gbs_measured": copy_gbs, "types": {}}

    def timed(call, reps):
        for _ in range(2):
            call()
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            call()
            s1.record()
            torch.cuda.synchronize()
            times.append(s0.elapsed_time(s1))
        return float(np.median(times)), float(min(times))

    for name, dtype, fill in (("float32", torch.float32, float("nan")), ("int16", torch.int16, -32767.0)):
        base_i = torch.rand((nz, Y_INNER.size, X_INNER.size), device=dev, generator=g) * 30 + 270
        base_o = torch.rand((nz, Y_OUTER.size, X_OUTER.size), device=dev, generator=g) * 30 + 270
        if dtype == torch.float32:
            inner, outer = base_i, base_o
        else:
            inner, outer = torch.round((base_i - 273.15) * 100).to(dtype), torch.round((base_o - 273.15) * 100).to(dtype)
            inner[:, ::97, ::89] = -32767
            outer[:, ::13, ::11] = -32767
        del base_i, base_o
        code = int(fb.cdm_type(dtype))
        sz = inner.element_size()
        out = torch.empty((nz, hs["inner_to_target"].getOutY(), hs["inner_to_target"].getOutX()), dtype=dtype, device=dev)
        st = _stream_ptr(None)

        def call():
            fb.capi.check(lib.fb200_merge_get_data_slice_device(mh._h, code, fb.capi.ptr(inner), inner.numel(), fill, fb.capi.ptr(outer),
                                                                outer.numel(), fill, code, fill, fb.capi.ptr(out), None, st))

        ms, ms_min = timed(call, args.reps)
        # one profiled call, in a pass of its own: device time per stage from the kernel records
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        stage_us = {}
        for ev in prof.key_averages():  # kernels carry their own device time; runtime calls have none of their own
            us = float(ev.self_device_time_total)
            if us > 0:
                k = stage_of(ev.key)
                stage_us[k] = stage_us.get(k, 0.0) + us
        chain = (win["outer_to_inner"] * (sz + 4)      # crop + convert for the outer -> inner gather
                 + win["outer_to_inner"] * 4 + I * 4   # outer -> inner gather
                 + win["inner_to_target"] * (sz + 4 + 4)  # smoothing: inner + outer on the inner grid in, smoothed window out
                 + win["inner_to_target"] * 4 + T * 4  # inner -> target gather
                 + win["outer_to_target"] * (sz + 4)   # crop + convert for the outer -> target gather
                 + win["outer_to_target"] * 4 + T * 4  # outer -> target gather
                 + T * (4 + 4 + sz)) * nz              # overlay
        minimum = (I * sz + O * sz + T * sz) * nz
        entry = {"device_call": {"ms": ms, "ms_min": ms_min, "stage_device_ms_profiled": {k: v / 1e3 for k, v in stage_us.items()},
                                 "chain_bytes": chain, "chain_gbs": chain / (ms * 1e-3) / 1e9,
                                 "chain_frac_of_copy_bw": chain / (ms * 1e-3) / 1e9 / copy_gbs,
                                 "minimum_bytes": minimum, "minimum_gbs": minimum / (ms * 1e-3) / 1e9,
                                 "minimum_frac_of_copy_bw": minimum / (ms * 1e-3) / 1e9 / copy_gbs}}
        if dtype == torch.float32:
            hi, ho = inner.cpu().numpy(), outer.cpu().numpy()
            host = m.getDataSlice(hi, ho)  # warm-up (and the pinned staging cache)
            times = []
            for _ in range(3):
                t0 = time.perf_counter()
                host = m.getDataSlice(hi, ho)
                times.append((time.perf_counter() - t0) * 1e3)
            old_times = []
            for _ in range(2):
                t0 = time.perf_counter()
                old = old_chain(m, hi, ho)
                old_times.append((time.perf_counter() - t0) * 1e3)
            same = bool(np.array_equal(np.isnan(host), np.isnan(old)) and
                        np.array_equal(host[~np.isnan(host)].view(np.uint32), old.astype(np.float32)[~np.isnan(old)].view(np.uint32)))
            entry["host_call"] = {"ms": float(np.median(times)), "ms_min": float(min(times)), "pcie_bytes": int(hi.nbytes + ho.nbytes + host.nbytes)}
            entry["pre_change_host_chain"] = {"ms": float(np.median(old_times)), "ms_min": float(min(old_times)),
                                              "pcie_bytes": int(ho.nbytes * 2 * 2 + I * nz * 8 * 2 + T * nz * 8 * 2)}
            entry["host_speedup"] = entry["pre_change_host_chain"]["ms"] / entry["host_call"]["ms"]
            entry["host_outputs_identical"] = same
            del hi, ho, host, old
        device_out = out.cpu().numpy()
        entry["device_output_defined_share"] = float(np.mean(~np.isnan(device_out))) if dtype == torch.float32 else \
            float(np.mean(device_out != -32767))
        result["types"][name] = entry
        del inner, outer, out
        torch.cuda.empty_cache()
    result["gpu"] = {"before": info_before, "after": gpu_info()}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
