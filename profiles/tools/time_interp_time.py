"""Time interpolation at ERA5 size: 1440 x 721 x 137 values per step, 8 three-hourly source steps (0, 3, ..., 21 h) to 22 hourly targets
(0, 1, ..., 21 h), float32 -> float32 and int16 -> int16 (with a fill value).  Prints one JSON line (and appends it to --out).

Per type: the stack kernel (fb200_tinterp_get_data_slice_device, one launch for all 22 targets) and the step-by-step alternative (22
calls of fb200_tinterp_get_step_device, each reading both source steps of its target), both timed with CUDA events over --reps warmed
repetitions; every stack is far larger than L2.  Algorithmic bytes: n (T_read sizeof(IN) + J sizeof(OUT)) for the stack, with T_read
the distinct source steps the targets need, and J n (2 sizeof(IN) + sizeof(OUT)) step by step; each over its time, and as a fraction
of the HBM figure bench.py uses.  The two outputs are compared bit for bit.  The card's name and power limit are read in the same run.

    python profiles/tools/time_interp_time.py [--out FILE] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vertical_time import gpu_info  # noqa: E402

NX, NY, NK = 1440, 721, 137
SOURCE_HOURS = np.arange(0.0, 24.0, 3.0)
TARGET_HOURS = np.arange(0.0, 22.0, 1.0)


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--reps", type=int, default=5)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_interp_time.py needs a GPU")
    import fimex_b200 as fb
    from bench import peaks
    from fimex_b200.cached import _stream_ptr

    peak, peak_src = peaks()
    info_before = gpu_info()
    n = NX * NY * NK
    T, J = SOURCE_HOURS.size, TARGET_HOURS.size
    ti = fb.TimeInterpolator(SOURCE_HOURS, "hours since 2000-01-01 00:00:00", new_times=TARGET_HOURS)
    steps = [ti.source_steps(j) for j in range(J)]
    t_read = len({k for ia, ib, _ in steps for k in (ia, ib)})
    lib = fb.load()
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(11)
    result = {"workload": f"{NX}x{NY}x{NK} values per step, {T} three-hourly source steps -> {J} hourly targets", "peak_gbs": peak,
              "peak_source": peak_src, "source_steps_read": t_read, "types": {}}

    def timed(call):
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
            times.append(e0.elapsed_time(e1))
        return float(np.median(times)), float(min(times))

    for name, dtype, fill in (("float32", torch.float32, float("nan")), ("int16", torch.int16, -32767.0)):
        if dtype == torch.float32:
            stack = torch.rand((T, n), device=dev, generator=g) * 100 + 200
        else:
            stack = torch.randint(-30000, 30000, (T, n), device=dev, generator=g, dtype=torch.int16)
            stack[:, ::101] = -32767
        code = int(fb.cdm_type(dtype))
        size = stack.element_size()
        out = torch.empty((J, n), dtype=dtype, device=dev)
        out_steps = torch.empty((J, n), dtype=dtype, device=dev)
        st = _stream_ptr(None)

        def stack_call():
            fb.capi.check(lib.fb200_tinterp_get_data_slice_device(ti._h, code, fb.capi.ptr(stack), n, fill, code, fb.capi.ptr(out), st))

        def step_calls():
            for j, (ia, ib, _) in enumerate(steps):
                fb.capi.check(lib.fb200_tinterp_get_step_device(ti._h, j, code, fb.capi.ptr(stack[ia]), fb.capi.ptr(stack[ib]), n, fill, code,
                                                                fb.capi.ptr(out_steps[j]), st))

        ms, ms_min = timed(stack_call)
        ms_s, ms_s_min = timed(step_calls)
        bytes_stack = n * (t_read * size + J * size)
        bytes_steps = J * n * (3 * size)
        gbs, gbs_s = bytes_stack / (ms * 1e-3) / 1e9, bytes_steps / (ms_s * 1e-3) / 1e9
        result["types"][name] = {
            "stack": {"ms": ms, "ms_min": ms_min, "algorithmic_bytes": bytes_stack, "gbs": gbs, "roofline_frac": gbs / peak},
            "step_by_step": {"ms": ms_s, "ms_min": ms_s_min, "algorithmic_bytes": bytes_steps, "gbs": gbs_s, "roofline_frac": gbs_s / peak},
            "stack_speedup": ms_s / ms,
            "outputs_bit_identical": bool(torch.equal(out.view(torch.int16 if size == 2 else torch.int32),
                                                      out_steps.view(torch.int16 if size == 2 else torch.int32))),
        }
        del stack, out, out_steps
        torch.cuda.empty_cache()
    result["gpu"] = {"before": info_before, "after": gpu_info()}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
