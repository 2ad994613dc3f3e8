#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config 2 (configs[1]):

    synthetic ERA5-shape 1440x721 x 137 levels x 24 times float32, bilinear to a 2.5 km rotated-pole 2000x2000 grid.

One "step" = one pass of the hot path over the whole (time x level) stack: 24*137 = 3288 levels through
CachedInterpolation::interpolateValues = 1.3152e10 regridded output values.  Inputs and outputs are resident in HBM for
`value`; `e2e` runs the same workload through the C ABI with HOST buffers (pinned), copies inside the timed region, next to
a plain-cudaMemcpyAsync ceiling measured in the same run (`e2e.link_ceiling`, `e2e.frac_of_link`).

N > 1: one process per GPU (torchrun).  Default `--scaling strong`: the ONE stack is split into contiguous slabs of levels,
GPU g owns [g*3288/N, (g+1)*3288/N) (411 levels at N = 8; SURVEY.md 8e, the reference's analogue is the rank-modulo time split
of src/NetCDF_CDMWriter.cc:632-645); `--scaling weak` gives every GPU a whole stack of its own.  There is no data-path
collective: rank 0 computes the index tables on its GPU and NCCL broadcasts the two fp64 position tables (timed, and
compared bit for bit with tables recomputed on every rank: `setup`).  After the timed region every rank checks a sample of
its own output against the CPU oracle (`ranks_verified`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--method bilinear|nearestneighbor|bicubic]
                    [--variant plain|fill|short] [--scaling strong|weak] [--no-extra] [--dump-outputs DIR]

--variant (default plain = CachedInterpolation::interpolateValues, the BASELINE workload) selects the whole slice body of
CDMInterpolator::getDataSlice instead, with its two adapter passes fused into the gather kernel: `fill` = float32 field
with 1 % fill values (9.96921e+36) in, float32 with fill values out; `short` = a packed int16 variable in and out.

At N = 1 the line also carries `extra`: nearest neighbour, bicubic (exact and fp32-tolerance arithmetic), int16 getDataSlice,
fused u/v + rotation, config 4 (bicubic u/v to a 3000 x 3000 polar-stereographic grid) and config 5 (forward mean / max of a
10 M-point swath), a few steps each.

FIMEX_B200_BICUBIC_FP32=1 / FIMEX_B200_BICUBIC_CONTRACT=1 in the environment switch --method bicubic to the opt-in arithmetic
modes (noted in the line).

--impl reference times the reference's own CPU implementation of the path (oracle/_ref: the reference's
interpolation.c compiled unmodified, inside the restated CachedInterpolation loop, OpenMP over all host cores) on a
bounded sample (one time step = 137 levels per step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SRC_PROJ = "+proj=latlong +a=6371000 +e=0 +no_defs"  # the default sphere the reference writes (ProjectionImpl.cc:139-160)
DST_PROJ = "+proj=ob_tran +o_proj=longlat +lon_0=-40 +o_lat_p=22 +R=6.371e+06 +no_defs"  # test/testInterpolator.cc:413
NX, NY, NZ, NT = 1440, 721, 137, 24
OUT_N = 2000
OUT_STEP_DEG = 0.0225  # ~2.5 km on R = 6371 km
METRIC = "regridded output values/sec"
METHODS = {"bilinear": 1, "nearestneighbor": 0, "bicubic": 2}


def axes():
    lon = np.arange(NX) * 0.25
    lat = 90.0 - np.arange(NY) * 0.25
    out = (np.arange(OUT_N) - (OUT_N - 1) / 2.0) * OUT_STEP_DEG
    return lon, lat, out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region"""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                                          str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline
# ----------------------------------------------------------------------------------------------------------------
def cpu_tables(method):
    """index tables with the CPU oracle (projection + points2position + createReducedDomain)"""
    from oracle import oracle as orc
    o = orc.Oracle()
    lon, lat, out = axes()
    rc, x, y = o.project_axes(DST_PROJ, SRC_PROJ, np.radians(out), np.radians(out))
    assert rc == 1
    px = o.points2position(x, np.radians(lon), orc.LONGITUDE)
    py = o.points2position(y, np.radians(lat), orc.LATITUDE)
    red, px, py, inX, inY, x0, y0 = o.reduced_domain(px, py, NX, NY)
    return px, py, inX, inY, x0, y0


def synth_field_np(nlev, inX, inY, x0, y0, t=0, seed=20261018):
    """v = 250 + 30 sin(lat) cos(2 lon) + 0.1 z + t + 0.5 N(0,1) on the cropped footprint (SURVEY.md 8d)"""
    lon, lat, _ = axes()
    lo = np.radians(lon[x0:x0 + inX])[None, None, :]
    la = np.radians(lat[y0:y0 + inY])[None, :, None]
    z = np.arange(nlev, dtype=np.float32)[:, None, None]
    rng = np.random.default_rng(seed + t)
    return (250 + 30 * np.sin(la) * np.cos(2 * lo) + 0.1 * z + t + 0.5 * rng.standard_normal((nlev, inY, inX))).astype(np.float32)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_driver():
    """(driver, kind, threads, description).  torchrun exports OMP_NUM_THREADS=1; the thread count is therefore passed
    explicitly: all the cores this process may run on."""
    from oracle import oracle as orc
    cores = host_cores()
    if orc.Reference.available():
        return orc.Reference(), "reference", cores, "reference src/interpolation.c (gcc -O2 -fopenmp, unmodified) in the restated " \
                                                     "CachedInterpolation.cc:118-147 loop"
    return orc.Oracle(), "port", cores, "oracle/mifi_oracle.c restatement (gcc -O2 -fopenmp)"


def run_cpu(method_id, steps, warmup, nlev=NZ):
    drv, kind, cores, how = cpu_driver()
    px, py, inX, inY, x0, y0 = cpu_tables(method_id)
    field = synth_field_np(nlev, inX, inY, x0, y0)
    out = np.empty(nlev * OUT_N * OUT_N, dtype=np.float32)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        drv.cached_interpolate(method_id, px, py, inX, inY, OUT_N, OUT_N, field, nthreads=cores, out=out)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    values = nlev * OUT_N * OUT_N
    total = sum(times)
    return {"value": values * len(times) / total, "ms_per_step": 1e3 * total / len(times), "cores": int(cores), "kind": kind,
            "sample": f"{nlev} levels (one time step) of the workload per step, {len(times)} steps after {warmup} warm-up; {how}",
            "footprint": [int(inX), int(inY)]}


def bench_config(args, method, inX, inY, x0, y0):
    """the `config` object: the SAME keys and values in both arms (the driver compares them), nothing arm-specific"""
    name = workload_name(method)
    if args.times != NT:
        name += f" [REDUCED to {args.times} time steps: profiling only]"
    return {"workload": name, "levels_total": NZ * args.times, "source_footprint": [int(inX), int(inY)], "crop_offset": [int(x0), int(y0)],
            "variant": args.variant, "parallelism": f"slab{args.gpus}", "scaling": args.scaling,
            "l2": "inputs+outputs >> L2 (52.6 GB written per pass over the stack), no flush needed"}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    method_id = METHODS[args.method]
    r = run_cpu(method_id, max(1, args.steps), max(0, args.warmup))
    px, py, inX, inY, x0, y0 = cpu_tables(method_id)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "values/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, args.method, inX, inY, x0, y0),
        "sample_levels_per_step": NZ,
        "cpu_baseline": {"value": r["value"], "unit": "values/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "values/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


def bind_host_memory_to_gpu_node(local_rank):
    """NUMA placement of this rank's page-locked host buffers: prefer the memory node the GPU hangs off, so that the 8 ranks of
    a node do not push all their downloads through one socket's memory (and the inter-socket link).  Returns a description."""
    try:
        import ctypes
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        if bus is None:
            return "numa: pci bus id unavailable"
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return "numa: node unknown"
        libc = ctypes.CDLL(None, use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        MPOL_PREFERRED, SYS_set_mempolicy = 1, 238  # x86-64
        rc = libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(64))
        return f"numa: host buffers prefer node {node}" if rc == 0 else f"numa: set_mempolicy failed (errno {ctypes.get_errno()})"
    except Exception as e:  # placement is an optimisation, never a requirement
        return f"numa: {type(e).__name__}: {e}"


def workload_name(method):
    return f"ERA5-shape {NX}x{NY}x{NZ}x{NT} float32 -> {OUT_N}x{OUT_N} rotated-pole {OUT_STEP_DEG} deg (~2.5 km), {method}"


KERNEL_SOURCES = {  # the files a measured-traffic entry of profiles/traffic.json is tied to
    "k_gather_bilinear_staged": ("staged_kernels.cu", "interp_math.cuh", "convert.cuh", "tables.cuh"),
    "k_gather_bilinear_staged<NN>": ("staged_kernels.cu", "interp_math.cuh", "convert.cuh", "tables.cuh"),
    "k_gather_bicubic_staged": ("bicubic_staged.cu", "interp_math.cuh", "convert.cuh"),
}


def kernel_source_hash(kernel="k_gather_bilinear_staged"):
    """sha256 (first 16 hex digits) of the sources of one gather kernel: profiles/traffic.json is only quoted for the kernel it
    was measured on"""
    import hashlib
    h = hashlib.sha256()
    for f in KERNEL_SOURCES.get(kernel, ("staged_kernels.cu", "bicubic_staged.cu", "interp_math.cuh", "convert.cuh")):
        with open(os.path.join(ROOT, "fimex_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def time_ms(fn, reps, warm=1):
    """mean device time of fn() over `reps` calls, CUDA events on the current stream, after `warm` untimed calls"""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
def main_b200(args):
    import torch
    import torch.distributed as dist

    import fimex_b200 as fb
    from fimex_b200 import slab

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path in fimex_b200)"
    torch.cuda.set_device(local)
    fb.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    method = args.method
    method_id = METHODS[method]
    lon, lat, out_ax = axes()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_sum(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def build_tables():
        c = fb.CachedInterpolation.fromProjection(method_id, DST_PROJ, out_ax, out_ax, True, True, SRC_PROJ, lon, lat, True)
        c.createReducedDomain()
        torch.cuda.synchronize()
        return c, [c.getInX(), c.getInY(), c.reducedDomain()[2], c.reducedDomain()[3]]

    # ---- index tables.  north_star: rank 0 builds them on its GPU and NCCL broadcasts the two fp64 position tables (64 MB);
    # the alternative -- every rank recomputes them on its own GPU -- is timed next to it and must give identical bits.
    barrier()  # (also the first collective: NCCL communicator set-up stays out of both timings)
    t0 = time.perf_counter()
    ci_own, geom_own = build_tables()
    setup = {"recompute_per_rank_s": all_max(time.perf_counter() - t0)}
    ci, geom = ci_own, geom_own
    if world > 1:
        barrier()
        t0 = time.perf_counter()
        if rank == 0:
            ci0, geom0 = build_tables()
        else:
            ci0, geom0 = None, [0, 0, 0, 0]
        t_build = time.perf_counter() - t0
        ci, geom = slab.broadcast_cached_interpolation(ci0, geom0, method_id, OUT_N, OUT_N, rank, dev)
        torch.cuda.synchronize()
        setup["rank0_build_plus_nccl_broadcast_s"] = all_max(time.perf_counter() - t0)
        setup["rank0_build_s"] = all_max(t_build if rank == 0 else 0.0)
        a, b = ci.device_points(), ci_own.device_points()
        same = float(geom == geom_own and torch.equal(a[0].view(torch.int64), b[0].view(torch.int64)) and
                     torch.equal(a[1].view(torch.int64), b[1].view(torch.int64)))
        t = torch.tensor([same], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        setup["broadcast_tables_identical_to_recomputed"] = bool(t.item() == 1.0)
        ci_own.close()
    inX, inY, x0, y0 = geom

    # ---- this rank's slab of the flattened (time x level) stack ----------------------------------------------------
    total_levels = NZ * args.times
    if args.scaling == "strong":  # ONE stack of 24 x 137 levels; GPU g owns levels [g S/G, (g+1) S/G)  (SURVEY.md 8e)
        z_begin, z_end = slab.slab_range(total_levels, rank, world)
    else:  # weak: every GPU regrids a whole stack of its own
        z_begin, z_end = rank * total_levels, (rank + 1) * total_levels
    nlev = z_end - z_begin
    g = torch.Generator(device=dev).manual_seed(20261018 + rank)
    lo = torch.deg2rad(torch.tensor(lon[x0:x0 + inX], device=dev, dtype=torch.float32))[None, None, :]
    la = torch.deg2rad(torch.tensor(lat[y0:y0 + inY], device=dev, dtype=torch.float32))[None, :, None]
    lev = torch.arange(z_begin, z_end, device=dev)
    zz = (lev % NZ).to(torch.float32)[:, None, None]
    tt = (lev // NZ).to(torch.float32)[:, None, None]
    d_in = 250 + 30 * torch.sin(la) * torch.cos(2 * lo) + 0.1 * zz + tt
    d_in = (d_in + 0.5 * torch.randn((nlev, inY, inX), generator=g, device=dev, dtype=torch.float32)).contiguous()
    values_per_rank = nlev * OUT_N * OUT_N
    values_per_step = (total_levels if args.scaling == "strong" else world * total_levels) * OUT_N * OUT_N  # whole job
    in_elem = out_elem = 4
    fill = None
    if args.variant == "fill":  # SURVEY.md 8d variant B: 1 % undefined values, marked with the NetCDF default fill value
        fill = fb.default_fill_value(np.float32)
        d_in[torch.rand(d_in.shape, generator=g, device=dev) < 0.01] = fill
    elif args.variant == "short":  # a packed variable: scale 0.01, offset 250 -> int16, fill -32767
        fill = -32767.0
        packed = torch.clamp(torch.round((d_in - 250.0) / 0.01), -32000, 32000).to(torch.int16)
        packed[torch.rand(d_in.shape, generator=g, device=dev) < 0.01] = -32767
        d_in = packed.contiguous()
        in_elem = out_elem = 2
    d_out = torch.empty(nlev * OUT_N * OUT_N, device=dev, dtype=d_in.dtype)

    def step():
        if fill is None:
            ci.interpolateValues(d_in, out=d_out)
        else:
            ci.getDataSlice(d_in, fill, out=d_out)

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = fb.kernel_launches()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for k in range(args.steps):
        step()
        ev[k + 1].record()
    barrier()
    launches = fb.kernel_launches() - launches0
    if args.dump_outputs and rank == 0:  # before the e2e and extra legs reuse d_out
        dump_outputs(args.dump_outputs, d_out.view(nlev, -1), torch)
    own_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    clocks = sampler.stop() if rank == 0 else None
    total_ms = all_max(own_ms)
    rank_ms = [own_ms / args.steps]
    if world > 1:
        gathered = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([own_ms / args.steps], device=dev, dtype=torch.float64))
        rank_ms = [float(x.item()) for x in gathered]
    value = values_per_step * args.steps / (total_ms * 1e-3)

    # ---- every rank checks a sample of ITS OWN output against the CPU oracle (the checker, outside the timed region) ----
    verified = 0.0
    try:
        from oracle import oracle as orc
        o = orc.Oracle()
        px, py = ci.points()
        rng = np.random.default_rng(100 + rank)
        idx = rng.integers(0, OUT_N * OUT_N, 1500)
        lv = sorted({0, nlev // 2, nlev - 1})
        sel = torch.tensor(lv, device=dev)
        if fill is None:
            host_in = d_in[sel].cpu().numpy()
            want = o.cached_interpolate(method_id, px[idx], py[idx], inX, inY, idx.size, 1, host_in).reshape(len(lv), -1)
            got = d_out.view(nlev, -1)[sel][:, torch.from_numpy(idx).to(dev)].cpu().numpy()
            if method_id == 2 and (os.environ.get("FIMEX_B200_BICUBIC_FP32", "")[:1] == "1" or os.environ.get("FIMEX_B200_BICUBIC_CONTRACT", "")[:1] == "1"):
                # the opt-in arithmetic modes are not bit-identical: same NaN mask, values within 1e-5 of the field's magnitude
                same = (np.isnan(got) == np.isnan(want)) & (np.isnan(want) | (np.abs(got - want) <= 1e-5 * float(np.nanmax(np.abs(host_in)))))
            else:
                same = (got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))
        else:
            host_in = o.as_float(d_in[sel].cpu().numpy(), fill)
            np_type = {torch.float32: np.float32, torch.int16: np.int16}[d_in.dtype]
            want = o.from_float(o.cached_interpolate(method_id, px[idx], py[idx], inX, inY, idx.size, 1, host_in), fill, np_type).reshape(len(lv), -1)
            got = d_out.view(nlev, -1)[sel][:, torch.from_numpy(idx).to(dev)].cpu().numpy()
            same = got == want
        verified = 1.0 if bool(same.all()) else 0.0
        if not verified:
            sys.stderr.write(f"[bench] rank {rank}: {int((~same).sum())} of {same.size} sampled output values differ from the oracle\n")
    except Exception as e:  # the oracle is test infrastructure: without it the run is reported as unverified, not failed
        sys.stderr.write(f"[bench] rank {rank}: verification skipped ({type(e).__name__}: {e})\n")
    ranks_verified = int(round(all_sum(verified)))

    # ---- roofline of the dominant (only) kernel of the step ------------------------------------------------------
    peak, peak_src = peaks()
    n_out, n_fp = OUT_N * OUT_N, inX * inY
    alg_bytes = out_elem * n_out * nlev + in_elem * n_fp * nlev + 16 * n_out  # SURVEY.md 8d: store + compulsory load + two fp64 positions
    kernel_ms = float(np.mean(per_launch_ms))
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    kernel_name = {0: "k_gather_bilinear_staged<NN>", 1: "k_gather_bilinear_staged", 2: "k_gather_bicubic_staged"}[method_id]
    if method_id == 1 and os.environ.get("FIMEX_B200_BULK_STORE", "0") in ("1", "2") and os.environ.get("FIMEX_B200_BILINEAR_QUAD", "0") != "1":
        kernel_name = "k_gather_bilinear_bulk"  # opt-in experiment
    elif method_id == 1 and os.environ.get("FIMEX_B200_BILINEAR_QUAD", "0") == "1":
        kernel_name = "k_gather_bilinear_staged<QUAD>"  # opt-in experiment
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": peak_src, "kernel": kernel_name,
                "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_output_value": alg_bytes / values_per_rank,
                "kernel_ms": kernel_ms,
                "formula": f"{out_elem}*N_out*Z (store) + {in_elem}*N_fp*Z (compulsory load of the cropped footprint) + 16*N_out (two fp64 positions)",
                "n_out": n_out, "n_fp": n_fp, "levels": nlev}
    if method_id == 2:
        roofline["note"] = bicubic_note()
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and world == 1 and args.times == NT:
        try:  # measured DRAM bytes per launch of the FULL workload (ncu), quoted only for the kernel source it was measured on
            with open(traffic_file) as f:
                tr = json.load(f)
            ent = tr.get(kernel_name)
            if isinstance(ent, dict) and ent.get("source_sha16") == kernel_source_hash(kernel_name) and ent.get("variant", "plain") == args.variant:
                roofline["traffic"] = ent["bytes_per_launch"]
                roofline["traffic_source"] = ent.get("how")
        except Exception:
            pass

    # ---- e2e: the same workload through the C ABI with HOST buffers (pinned); copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        numa = bind_host_memory_to_gpu_node(local) if world > 1 else "numa: single rank, default placement"
        call_lev = min(NZ, nlev)
        ncalls = (nlev + call_lev - 1) // call_lev  # one getDataSlice-sized call (137 levels) per time step, the way a Fimex host calls it
        h_in = torch.empty((call_lev, inY, inX), dtype=d_in.dtype, pin_memory=True)
        h_in.copy_(d_in[:call_lev].cpu())
        h_out = torch.empty(call_lev * OUT_N * OUT_N, dtype=d_in.dtype, pin_memory=True)
        hin_np, hout_np = h_in.numpy(), h_out.numpy()
        e2e_steps = max(1, min(args.steps, args.e2e_steps))

        def host_call(nl):
            if fill is None:
                ci.interpolateValues(hin_np[:nl], out=hout_np)
            else:
                ci.getDataSlice(hin_np[:nl], fill, out=hout_np)

        host_call(call_lev)  # warm-up: scratch pool, page mapping
        # the ceiling under this number: plain cudaMemcpyAsync of the same buffers, one per rank, all ranks at once
        link = {}
        d_tmp = d_out[:h_out.numel()]
        for name, fn in (("d2h", lambda: h_out.copy_(d_tmp, non_blocking=True)), ("h2d", lambda: d_tmp.copy_(h_out, non_blocking=True))):
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            own = 3 * h_out.numel() * h_out.element_size() / (time.perf_counter() - t0) / 1e9
            link[name + "_gbs_sum_over_ranks"] = all_sum(own)
            link[name + "_gbs_min_rank"] = -all_max(-own)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            done = 0
            for _c in range(ncalls):
                nl = min(call_lev, nlev - done)
                host_call(nl)
                done += nl
        barrier()
        dt = all_max(time.perf_counter() - t0)
        d2h_job = out_elem * n_out * (values_per_step // n_out)
        e2e = {"value": values_per_step * e2e_steps / dt, "unit": "values/s", "h2d_bytes_per_step": int(in_elem * n_fp * (values_per_step // n_out)),
               "d2h_bytes_per_step": int(d2h_job), "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps,
               "how": ("fb200_interp_interpolate_values" if fill is None else "fb200_interp_get_data_slice") +
                      f" (C ABI) on pinned host buffers, {ncalls} calls of <= {call_lev} levels per rank and step, H2D + kernel + D2H pipelined "
                      "in 3 streams inside the call; " + numa,
               "d2h_gbs": d2h_job * e2e_steps / dt / 1e9,
               "link_ceiling": dict(link, how="plain pinned cudaMemcpyAsync of one call's output / the same bytes back, 3 copies, every rank at "
                                              "the same time (sum and slowest rank), measured in this run on this box"),
               "frac_of_link": (d2h_job * e2e_steps / dt / 1e9) / link["d2h_gbs_sum_over_ranks"] if link.get("d2h_gbs_sum_over_ranks") else None,
               "checksum": float(hout_np[::100003].astype(np.float64).sum())}
        del h_in, h_out

    # ---- CPU baseline (rank 0, N == 1 only): the reference's kernels on this box's host cores -----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            r = run_cpu(method_id, steps=2, warmup=1)
            cpu = {"value": r["value"], "unit": "values/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        except Exception as e:  # the baseline is reported, never required
            cpu = {"value": None, "unit": "values/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": str(e)}

    # ---- the other BASELINE configs, a few steps each (N == 1): driver-visible numbers beside the headline ---------
    extra = None
    if rank == 0 and world == 1 and not args.no_extra and args.variant == "plain" and args.times == NT:
        try:
            extra = run_extras(fb, torch, dev, d_in, d_out, geom, peak)
        except Exception as e:
            extra = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "values/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if args.variant != "short" else "f32 (int16 in HBM)",
            "data": "synthetic",
            "config": bench_config(args, method, inX, inY, x0, y0),
            "levels_per_gpu": nlev, "level_range_rank0": [int(z_begin), int(z_end)], "ms_per_step_by_rank": rank_ms, "setup": setup,
            "ranks_verified": ranks_verified,
            "hbm_gbs": achieved, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "extra": extra,
        }
        emit(line)  # written straight to the real stdout before the NCCL teardown: a buffered line is lost if that dies
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_LEVELS, DUMP_POINTS, DUMP_SEED = 3, 2_000_000, 20261021


def dump_outputs(path, out, torch):
    """What the last timed step returned, as float32 .npy (int16 outputs convert exactly): `levels.npy` = DUMP_LEVELS whole
    output levels [k][OUT_N][OUT_N] and `sample.npy` = DUMP_POINTS values at seeded positions of the whole [levels][points]
    stack, 56 MB in all.  The positions depend only on the stack's shape, so two builds can be compared value for value."""
    nlev, npts = out.shape
    rng = np.random.default_rng(DUMP_SEED)
    lv = np.sort(rng.choice(nlev, min(DUMP_LEVELS, nlev), replace=False))
    flat = rng.integers(0, nlev * npts, DUMP_POINTS)
    os.makedirs(path, exist_ok=True)
    levels = out[torch.from_numpy(lv).to(out.device)].to(torch.float32).cpu().numpy().reshape(-1, OUT_N, OUT_N)
    sample = out.reshape(-1)[torch.from_numpy(flat).to(out.device)].to(torch.float32).cpu().numpy()
    np.save(os.path.join(path, "levels.npy"), levels)
    np.save(os.path.join(path, "sample.npy"), sample)


def bicubic_note():
    if os.environ.get("FIMEX_B200_BICUBIC_CONTRACT", "")[:1] == "1":
        return ("FIMEX_B200_BICUBIC_CONTRACT=1: fp64 FMA chains with one final rounding (20 fp64 instructions per output), not "
                "bit-identical to the reference, within 1e-5 of the field's magnitude; the default is the exact kernel")
    if os.environ.get("FIMEX_B200_BICUBIC_FP32", "")[:1] == "1":
        return ("FIMEX_B200_BICUBIC_FP32=1: separable weights computed in fp64 as the reference does and rounded to fp32 once per "
                "table, 20 FFMA per output; not bit-identical, within 1e-5 relative (north_star's bar for bicubic); default = exact")
    return ("bit-exact bicubic needs 35 fp64 instructions per output (separately rounded multiplies and adds, as the "
            "reference on x86-64): the fp64 pipe (64 lanes/clk/SM) caps it at about 0.35 of the HBM roofline; see DESIGN.md section 4")


def run_extras(fb, torch, dev, d_in, d_out, geom, peak):
    """NN, bicubic (both arithmetic modes), fused u/v + rotation, int16 getDataSlice (with its own e2e) on the headline geometry;
    config 4 (bicubic u/v to a 3000 x 3000 polar-stereographic grid) and config 5 (forward mean / max of a 10 M-point swath).
    3 timed steps each after one warm-up; roofline fractions with SURVEY.md 8d's byte formulas."""
    lon, lat, out_ax = axes()
    inX, inY, x0, y0 = geom
    nlev = d_in.shape[0]
    n_out, n_fp = OUT_N * OUT_N, inX * inY
    out = {}

    def entry(ms, alg, units, unit="values/s", **kw):
        gbs = alg / (ms * 1e-3) / 1e9
        return dict({"ms": ms, "value": units / (ms * 1e-3), "unit": unit, "algorithmic_bytes": int(alg), "hbm_gbs": gbs, "roofline_frac": gbs / peak}, **kw)

    def with_env(name, val, fn):
        old = os.environ.get(name)
        os.environ[name] = val
        try:
            return fn()
        finally:
            if old is None:
                os.environ.pop(name, None)
            else:
                os.environ[name] = old

    alg_scalar = 4 * n_out * nlev + 4 * n_fp * nlev + 16 * n_out
    # config 3(i): nearest neighbour, whole stack
    ci = fb.CachedInterpolation.fromProjection(0, DST_PROJ, out_ax, out_ax, True, True, SRC_PROJ, lon, lat, True)
    ci.createReducedDomain()
    assert (ci.getInX(), ci.getInY()) == (inX, inY)
    out["nearestneighbor"] = entry(time_ms(lambda: ci.interpolateValues(d_in, out=d_out), 3), alg_scalar, nlev * n_out, levels=nlev)
    ci.close()
    # bicubic on the headline geometry: exact (default) and the fp32 tolerance mode
    ci = fb.CachedInterpolation.fromProjection(2, DST_PROJ, out_ax, out_ax, True, True, SRC_PROJ, lon, lat, True)
    ci.createReducedDomain()
    bx, by = ci.getInX(), ci.getInY()
    d_bic = d_in if (bx, by) == (inX, inY) else torch.randn((nlev, by, bx), device=dev)
    alg_bic = 4 * n_out * nlev + 4 * bx * by * nlev + 16 * n_out
    out["bicubic_exact"] = entry(time_ms(lambda: ci.interpolateValues(d_bic, out=d_out), 3), alg_bic, nlev * n_out, levels=nlev, note="bit-identical to the reference")
    if hasattr(fb, "BICUBIC_FP32_AVAILABLE"):
        out["bicubic_fp32"] = with_env("FIMEX_B200_BICUBIC_FP32", "1", lambda: entry(
            time_ms(lambda: ci.interpolateValues(d_bic, out=d_out), 3), alg_bic, nlev * n_out, levels=nlev,
            note="FIMEX_B200_BICUBIC_FP32=1: <= 1e-5 relative, identical NaN masks"))
    ci.close()
    # int16 in / int16 out through getDataSlice (fill -> NaN, gather, NaN -> fill + round + cast in one kernel), device and host
    ci = fb.CachedInterpolation.fromProjection(1, DST_PROJ, out_ax, out_ax, True, True, SRC_PROJ, lon, lat, True)
    ci.createReducedDomain()
    packed = torch.clamp(torch.round((d_in - 250.0) / 0.01), -32000, 32000).to(torch.int16)
    packed[torch.rand(packed.shape, device=dev) < 0.01] = -32767
    packed = packed.contiguous()
    out16 = d_out.view(torch.int16)[:nlev * n_out]
    ms = time_ms(lambda: ci.getDataSlice(packed, -32767.0, out=out16), 3)
    alg16 = 2 * n_out * nlev + 2 * n_fp * nlev + 16 * n_out
    e16 = entry(ms, alg16, nlev * n_out, levels=nlev)
    h_in = torch.empty((NZ, inY, inX), dtype=torch.int16, pin_memory=True)
    h_in.copy_(packed[:NZ].cpu())
    h_out = torch.empty(NZ * n_out, dtype=torch.int16, pin_memory=True)
    hi, ho = h_in.numpy(), h_out.numpy()
    ci.getDataSlice(hi, -32767.0, out=ho)
    t0 = time.perf_counter()
    for _ in range(6):
        ci.getDataSlice(hi, -32767.0, out=ho)
    dt = (time.perf_counter() - t0) / 6
    e16["e2e"] = {"value": NZ * n_out / dt, "unit": "values/s", "ms_per_call": 1e3 * dt, "levels_per_call": NZ,
                  "how": "fb200_interp_get_data_slice on pinned host int16 buffers, copies inside"}
    out["getDataSlice_int16"] = e16
    del packed, h_in, h_out
    # fused x_wind / y_wind + rotation, bilinear, one time step
    cvr = fb.CachedVectorReprojection.fromProjection(fb.MIFI_VECTOR_KEEP_SIZE, SRC_PROJ, DST_PROJ, out_ax, out_ax, fb.LONGITUDE, fb.LATITUDE)
    u, v = d_in[:NZ], d_in[NZ:2 * NZ] if nlev >= 2 * NZ else d_in[:NZ]
    ms = time_ms(lambda: ci.interpolateVector(u, v, cvr), 3)
    out["bilinear_uv_rotated"] = entry(ms, 8 * n_out * NZ + 8 * n_fp * NZ + 32 * n_out, NZ * n_out, unit="pairs/s", levels=NZ)
    ci.close()
    cvr.close()
    # config 4: bicubic u/v, 137 levels, to polar stereographic 3000 x 3000 with CachedVectorReprojection
    stere = "+proj=stere +lat_0=90 +lon_0=0 +lat_ts=60 +a=6371000 +e=0"
    ax4 = -3748750.0 + 2500.0 * np.arange(3000)
    ci = fb.CachedInterpolation.fromProjection(2, stere, ax4, ax4, False, False, SRC_PROJ, lon, lat, True)
    ci.createReducedDomain()
    cvr = fb.CachedVectorReprojection.fromProjection(fb.MIFI_VECTOR_KEEP_SIZE, SRC_PROJ, stere, ax4, ax4, fb.PROJ_AXIS, fb.PROJ_AXIS)
    cx, cy = ci.getInX(), ci.getInY()
    u = torch.randn((NZ, cy, cx), device=dev) * 10
    v = torch.randn((NZ, cy, cx), device=dev) * 10
    alg4 = 8 * 9_000_000 * NZ + 8 * cx * cy * NZ + 32 * 9_000_000
    out["config4_bicubic_uv_rotated_exact"] = entry(time_ms(lambda: ci.interpolateVector(u, v, cvr), 2), alg4, NZ * 9_000_000, unit="pairs/s", levels=NZ)
    if hasattr(fb, "BICUBIC_FP32_AVAILABLE"):
        out["config4_bicubic_uv_rotated_fp32"] = with_env("FIMEX_B200_BICUBIC_FP32", "1", lambda: entry(
            time_ms(lambda: ci.interpolateVector(u, v, cvr), 2), alg4, NZ * 9_000_000, unit="pairs/s", levels=NZ))
    ci.close()
    cvr.close()
    del u, v
    # config 5: 10 M swath points, forward_mean / forward_max onto the 1 km Lambert grid (one level per call, and 16 levels)
    lcc = "+proj=lcc +lat_0=63 +lon_0=15 +lat_1=63 +lat_2=63 +no_defs +R=6.371e+06"
    wgs = "+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs"
    ny, nx = 5000, 2000
    rng = np.random.default_rng(20261020)
    az = np.arcsin(np.cos(np.radians(98.7)) / np.cos(np.radians(63.0)))
    along = (np.arange(ny) - ny / 2)[:, None] * 1000.0
    across = (np.arange(nx) - nx / 2)[None, :] * 1000.0
    sx = along * np.sin(az) + across * np.cos(az)
    sy = along * np.cos(az) - across * np.sin(az)
    rc, slon, slat = fb.mifi_project_values(lcc, wgs, sx.ravel(), sy.ravel())
    slon = np.degrees(slon) + rng.normal(0, 2e-3, slon.shape)
    slat = np.degrees(slat) + rng.normal(0, 1e-3, slat.shape)
    oxa, oya = -1500e3 + 1000.0 * np.arange(3000), -3000e3 + 1000.0 * np.arange(6000)
    n_in, n_cells = nx * ny, 3000 * 6000
    for name, m in (("forward_mean", 6), ("forward_max", 8)):
        cfi = fb.CachedForwardInterpolation.fromCoordinates(m, lcc, oxa, oya, False, False, slon, slat, nx, ny)
        for z in (1, 16):
            val = 280 + torch.randn((z, ny, nx), device=dev)
            val[torch.rand(val.shape, device=dev) < 0.02] = float("nan")
            o = d_out[:z * n_cells]
            ms = time_ms(lambda: cfi.interpolateValues(val, out=o), 5, warm=2)
            alg = 4 * n_in * z + 4 * n_cells * z + 4 * n_in + 4 * (n_cells + 1)
            out[f"config5_{name}_z{z}"] = entry(ms, alg, n_in * z, unit="input points/s", levels=z)
        cfi.close()
    return out


_REAL_STDOUT = None


def claim_stdout():
    """Keep file descriptor 1 for the ONE JSON line: everything else that writes to stdout from here on (the NCCL version
    banner, library chatter of any rank) goes to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    fd = _REAL_STDOUT if _REAL_STDOUT is not None else 1
    while data:
        data = data[os.write(fd, data):]


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--method", default="bilinear", choices=sorted(METHODS))
    ap.add_argument("--variant", default="plain", choices=["plain", "fill", "short"],
                    help="plain: interpolateValues (BASELINE workload); fill / short: the whole getDataSlice body with fused adapters")
    ap.add_argument("--times", type=int, default=NT, help="time steps per GPU slab (24 = the BASELINE workload; fewer only for profiling)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra block (the other BASELINE configs, N = 1 only)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): ONE stack of 24 x 137 levels split across the GPUs (SURVEY.md 8e); weak: a whole stack per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded float32 sample of rank 0's output of the last timed step "
                                                          "to DIR/levels.npy and DIR/sample.npy (56 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the GPU path (--impl b200)")
    if args.impl == "reference":
        return main_reference(args)
    return main_b200(args)


if __name__ == "__main__":
    sys.exit(main())
