"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm's JSON line (driver keys, the
`config` object both arms share), the slab split, the --dump-outputs sample, and the bookkeeping of profiles/traffic.json."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_reference_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout  # ONE JSON line on stdout, everything else on stderr
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "values/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "values/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the config object is what both arms print: the same function builds it, nothing arm-specific inside
    class A:
        times, variant, gpus, scaling = bench.NT, "plain", 1, "strong"
    fp = d["config"]["source_footprint"]
    assert d["config"] == bench.bench_config(A, "bilinear", fp[0], fp[1], *d["config"]["crop_offset"])
    assert d["config"]["workload"].startswith("ERA5-shape 1440x721x137x24 float32 -> 2000x2000 rotated-pole") and d["config"]["levels_total"] == 3288
    assert fp == [1440, 202]  # the cropped footprint the byte formula uses


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_strong_scaling_slabs_cover_the_stack_once():
    from fimex_b200.slab import slab_range
    total = bench.NZ * bench.NT
    for world in (1, 2, 4, 8):
        parts = [slab_range(total, r, world) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == total
        assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
    assert slab_range(total, 0, 8) == (0, 411)


def test_dump_outputs_is_a_fixed_float32_sample_of_the_output(tmp_path):
    import numpy as np
    import torch
    nlev, npts = 4, bench.OUT_N * bench.OUT_N
    out = torch.arange(nlev * npts, dtype=torch.float32).view(nlev, npts)  # every value names its own position (< 2**24)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out, torch)
    assert sorted(os.listdir(tmp_path / "a")) == ["levels.npy", "sample.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in ("levels.npy", "sample.npy")) <= 64 << 20
    levels, sample = np.load(tmp_path / "a" / "levels.npy"), np.load(tmp_path / "a" / "sample.npy")
    assert np.array_equal(levels, np.load(tmp_path / "b" / "levels.npy")) and np.array_equal(sample, np.load(tmp_path / "b" / "sample.npy"))
    assert levels.dtype == sample.dtype == np.float32
    assert levels.shape == (bench.DUMP_LEVELS, bench.OUT_N, bench.OUT_N) and sample.shape == (bench.DUMP_POINTS,)
    first = levels[:, 0, 0]
    assert np.all(first % npts == 0) and np.all(np.diff(first) > 0)  # whole levels, in order
    assert all(np.array_equal(levels[i].ravel(), first[i] + np.arange(npts, dtype=np.float32)) for i in range(bench.DUMP_LEVELS))
    assert sample.min() >= 0 and sample.max() < nlev * npts and np.unique(sample).size > 0.9 * sample.size


def test_traffic_json_names_the_sources_it_was_measured_on():
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
        tr = json.load(f)
    for kernel, ent in tr.items():
        assert kernel in bench.KERNEL_SOURCES, kernel
        assert len(ent["source_sha16"]) == 16 and ent["bytes_per_launch"] == ent["dram_bytes_read"] + ent["dram_bytes_write"]
        assert ent["source_files"] == list(bench.KERNEL_SOURCES[kernel])
        # algorithmic bytes of the full workload: 4 N_out Z + 4 N_fp Z + 16 N_out; measured traffic within 5 % of it
        alg = 4 * 4_000_000 * 3288 + 4 * 1440 * 202 * 3288 + 16 * 4_000_000
        assert 0.9 < ent["bytes_per_launch"] / alg < 1.05
