"""Build libfimex_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m fimex_b200.build [--force]

The library is written to fimex_b200/lib/libfimex_b200.so (git-ignored; it travels to the GPU box with the
gpurun snapshot).  Flags: -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 (B200 only; no other
architecture is built).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libfimex_b200.so")

SOURCES = ["api.cu", "setup_kernels.cu", "gather_kernels.cu", "forward_kernels.cu", "coordnn_kernels.cu", "adapter_kernels.cu", "staged_kernels.cu", "bicubic_staged.cu", "fill_kernels.cu",
           "vertical_kernels.cu", "time_kernels.cu", "merge_kernels.cu", "proj_parse.cpp"]
HEADERS = ["common.cuh", "proj.cuh", "kernels.h", "tables.cuh", "interp_math.cuh", "convert.cuh", os.path.join("..", "..", "include", "fimex_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function", "-Xptxas", "-v", "--threads", "4",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _host_cxx() -> list:
    # the image exports CXX=/opt/gcc/bin/g++ (a wrapper); the distribution g++ is what nvcc 12.9 is validated with
    if os.path.exists("/usr/bin/g++"):
        return ["-ccbin", "/usr/bin/g++"]
    return []


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS] + [__file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra_flags=None, lib_out: str = None, objdir_name: str = "obj") -> str:
    """extra_flags / out / objdir_name: experiment builds (-DFB_... macros) next to the shipped library, e.g.
    build(force=True, extra_flags=["-DFB_BLQ_CTAS=2"], lib_out=".../libfimex_b200_ctas2.so", objdir_name="obj_ctas2"); load one with
    FIMEX_B200_LIB=<path> in the environment"""
    if not force and not needs_build() and lib_out is None:
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    objdir = os.path.join(LIBDIR, objdir_name)
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    for s in SOURCES:
        o = os.path.join(objdir, os.path.splitext(s)[0] + ".o")
        objs.append(o)
        cmd = [nvcc] + _host_cxx() + NVCC_FLAGS + list(extra_flags or []) + ["-x", "cu", "-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {s}\n{out}")
        failed = failed or p.returncode != 0
    with open(os.path.join(LIBDIR, "build.log" if lib_out is None else os.path.basename(lib_out) + ".log"), "w") as f:
        f.write("\n".join(log))
    if failed:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("nvcc failed; see fimex_b200/lib/build.log")
    link = [nvcc] + _host_cxx() + ["-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_out or LIB] + objs + ["-Xlinker", "-Bsymbolic"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    if verbose:
        print("\n".join(log))
    return lib_out or LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
