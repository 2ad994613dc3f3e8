"""The C++ side of the boundary: include/fimex_b200/Cached.h (mirror of the reference's Cached* classes) and the
mifi_* drop-in symbols, exercised by tests/cpp/testInterpolation_b200.cc -- the reference's own
test/testInterpolation.cc cases restated.  Compiling and linking against libfimex_b200.so is a CPU test; running
needs a GPU."""
import os
import subprocess
import tempfile

import pytest

from fimex_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "testInterpolation_b200.cc")
# built outside the repository tree, which may be read-only where the suite runs
EXE = os.path.join(tempfile.gettempdir(), f"fimex_b200_testInterpolation_b200_{os.getuid()}_{os.getpid()}")


def _build():
    capi.load()  # makes sure the library exists
    libdir = os.path.dirname(capi.lib_path())
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), SRC, "-o", EXE, "-L", libdir, "-lfimex_b200",
           f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return EXE


def test_cpp_mirror_compiles_and_links():
    exe = _build()
    assert os.path.exists(exe)


@pytest.mark.gpu
def test_reference_unit_tests_through_cpp_mirror():
    exe = _build()
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failures" in r.stdout
