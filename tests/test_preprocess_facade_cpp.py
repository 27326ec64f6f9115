"""flb::PreprocessGpu (include/fastlio_b200/preprocess_facade.hpp) compiles against PointCloud2 / CustomMsg look-alikes
without ROS or PCL; on a GPU its result equals the C ABI call on the same points (tests/cpp/preprocess_facade_smoke.cpp)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "preprocess_facade_smoke")


def _build():
    from better_fastlio2_b200 import capi
    if not os.path.exists(capi.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    libdir = os.path.dirname(capi.LIB_PATH)
    cmd = ["/usr/bin/g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "oracle", "shim"), "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "preprocess_facade_smoke.cpp"), "-L", libdir, "-lfastlio_b200", f"-Wl,-rpath,{libdir}",
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-o", EXE]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_preprocess_facade_compiles():
    _build()
    out = subprocess.run([EXE], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "NO_GPU compile-only ok" in out.stdout or "PREPROCESS_FACADE_OK" in out.stdout


@pytest.mark.gpu
def test_preprocess_facade_matches_abi_on_gpu():
    _build()
    out = subprocess.run([EXE], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "PREPROCESS_FACADE_OK" in out.stdout
