"""CPU tests of the C-ABI boundary: the library loads, exports every symbol include/fastlio_b200.h declares, and —
with no GPU in this container — fails loudly instead of falling back to any CPU path."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fastlio_b200.h")


@pytest.fixture(scope="module")
def lib():
    from better_fastlio2_b200 import capi
    if not os.path.exists(capi.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return ctypes.CDLL(capi.LIB_PATH)


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(flb_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(lib):
    names = declared_functions()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/fastlio_b200.h but not exported"
    from better_fastlio2_b200 import capi
    assert sorted(capi.EXPORTS) == names


def test_header_cites_reference_interfaces():
    src = open(HEADER).read()
    for cite in ("ikd_Tree.cpp:413-489", "ikd_Tree.cpp:535-556", "ikd_Tree.cpp:366-397", "laserMapping.cpp:1876-2004",
                 "esekfom.hpp:1620-1938", "laserMapping.cpp:1440-1496", "laserMapping.cpp:1136-1200"):
        assert cite in src


def test_no_cpu_fallback(lib):
    """Without a CUDA device the product path must refuse to run (never route through the oracle / a CPU path).  Checked
    in a process that sees no device, so that it also runs on a machine with a GPU."""
    code = ("from better_fastlio2_b200 import capi\n"
            "try:\n    capi.KDTree(voxel_size=0.2)\nexcept capi.FlbError as e:\n    print('FlbError:', e)\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "FlbError:" in out.stdout and "no CUDA device" in out.stdout, out.stdout + out.stderr
    # the package never imports the oracle
    import better_fastlio2_b200
    pkg = os.path.dirname(better_fastlio2_b200.__file__)
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h")):
                txt = open(os.path.join(root, f)).read()
                assert "pyoracle" not in txt and "liblio_oracle" not in txt and "libikd_ref" not in txt, f


def test_struct_layouts_match_header(lib):
    """ctypes mirrors must have the sizes the C compiler gives the header structs."""
    import subprocess
    import tempfile
    from better_fastlio2_b200 import capi
    prog = r'''
#include <stdio.h>
#include "fastlio_b200.h"
int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(flb_map_config), sizeof(flb_map_stats), sizeof(flb_session_config),
 sizeof(flb_pass_result), sizeof(flb_update_stats), sizeof(flb_fov_state), sizeof(flb_scan_result), sizeof(flb_profile));return 0;}
'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(prog)
        exe = os.path.join(d, "t")
        subprocess.run(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    mine = [ctypes.sizeof(x) for x in (capi.MapConfig, capi.MapStats, capi.SessionConfig, capi.PassResult, capi.UpdateStats,
                                       capi.FovState, capi.ScanResult, capi.Profile)]
    assert sizes == mine, (sizes, mine)


def test_frontend_entry_points_reject_bad_arguments(lib):
    """Argument validation of the front-end rows runs before any device work: callable without a GPU."""
    lib.flb_last_error.restype = ctypes.c_char_p
    n = ctypes.c_int(-1)
    vp = ctypes.c_void_p
    lib.flb_voxel_grid_filter.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, vp, ctypes.c_int,
                                          ctypes.POINTER(ctypes.c_int)]
    assert lib.flb_voxel_grid_filter(None, None, 10, 48, 32, ctypes.c_float(0.5), None, 0, ctypes.byref(n)) != 0
    assert b"null map" in lib.flb_last_error()
    lib.flb_frontend_create.argtypes = [vp, ctypes.c_int, ctypes.POINTER(vp)]
    h = vp()
    assert lib.flb_frontend_create(None, 1000, ctypes.byref(h)) != 0 and not h.value
    lib.flb_frontend_upload.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    assert lib.flb_frontend_upload(None, None, 0, 48, 32, 36) != 0
    assert b"null front end" in lib.flb_last_error()
    lib.flb_map_reconstruct_keyframes.argtypes = [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_float, vp,
                                                  ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    assert lib.flb_map_reconstruct_keyframes(None, None, None, 0, 48, 32, None, ctypes.c_float(0.4), None, 0, ctypes.byref(n)) != 0
    lib.flb_frontend_destroy.argtypes = [vp]
    lib.flb_frontend_destroy.restype = None
    lib.flb_frontend_destroy(None)   # destroying a null handle is a no-op


def test_header_cites_frontend_reference_interfaces():
    src = open(HEADER).read()
    for cite in ("IMU_Processing.hpp:243", ":334-386", "laserMapping.cpp:2322-2323", "laserMapping.cpp:1502-1540",
                 "laserMapping.cpp:632-664", "common_lib.h:711-734", "msg/Pose6D.msg"):
        assert cite in src, cite
