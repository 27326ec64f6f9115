"""TEST INFRASTRUCTURE ONLY — ctypes binding of the REFERENCE's own Preprocess (src/preprocess.cpp compiled unmodified
into oracle/_ref/libpreprocess_ref.so by oracle/preprocess_ref.mk, wrapped by oracle/preprocess_ref_wrap.cpp).

May be imported only by tests/, tests/golden/ and tools/preprocess_bench.py; the shipped GPU path never imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_ref", "libpreprocess_ref.so")
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_lib = None


def build(force=False):
    """Compile _ref/libpreprocess_ref.so where the reference tree is present. Building the checker is not using it."""
    if force or (os.path.isdir("/root/reference") and not os.path.exists(_LIB)):
        subprocess.run(["make", "-C", _HERE, "-f", "preprocess_ref.mk", "all"], check=True, capture_output=True)


def available():
    return os.path.exists(_LIB)


def _load():
    global _lib
    if _lib is None:
        build()
        if not available():
            raise RuntimeError("oracle/_ref/libpreprocess_ref.so not built (reference tree absent at build time)")
        L = C.CDLL(_LIB)
        L.ppref_create.restype = C.c_void_p
        L.ppref_destroy.argtypes = [C.c_void_p]
        L.ppref_process.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int,
                                    _f32p, C.c_int, C.POINTER(C.c_int)]
        L.ppref_process.restype = C.c_int
        _lib = L
    return _lib


class RefPreprocess:
    """The reference's Preprocess object (one instance, reused across calls as the node does)."""

    def __init__(self):
        self.L = _load()
        self.h = C.c_void_p(self.L.ppref_create())
        self.out = np.zeros((1, 12), np.float32)

    def close(self):
        if self.h:
            self.L.ppref_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process_into(self, records, lidar_type, n_scans=16, scan_rate=10, point_filter_num=1, time_unit=2, blind=0.01):
        """Preprocess::process on records (the reference's own point structs, see capi.*_RECORD); pl_surf is left in
        self.out[:m] as 48-byte PointType records. Returns (m, given_offset_time)."""
        n = len(records)
        if len(self.out) < max(n, 1):
            self.out = np.zeros((max(n, 1), 12), np.float32)
        g = C.c_int(0)
        m = self.L.ppref_process(self.h, int(lidar_type), int(n_scans), int(scan_rate), int(point_filter_num), int(time_unit),
                                 float(blind), records.ctypes.data if n else None, n, self.out, len(self.out), C.byref(g))
        if m < 0:
            raise ValueError(f"unknown lidar_type {lidar_type}")
        return m, g.value

    def process(self, records, lidar_type, **cfg):
        """As process_into, returning a copy of pl_surf as (m, 12) float32 PointType records and given_offset_time."""
        m, g = self.process_into(np.ascontiguousarray(records), lidar_type, **cfg)
        return self.out[:m].copy(), g
