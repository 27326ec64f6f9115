"""NumPy statement of Preprocess::process's non-feature branch (src/preprocess.cpp), used by the preprocess tests to
explain the reference's outputs (which point was kept, the per-ring time chain of the Velodyne handler without a time
field and how close each wrap decision was).  The GPU kernels implement the same rules (csrc/frontend_kernels.cuh)."""
import ctypes
import ctypes.util

import numpy as np

from better_fastlio2_b200 import capi

_libm = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
_libm.atan2f.restype = ctypes.c_float
_libm.atan2f.argtypes = [ctypes.c_float, ctypes.c_float]


def atan2f(y, x):
    """The host libm's atan2f, elementwise (the reference calls the float overload)."""
    return np.array([_libm.atan2f(float(a), float(b)) for a, b in zip(y, x)], np.float32)


TIME_SCALE = {0: np.float32(1e3), 1: np.float32(1.0), 2: np.float32(1e-3), 3: np.float32(1e-6)}


def r2(rec):
    x, y, z = rec["x"].astype(np.float32), rec["y"].astype(np.float32), rec["z"].astype(np.float32)
    return ((x * x + y * y) + z * z).astype(np.float64)


def velodyne_yaw_chain(rec, n_scans, scan_rate):
    """Synthesised times of velodyne_handler without a time field (:433-463).  Returns (t, head, margin): t = final
    float32 time per raw point, head = the ring's first point (dropped), margin = |c - time_last| of the wrap test."""
    n = len(rec)
    omega = 0.361 * scan_rate
    yaw = atan2f(rec["y"], rec["x"]).astype(np.float64) * 57.2957
    t = np.zeros(n, np.float32)
    head = np.zeros(n, bool)
    margin = np.full(n, np.inf)
    yaw_fp, t_last = {}, {}
    for i in range(n):
        r = int(rec["ring"][i])
        if r >= n_scans:
            raise IndexError(f"ring {r} of point {i} >= N_SCANS")
        if r not in yaw_fp:
            yaw_fp[r], t_last[r], head[i] = yaw[i], np.float32(0.0), True
            continue
        d = yaw_fp[r] - yaw[i]
        c = np.float32(d / omega) if yaw[i] <= yaw_fp[r] else np.float32((d + 360.0) / omega)
        margin[i] = abs(float(c) - float(t_last[r]))
        if c < t_last[r]:
            c = np.float32(np.float64(c) + 360.0 / omega)
        t[i] = t_last[r] = c
    return t, head, margin


def keep_and_time(rec, lidar_type, n_scans=16, scan_rate=10, point_filter_num=1, time_unit=2, blind=0.01):
    """-> (keep mask over raw points, curvature per raw point, given_offset_time)."""
    n = len(rec)
    idx = np.arange(n)
    b2 = blind * blind
    pf = point_filter_num
    if lidar_type == capi.LIDAR_OUST64:
        return (idx % pf == 0) & ~(r2(rec) < b2), (rec["t"].astype(np.float32) * TIME_SCALE.get(time_unit, 1)), 0
    if lidar_type == capi.LIDAR_VELO16:
        if n == 0:
            return np.zeros(0, bool), np.zeros(0, np.float32), 0
        if rec["time"][-1] > 0:
            return (idx % pf == 0) & (r2(rec) > b2), rec["time"] * TIME_SCALE.get(time_unit, 1), 1
        t, head, _ = velodyne_yaw_chain(rec, n_scans, scan_rate)
        return (idx % pf == 0) & ~head & (r2(rec) > b2), t, 0
    tag = rec["tag"] & 0x30
    valid = (idx >= 1) & (rec["line"] < n_scans) & ((tag == 0x10) | (tag == 0x00))
    sel = valid & ((np.cumsum(valid) % pf) == 0)
    xyz = np.stack([rec["x"], rec["y"], rec["z"]], 1).astype(np.float32)
    prev = np.zeros_like(xyz)
    prev[1:] = np.where(sel[:-1, None], xyz[:-1], 0.0)
    dd = np.abs(xyz - prev).astype(np.float64) > 1e-7
    keep = sel & (dd[:, 0] | dd[:, 1] | (dd[:, 2] & (r2(rec) > b2)))
    return keep, rec["offset_time"].astype(np.float32) / np.float32(1000000), 0


def expected(rec, lidar_type, **cfg):
    """(m, 5) float32 x, y, z, intensity, curvature as pl_surf."""
    keep, t, _ = keep_and_time(rec, lidar_type, **cfg)
    inten = rec["reflectivity"].astype(np.float32) if lidar_type == capi.LIDAR_LIVOX else rec["intensity"]
    cols = [rec["x"], rec["y"], rec["z"], inten, t]
    return np.stack([np.asarray(c, np.float32) for c in cols], 1)[keep]
