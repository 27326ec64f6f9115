"""LiDAR preprocessing on the GPU (flb_frontend_preprocess) per sensor: one JSON line each.

    python tools/preprocess_bench.py [--scans 200] [--warmup 20]

Sensors: HDL-64 (120 000 returns, column-major) with and without a time field, Ouster-64 (64 x 1024), Livox HAP
(240 000 returns).  Reported per scan, medians over --scans scans after --warmup:
  * preprocess_device_ms: CUDA-event time of flb_frontend_preprocess on the session stream (the H2D copy of the
    records, the kernels and the read-back of count / last curvature);
  * gpu_path_ms: raw records -> feats_down_body as flb_frontend_preprocess + undistort + voxel filter (wall clock);
  * host_path_ms: the same with the reference's own Preprocess::process on the host (oracle/_ref, one core) followed
    by flb_frontend_process on its PointType cloud -- the path a node takes without the GPU preprocess (wall clock).
The two paths alternate scan by scan in the same process.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from better_fastlio2_b200 import capi, synth  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        pl = f"unavailable ({e.__class__.__name__})"
    return name, pl


def spinning(world, model, rng):
    d = synth.lidar_dirs(model)
    n_rings = 64
    d = d.reshape(n_rings, -1, 3)[:, ::-1].transpose(1, 0, 2).reshape(-1, 3)   # column-major, clockwise
    r = synth.raycast(world, (0.0, 0.0, 1.8), d, max_range=100.0, min_range=1.0)
    miss = ~np.isfinite(r)
    r[miss] = rng.uniform(30.0, 90.0, miss.sum())   # keep every return so the scan has the sensor's full size
    xyz = (d * r[:, None]).astype(np.float32)
    cols = len(d) // n_rings
    ring = np.tile(np.arange(n_rings), cols)
    col = np.repeat(np.arange(cols), n_rings)
    return xyz, ring, col, cols


def scans(seed=1):
    rng = np.random.default_rng(seed)
    world = synth.city_world(half_extent=150, seed=seed)
    xyz, ring, col, cols = spinning(world, "hdl64", rng)
    t = ((col + 1) / cols * 0.1).astype(np.float32)
    yield "hdl64_time", synth.velodyne_records(xyz, ring, t, rng), capi.LIDAR_VELO16, dict(n_scans=64, time_unit=0, blind=2.0)
    yield "hdl64_notime", synth.velodyne_records(xyz, ring, np.zeros_like(t), rng), capi.LIDAR_VELO16, dict(n_scans=64, blind=2.0)
    xyz, ring, col, cols = spinning(world, "os64", rng)
    yield "os64_1024", synth.ouster_records(xyz, ring, (col * (1e8 / cols)).astype(np.uint32), rng), capi.LIDAR_OUST64, \
        dict(n_scans=64, time_unit=3, blind=2.0)
    d = synth.lidar_dirs("hap", np.random.default_rng(seed))
    r = synth.raycast(world, (0.0, 0.0, 1.0), d, max_range=150.0, min_range=0.5)
    miss = ~np.isfinite(r)
    r[miss] = rng.uniform(30.0, 140.0, miss.sum())
    xyz = (d * r[:, None]).astype(np.float32)
    idx = np.arange(len(d))
    yield "hap_240k", synth.livox_records(xyz, idx % 6, (idx * 416).astype(np.uint32), rng), capi.LIDAR_LIVOX, dict(n_scans=6, blind=0.5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--leaf", type=float, default=0.5)
    args = ap.parse_args()
    import torch
    from oracle import preprocess_ref as po
    name, power = card()
    ref = po.RefPreprocess() if po.available() else None
    tree = capi.KDTree(voxel_size=0.5, max_points=1 << 20, max_blocks=1 << 16)
    ses = capi.Session(tree, max_scan_points=1 << 18, max_iterations=3)
    fe = capi.FrontEnd(ses, max_raw_points=1 << 18)
    stream = torch.cuda.ExternalStream(ses.stream_ptr())
    poses, end = synth.imu_pose_sequence(synth.trajectory_state(1), np.random.default_rng(0))
    poses = np.ascontiguousarray(poses, np.float64)
    end = np.ascontiguousarray(end, np.float64)
    for sensor, rec, lt, cfg in scans():
        cfg = dict(cfg, scan_rate=10, point_filter_num=1)
        cfg.setdefault("time_unit", 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dev, gpu_path, host_path, host_pre = [], [], [], []
        n_out = n_down = 0
        for k in range(args.warmup + args.scans):
            timed = k >= args.warmup
            # (a) GPU preprocess + undistort + voxel filter
            t0 = time.perf_counter()
            e0.record(stream)
            n_out, _ = fe.preprocess(rec, lt, **cfg)
            e1.record(stream)
            fe.undistort(poses, end)
            n_down = fe.voxel_filter(args.leaf)
            t1 = time.perf_counter()
            if timed:
                gpu_path.append((t1 - t0) * 1e3)
                e1.synchronize()
                dev.append(e0.elapsed_time(e1))
            # (b) the reference's host preprocess + flb_frontend_process on its PointType cloud
            if ref is not None:
                t0 = time.perf_counter()
                m, _ = ref.process_into(rec, lt, **cfg)
                t1 = time.perf_counter()
                nd = fe.process_ptr(ref.out.ctypes.data, m, poses, end, args.leaf)
                t2 = time.perf_counter()
                if timed:
                    host_pre.append((t1 - t0) * 1e3)
                    host_path.append((t2 - t0) * 1e3)
                assert m == n_out and nd == n_down, (sensor, m, n_out, nd, n_down)
        med = lambda v: round(float(np.median(v)), 4) if v else None
        print(json.dumps(dict(
            sensor=sensor, points=len(rec), record_bytes=rec.dtype.itemsize, points_out=n_out, feats_down=n_down,
            scans=args.scans, warmup=args.warmup, preprocess_device_ms=med(dev),
            preprocess_device_ms_p90=round(float(np.percentile(dev, 90)), 4), gpu_path_ms=med(gpu_path),
            host_preprocess_ms=med(host_pre), host_path_ms=med(host_path),
            gpu_path_scans_per_s=round(1e3 / med(gpu_path), 1),
            host_path_scans_per_s=round(1e3 / med(host_path), 1) if host_path else None,
            card=name, power_limit=power)), flush=True)
    fe.close()
    ses.close()
    tree.close()


if __name__ == "__main__":
    main()
