"""Regenerates tests/golden/preprocess/ref_preprocess.npz: driver records of the three supported LiDAR handlers and what the
REFERENCE's own Preprocess::process (src/preprocess.cpp, compiled unmodified into oracle/_ref/libpreprocess_ref.so)
returns for them, so that the GPU preprocess is checked against the reference from any checkout.

    python tests/golden/make_golden_preprocess.py        (needs oracle/_ref/libpreprocess_ref.so)

Layout: scan_<name> = the records as bytes (dtype per `kind`: capi.VELODYNE_RECORD / OUSTER_RECORD / LIVOX_RECORD);
case_<name>_out = pl_surf as (m, 5) float32 x, y, z, intensity, curvature; `cases` = one row per case:
name, scan, lidar_type, n_scans, scan_rate, point_filter_num, time_unit, blind, given_offset_time.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from better_fastlio2_b200 import capi, synth  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "preprocess", "ref_preprocess.npz")
KIND = {capi.LIDAR_VELO16: capi.VELODYNE_RECORD, capi.LIDAR_OUST64: capi.OUSTER_RECORD, capi.LIDAR_LIVOX: capi.LIVOX_RECORD}
CASE_FIELDS = ("name", "scan", "lidar_type", "n_scans", "scan_rate", "point_filter_num", "time_unit", "blind", "given_offset_time")


def make_scans():
    rng = np.random.default_rng(23)
    world = synth.city_world(half_extent=120, seed=23)
    sc = {}
    # HDL-64 ordering (column-major, clockwise), 64 columns over the full turn
    xyz, ring, col = synth.sensor_scan(world, "hdl64", rng, columns=64)
    t_s = (col / 64.0 * 0.1).astype(np.float32)
    t_s[rng.integers(0, len(t_s), len(t_s) // 50)] = 0.0   # a few returns without a stamp
    sc["hdl64_time"] = synth.velodyne_records(xyz, ring, t_s, rng)
    sc["hdl64_notime"] = synth.velodyne_records(xyz, ring, np.zeros(len(xyz), np.float32), rng)
    # last point stamped 0 although the others carry times -> the reference synthesises from yaw
    r = sc["hdl64_time"][:700].copy()
    r["time"][-1] = 0.0
    sc["hdl64_last_time0"] = r
    # rings whose azimuth sweeps 2.5 turns (clockwise) or 1.5 turns (counter-clockwise): several wraps past yaw_fp
    n_per, rings = 150, 8
    pts = []
    for k in range(n_per):
        for rg in range(rings):
            turns = -900.0 if rg % 2 == 0 else 540.0
            az = np.deg2rad(turns * k / (n_per - 1) + 7.0 * rg + rng.uniform(-0.05, 0.05))
            rr = 5.0 + 10.0 * rng.random()
            pts.append((rr * np.cos(az), rr * np.sin(az), 0.3 * rg - 1.0, rg))
    pts = np.array(pts)
    sc["multiwrap"] = synth.velodyne_records(pts[:, :3].astype(np.float32), pts[:, 3].astype(int), np.zeros(len(pts), np.float32), rng)
    # Ouster-64, 32 columns; t in ns (time_unit 3) and in us (time_unit 2)
    xyz, ring, col = synth.sensor_scan(world, "os64", rng, columns=32)
    t_ns = (col / 32.0 * 1e8).astype(np.uint32) + rng.integers(0, 1000, len(col)).astype(np.uint32)
    sc["os64_ns"] = synth.ouster_records(xyz, ring, t_ns, rng)
    sc["os64_us"] = synth.ouster_records(xyz, ring, (t_ns // 1000).astype(np.uint32), rng)
    # Livox HAP, first 3000 returns: mixed tags, lines 0..7 (6 and 7 >= N_SCANS = 6), consecutive duplicates, zeros
    xyz, line, col = synth.sensor_scan(world, "hap", np.random.default_rng(3), columns=3000, origin=(0.0, 0.0, 1.0))
    n = len(xyz)
    line = line.copy()
    line[rng.integers(0, n, n // 20)] = rng.integers(6, 8, n // 20)
    xyz = xyz.copy()
    dup = rng.integers(1, n, n // 15)
    xyz[dup] = xyz[dup - 1]                                       # exact duplicate of the previous return
    dz = rng.integers(1, n, n // 30)
    xyz[dz, :2] = xyz[dz - 1, :2]                                 # same x, y; z differs -> only the z term decides
    xyz[dz, 2] += 0.5
    near = rng.integers(1, n, n // 30)
    xyz[near] *= 0.05                                             # inside the blind range
    zero = rng.integers(1, n, n // 100)
    xyz[zero] = 0.0
    off = (col.astype(np.int64) * 33333).astype(np.uint32)
    sc["hap_mixed"] = synth.livox_records(xyz, line, off, rng)
    # tiny scans
    sc["velo_one"] = sc["hdl64_time"][-1:].copy()
    sc["velo_one_notime"] = sc["hdl64_notime"][5:6].copy()
    sc["velo_empty"] = sc["hdl64_time"][:0].copy()
    sc["os_one"] = sc["os64_ns"][3:4].copy()
    sc["os_empty"] = sc["os64_ns"][:0].copy()
    sc["livox_one"] = sc["hap_mixed"][:1].copy()
    sc["livox_two"] = sc["hap_mixed"][:2].copy()
    sc["livox_empty"] = sc["hap_mixed"][:0].copy()
    return {k: _clean(v) for k, v in sc.items()}


def _clean(rec):
    """The same records with zeroed padding (slicing copies of structured arrays leave it undefined)."""
    out = np.zeros(len(rec), rec.dtype)
    for f in rec.dtype.names:
        out[f] = rec[f]
    return out


V, O, L = capi.LIDAR_VELO16, capi.LIDAR_OUST64, capi.LIDAR_LIVOX
# name, scan, lidar_type, n_scans, scan_rate, point_filter_num, time_unit, blind
CASES = [
    ("velo_time", "hdl64_time", V, 64, 10, 1, 0, 0.01),
    ("velo_time_pf4_blind", "hdl64_time", V, 64, 10, 4, 0, 6.0),
    ("velo_yaw", "hdl64_notime", V, 64, 10, 1, 0, 0.01),
    ("velo_yaw_pf3_blind", "hdl64_notime", V, 64, 10, 3, 0, 6.0),
    ("velo_yaw_rate20", "hdl64_notime", V, 64, 20, 1, 2, 4.0),
    ("velo_last_time0", "hdl64_last_time0", V, 64, 10, 1, 0, 0.01),
    ("velo_multiwrap", "multiwrap", V, 8, 10, 1, 0, 0.01),
    ("velo_multiwrap_pf3", "multiwrap", V, 16, 10, 3, 0, 8.0),
    ("oust_ns", "os64_ns", O, 64, 10, 1, 3, 0.5),
    ("oust_us_pf3_blind", "os64_us", O, 64, 10, 3, 2, 5.0),
    ("livox", "hap_mixed", L, 6, 10, 1, 3, 0.01),
    ("livox_pf3_blind", "hap_mixed", L, 6, 10, 3, 3, 2.0),
    ("livox_pf4_blind", "hap_mixed", L, 4, 10, 4, 3, 0.5),
    ("velo_one", "velo_one", V, 64, 10, 1, 0, 0.01),
    ("velo_one_notime", "velo_one_notime", V, 64, 10, 1, 0, 0.01),
    ("velo_empty", "velo_empty", V, 64, 10, 1, 0, 0.01),
    ("oust_one", "os_one", O, 64, 10, 1, 3, 0.01),
    ("oust_empty", "os_empty", O, 64, 10, 1, 3, 0.01),
    ("livox_one", "livox_one", L, 6, 10, 1, 3, 0.01),
    ("livox_two", "livox_two", L, 6, 10, 1, 3, 0.01),
    ("livox_empty", "livox_empty", L, 6, 10, 1, 3, 0.01),
]


def load(path=OUT):
    """-> list of dicts: name, records (structured array), cfg (kwargs of FrontEnd.preprocess), out (m,5), given_offset_time."""
    z = np.load(path)
    res = []
    for row in z["cases"]:
        d = dict(zip(CASE_FIELDS, row))
        lt = int(d["lidar_type"])
        rec = np.frombuffer(z["scan_" + d["scan"]].tobytes(), KIND[lt]).copy()
        cfg = dict(n_scans=int(d["n_scans"]), scan_rate=int(d["scan_rate"]), point_filter_num=int(d["point_filter_num"]),
                   time_unit=int(d["time_unit"]), blind=float(d["blind"]))
        res.append(dict(name=str(d["name"]), scan=str(d["scan"]), lidar_type=lt, records=rec, cfg=cfg,
                        out=z["case_" + d["name"] + "_out"], given_offset_time=int(d["given_offset_time"])))
    return res


def reference_outputs(scans, cases=CASES):
    from oracle import preprocess_ref as po
    ref = po.RefPreprocess()
    outs = {}
    for name, scan, lt, ns, sr, pf, tu, bl in cases:
        o, g = ref.process(scans[scan], lt, n_scans=ns, scan_rate=sr, point_filter_num=pf, time_unit=tu, blind=bl)
        outs[name] = (o[:, [0, 1, 2, 8, 9]].copy(), g)
    return outs


def main():
    scans = make_scans()
    outs = reference_outputs(scans)
    arrays = {"scan_" + k: np.frombuffer(v.tobytes(), np.uint8) for k, v in scans.items()}
    rows = []
    for name, scan, lt, ns, sr, pf, tu, bl in CASES:
        o, g = outs[name]
        arrays["case_" + name + "_out"] = o
        rows.append((name, scan, str(lt), str(ns), str(sr), str(pf), str(tu), repr(bl), str(g)))
        print(f"{name:22s} {len(scans[scan]):6d} -> {len(o):6d}  given_offset_time={g}")
    arrays["cases"] = np.array(rows)
    np.savez_compressed(OUT, **arrays)
    print("ref_preprocess.npz", os.path.getsize(OUT) // 1024, "KiB")


if __name__ == "__main__":
    main()
