"""GPU LiDAR preprocessing (flb_frontend_preprocess) against the reference's own Preprocess::process: the recorded
outputs of tests/golden/preprocess/ref_preprocess.npz everywhere, and live on full-size random scans where oracle/_ref is built.

Tolerances: count, order, x/y/z/intensity and copied or scaled times are bit-equal.  Synthesised Velodyne times (no
time field) use a device restatement of the host libm's atan2f; should the host libm compute atan2f differently, a
time may differ by at most 2 float ulp (>= 99.9 % bit-equal), and a wrap decision may flip only where the reference's
own |c - time_last| is within that error (the rest of that ring then follows the flipped chain)."""
import os
import sys

import numpy as np
import pytest

from better_fastlio2_b200 import capi, synth
from tests import preprocess_model as pm

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_preprocess as mg  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = {c["name"]: c for c in mg.load()}


@pytest.fixture(scope="module")
def rig():
    tree = capi.KDTree(voxel_size=0.2, max_points=1 << 21, max_blocks=1 << 18)
    ses = capi.Session(tree, max_scan_points=1 << 18, max_iterations=3)
    fe = capi.FrontEnd(ses, max_raw_points=1 << 18)
    yield tree, ses, fe
    fe.close()
    ses.close()
    tree.close()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _run(fe, rec, lt, cfg):
    n, last = fe.preprocess(rec, lt, **cfg)
    xyzi, cur, _ = fe.download_undistorted()
    assert len(xyzi) == n
    return np.column_stack([xyzi, cur]).astype(np.float32), last


def _check(got, last, ref, rec, lt, cfg, yaw_times):
    assert got.shape == ref.shape
    assert np.array_equal(_bits(got[:, :4]), _bits(ref[:, :4]))
    assert np.float32(last) == (ref[-1, 4] if len(ref) else np.float32(0.0))
    if not yaw_times:
        assert np.array_equal(_bits(got[:, 4]), _bits(ref[:, 4]))
        return
    d = np.abs(_bits(got[:, 4]).astype(np.int64) - _bits(ref[:, 4]).astype(np.int64))
    if len(d) == 0 or (d == 0).all():
        return
    # a point more than 2 ulp off must follow a wrap decision that was a near-tie in the reference
    keep, _, _ = pm.keep_and_time(rec, lt, **cfg)
    raw = np.nonzero(keep)[0]
    _, head, margin = pm.velodyne_yaw_chain(rec, cfg["n_scans"], cfg["scan_rate"])
    ring = rec["ring"][raw]
    for r in np.unique(ring[d > 2]):
        first = raw[(ring == r) & (d > 2)][0]
        ring_pts = np.nonzero((rec["ring"] == rec["ring"][first]) & ~head)[0]
        before = ring_pts[ring_pts <= first]
        assert (margin[before] <= 4 * np.spacing(np.float32(200.0))).any(), f"ring {r}: wrap flipped without a near-tie"
    assert (d[d <= 2] == 0).mean() >= 0.999


@pytest.mark.parametrize("name", sorted(GOLDEN))
def test_golden_case(rig, name):
    c = GOLDEN[name]
    got, last = _run(rig[2], c["records"], c["lidar_type"], c["cfg"])
    yaw = c["lidar_type"] == capi.LIDAR_VELO16 and c["given_offset_time"] == 0
    _check(got, last, c["out"], c["records"], c["lidar_type"], c["cfg"], yaw)


def test_consecutive_scans_of_different_types(rig):
    """The front end keeps no state from one preprocess call to the next."""
    fe = rig[2]
    for name in ("velo_yaw", "livox", "oust_ns", "velo_multiwrap", "velo_time", "velo_empty", "livox_pf3_blind"):
        c = GOLDEN[name]
        got, last = _run(fe, c["records"], c["lidar_type"], c["cfg"])
        yaw = c["lidar_type"] == capi.LIDAR_VELO16 and c["given_offset_time"] == 0
        _check(got, last, c["out"], c["records"], c["lidar_type"], c["cfg"], yaw)


def _full_scans(seed):
    rng = np.random.default_rng(seed)
    world = synth.city_world(half_extent=150, seed=seed)
    xyz, ring, col = synth.sensor_scan(world, "hdl64", rng)
    xyz = np.concatenate([xyz, rng.normal(0, 1.5, (2000, 3)).astype(np.float32)])   # returns inside the blind range
    ring = np.concatenate([ring, rng.integers(0, 64, 2000)])
    col = np.concatenate([col, rng.integers(0, 1875, 2000)])
    perm = np.argsort(col, kind="stable")
    xyz, ring, col = xyz[perm], ring[perm], col[perm]
    t = (col / 1875.0 * 0.1).astype(np.float32)
    yield "hdl64_time", synth.velodyne_records(xyz, ring, t, rng), capi.LIDAR_VELO16, dict(n_scans=64, time_unit=0, blind=4.0)
    yield "hdl64_yaw", synth.velodyne_records(xyz, ring, np.zeros_like(t), rng), capi.LIDAR_VELO16, dict(n_scans=64, blind=4.0)
    xo, ro, co = synth.sensor_scan(world, "os64", rng)
    yield "os64", synth.ouster_records(xo, ro, (co * 97656).astype(np.uint32), rng), capi.LIDAR_OUST64, dict(n_scans=64, time_unit=3,
                                                                                                          blind=2.0)
    xl, ll, cl = synth.sensor_scan(world, "hap", np.random.default_rng(seed + 1), origin=(0.0, 0.0, 1.0))
    yield "hap", synth.livox_records(xl, ll, (cl * 416).astype(np.uint32), rng), capi.LIDAR_LIVOX, dict(n_scans=6, blind=0.5)


@pytest.mark.parametrize("pfn", [1, 3])
def test_full_size_against_live_reference(rig, pfn):
    from oracle import preprocess_ref as po
    if not po.available():
        pytest.skip("oracle/_ref/libpreprocess_ref.so not built")
    ref = po.RefPreprocess()
    for name, rec, lt, cfg in _full_scans(5 + pfn):
        cfg = dict(cfg, point_filter_num=pfn, scan_rate=10)
        cfg.setdefault("time_unit", 0)
        out, g = ref.process(rec, lt, **cfg)
        got, last = _run(rig[2], rec, lt, cfg)
        _check(got, last, out[:, [0, 1, 2, 8, 9]], rec, lt, cfg, lt == capi.LIDAR_VELO16 and g == 0)


def test_preprocess_then_filter_equals_upload_of_reference_cloud(rig):
    """Preprocess -> undistort -> voxel filter == upload of the reference's pl_surf -> the same two calls, bit for bit."""
    tree, ses, fe = rig
    rng = np.random.default_rng(3)
    poses, end = synth.imu_pose_sequence(synth.trajectory_state(2), rng)
    for name in ("velo_yaw", "velo_time", "oust_ns", "livox"):
        c = GOLDEN[name]
        fe.preprocess(c["records"], c["lidar_type"], **c["cfg"])
        fe.undistort(poses, end)
        n1 = fe.voxel_filter(0.5)
        und1 = fe.download_undistorted()
        d1 = fe.download_down()
        o = c["out"]
        fe.upload(capi.pack_pointtype(o[:, :3], o[:, 3], o[:, 4]))
        fe.undistort(poses, end)
        n2 = fe.voxel_filter(0.5)
        und2 = fe.download_undistorted()
        d2 = fe.download_down()
        assert n1 == n2 > 0
        for a, b in zip(und1 + d1, und2 + d2):
            assert np.array_equal(np.asarray(a).view(np.int32), np.asarray(b).view(np.int32)), name


def test_argument_and_capacity_errors(rig):
    tree, ses, fe = rig
    c = GOLDEN["velo_time"]
    rec = c["records"]
    with pytest.raises(capi.FlbError, match="feature"):
        fe.preprocess(rec, capi.LIDAR_VELO16, feature_enabled=1)
    with pytest.raises(capi.FlbError, match="lidar_type"):
        fe.preprocess(rec, 4)
    with pytest.raises(capi.FlbError, match="point_filter_num"):
        fe.preprocess(rec, capi.LIDAR_VELO16, point_filter_num=0)
    with pytest.raises(capi.FlbError, match="n_scans"):
        fe.preprocess(rec, capi.LIDAR_VELO16, n_scans=0)
    with pytest.raises(capi.FlbError, match="outside"):
        lay = capi.raw_layout(rec.dtype, capi.LIDAR_VELO16)
        lay.off_ring = 31
        fe.preprocess(rec, capi.LIDAR_VELO16, layout=lay)
    with pytest.raises(capi.FlbError, match="aligned"):
        lay = capi.raw_layout(rec.dtype, capi.LIDAR_VELO16)
        lay.off_time = 18
        fe.preprocess(rec, capi.LIDAR_VELO16, layout=lay)
    with pytest.raises(capi.FlbError, match="required"):
        lay = capi.raw_layout(rec.dtype, capi.LIDAR_VELO16)
        lay.off_z = -1
        fe.preprocess(rec, capi.LIDAR_VELO16, layout=lay)
    big = np.zeros(fe.cap + 1, capi.OUSTER_RECORD)
    with pytest.raises(capi.FlbError, match="max_raw_points"):
        fe.preprocess(big, capi.LIDAR_OUST64)
    # a ring >= N_SCANS with synthesised times names the ring and the point; with a time field the ring is not read
    bad = GOLDEN["velo_yaw"]["records"].copy()
    bad["ring"][37] = 64
    with pytest.raises(capi.FlbError, match="point 37 has ring 64"):
        fe.preprocess(bad, capi.LIDAR_VELO16, n_scans=64)
    timed = GOLDEN["velo_time"]["records"].copy()
    timed["ring"][37] = 64
    n, _ = fe.preprocess(timed, capi.LIDAR_VELO16, n_scans=64, time_unit=0)
    assert n == len(timed)
    # the front end stays usable after an error
    c = GOLDEN["oust_ns"]
    got, last = _run(fe, c["records"], c["lidar_type"], c["cfg"])
    assert np.array_equal(_bits(got), _bits(c["out"]))
