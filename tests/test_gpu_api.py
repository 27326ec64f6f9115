"""GPU tests of the rest of the KD_TREE API surface and of the other BASELINE configurations (cfg3/cfg4 shapes)."""
import numpy as np
import pytest

from better_fastlio2_b200 import capi, synth
from tests.helpers import small_scene, sort_rows, knn_equal, maps_match, RecordedMap, assert_matches_reference

pytestmark = pytest.mark.gpu


def api_scene():
    return small_scene(seed=4, map_half=35.0, half_extent=100.0)


@pytest.fixture(scope="module")
def scene():
    return api_scene()


# Call sequences run on the GPU map here and on the reference ikd-Tree by tests/golden/make_golden_ref.py, which records the
# reference's results in tests/golden/ref_ikdtree.json.
def nearest_search_calls(m, scene):
    m.Build(scene["map"])
    rng = np.random.default_rng(1)
    world = synth.body_to_world_np(scene["st_true"], scene["body"])[::7]
    q = np.concatenate([world, world[:500] + rng.normal(0, 2.0, (500, 3)).astype(np.float32)]).astype(np.float32)
    for k in (1, 3, 8, 20):
        m.Nearest_Search(q, k)
    for md in (0.3, 1.0):
        xg, dg, cg = m.Nearest_Search(q, 5, max_dist=md)
        assert (dg[np.isfinite(dg)] <= np.float32(md * md) * (1 + 1e-6)).all()


def delete_points_calls(m, scene):
    m.Build(scene["map"])
    victims = scene["map"][::50].copy()
    nd = m.Delete_Points(victims)
    m.validnum()
    m.flatten()
    return nd, len(victims)


def intensity_calls(m, scene):
    """Verbatim Build (multi-point voxels), downsampled Add_Points (voxel winners keep THEIR intensity), verbatim Add_Points,
    a box delete (overflow nodes move into head slots), then Nearest_Search with intensities."""
    rng = np.random.default_rng(11)
    mp = scene["map"]
    m4 = np.column_stack([mp, rng.uniform(0, 255, len(mp)).astype(np.float32)]).astype(np.float32)
    half = len(m4) // 2
    m.Build_xyzi(m4[:half])
    m.flatten_xyzi()
    m.Add_Points_xyzi(m4[half:], True)
    extra = (m4[:3000] + np.array([0.01, 0.0, 0.0, 1.0], np.float32)).astype(np.float32)
    m.Add_Points_xyzi(extra, False)
    m.flatten_xyzi()
    box = np.array([[-8, -8, -3, 8, 8, 1]], np.float32)
    m.Delete_Point_Boxes(box)
    fg = m.flatten_xyzi()
    assert len(fg) == m.validnum()
    # neighbours carry their intensity (compared where the 5 distances are distinct: ties may be ordered differently)
    q = (mp[::97] + rng.normal(0, 0.05, (len(mp[::97]), 3))).astype(np.float32)
    og, dg, cg = m.Nearest_Search_xyzi(q, 5)
    assert (np.diff(dg, axis=1) > 0).all(axis=1).sum() > 100


def test_nearest_search_other_k_and_max_dist(scene):
    t = RecordedMap(capi.KDTree(voxel_size=0.2, max_points=1 << 20, max_blocks=1 << 17))
    nearest_search_calls(t, scene)
    assert_matches_reference(t, "nearest_search_other_k_and_max_dist")
    t.close()


def test_delete_points(scene):
    t = RecordedMap(capi.KDTree(voxel_size=0.2, max_points=1 << 20, max_blocks=1 << 17))
    nd, n = delete_points_calls(t, scene)
    assert nd == n
    assert_matches_reference(t, "delete_points")
    t.close()


def test_capacity_exhaustion_fails_loudly(scene):
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 16, max_blocks=256)
    with pytest.raises(capi.FlbError, match="block pool exhausted|error flags"):
        t.Build(scene["map"])
    t.close()
    # a NaN / unrepresentable point is skipped with a warning, it does not poison the map (the reference keeps running too):
    # the call succeeds, the good points are in, and later calls keep working
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 20, max_blocks=1 << 17)
    t.Build(np.array([[0, 0, 0], [np.nan, 0, 0], [1e12, 0, 0], [1, 1, 1]], np.float32))
    assert t.validnum() == 2
    assert t.Add_Points(np.array([[2, 2, 2], [np.inf, 0, 0]], np.float32), True) == 1
    assert t.validnum() == 3 and len(t.flatten()) == 3
    t.close()
    # scan larger than the session capacity
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 18, max_blocks=1 << 14)
    ses = capi.Session(t, max_scan_points=100)
    with pytest.raises(capi.FlbError, match="exceeds max_scan_points"):
        ses.scan_upload(np.zeros((101, 3), np.float32))
    ses.close()
    t.close()


def test_strided_point_input(scene):
    """PointType = pcl::PointXYZINormal is 48 bytes (common_lib.h:161): xyz at the front of each record."""
    pts48 = np.zeros((len(scene["map"]), 12), np.float32)
    pts48[:, :3] = scene["map"]
    pts48[:, 3:] = 7.0
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 20, max_blocks=1 << 17)
    import ctypes as C
    L = capi.lib()
    assert L.flb_map_build(t.h, pts48.ctypes.data_as(C.c_void_p), len(pts48), 48) == 0
    assert t.validnum() == len(pts48)
    assert np.array_equal(sort_rows(t.flatten()), sort_rows(scene["map"]))
    t.close()


def test_rehash_after_many_deletes(oracle):
    """Deleting most blocks leaves tombstones; the key table is rebuilt and searches / inserts stay exact."""
    rng = np.random.default_rng(2)
    pts = rng.uniform(-40, 40, (60000, 3)).astype(np.float32)   # sparse: ~1 point per block
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 18, max_blocks=1 << 16)
    ref = oracle.make_map(ds=0.2)
    t.Build(pts)
    ref.Build(pts)
    boxes = np.array([[-41, -41, -41, 30, 41, 41]], np.float32)
    assert t.Delete_Point_Boxes(boxes) == ref.Delete_Point_Boxes(boxes)
    st = t.stats()
    assert st["rehash_count"] >= 1 and st["hash_tombstones"] == 0
    q = rng.uniform(-40, 40, (3000, 3)).astype(np.float32)
    xg, dg, cg = t.Nearest_Search(q, 5)
    xr, dr, cr = ref.Nearest_Search(q, 5)
    knn_equal(dg, xg, cg, dr, xr, cr)
    add = rng.uniform(-40, 40, (20000, 3)).astype(np.float32)
    t.Add_Points(add, True)
    ref.Add_Points(add, True)
    assert np.array_equal(sort_rows(t.flatten()), sort_rows(ref.flatten()))
    t.close()


def test_two_sessions_are_independent(oracle):
    """Multi-session replay (cfg5): handles do not share state; interleaved calls give the single-session results."""
    scs = [small_scene(seed=s, map_half=25.0, half_extent=80.0) for s in (5, 6)]
    single = []
    for sc in scs:
        t = capi.KDTree(voxel_size=0.2, max_points=1 << 19, max_blocks=1 << 16)
        t.Build(sc["map"])
        ses = capi.Session(t, max_scan_points=len(sc["body"]), max_iterations=3)
        s, P, r = ses.scan_step(None, sc["body"], sc["prior"], sc["P"], True)
        # with the scan passed in the call the whole step is bracketed by events; the update times itself on the device
        assert 0.0 < r.update.gpu_ms <= r.gpu_ms_total < 1e3
        single.append((s, P, sort_rows(t.flatten())))
        ses.close()
        t.close()
    trees = [capi.KDTree(voxel_size=0.2, max_points=1 << 19, max_blocks=1 << 16) for _ in scs]
    for t, sc in zip(trees, scs):
        t.Build(sc["map"])
    sess = [capi.Session(t, max_scan_points=len(sc["body"]), max_iterations=3) for t, sc in zip(trees, scs)]
    for ses, sc in zip(sess, scs):
        ses.scan_upload(sc["body"])
    outs = [ses.scan_step(None, None, sc["prior"], sc["P"], True) for ses, sc in zip(sess, scs)]
    for (s, P, r), t, ref in zip(outs, trees, single):
        assert np.array_equal(s, ref[0]) and np.array_equal(P, ref[1])
        # scan already on the device: no event pair around the step, update and whole sequence from the device-side stamps
        assert 0.0 < r.update.gpu_ms <= r.gpu_ms_total < 1e3
        assert np.array_equal(sort_rows(t.flatten()), ref[2])
    for ses in sess:
        ses.close()
    for t in trees:
        t.close()


@pytest.mark.parametrize("model,ds,ext,stride", [("hap", 0.1, True, 40), ("os64", 0.2, False, 12), ("hdl64", 0.5, False, 30)])
def test_other_sensor_configs_match_oracle(oracle, model, ds, ext, stride):
    """cfg3 (Livox-HAP shape, 0.1 m voxels, extrinsic estimation, reconstruct), cfg4 (Ouster-64 shape) and a coarse
    voxel size: 3 consecutive scans incl. a reconstruct, per-frame parity with the oracle."""
    seed = 9
    rng = np.random.default_rng(seed)
    world = synth.city_world(half_extent=100, seed=seed)
    dirs = synth.lidar_dirs(model, rng)
    t = capi.KDTree(voxel_size=ds, max_points=1 << 21, max_blocks=1 << 18)
    ref = oracle.make_map(ds=ds)
    st0 = synth.trajectory_state(0)
    mp = synth.sample_surface_map(world, (0, 0, 0), 30.0, ds, rng)
    t.Build(mp)
    ref.Build(mp)
    ses = capi.Session(t, max_scan_points=140000, extrinsic_est_en=ext, max_iterations=3, filter_size_map_min=ds)
    for k in range(3):
        st_true = synth.trajectory_state(k, speed=15.0)
        body = synth.scan_from_pose(world, st_true, dirs, rng, max_range=40.0)[::stride]
        prior = synth.perturb_state(st_true, rng, 0.03, 0.3)
        P = synth.default_cov()
        s_g, P_g, r = ses.scan_step(None, body, prior, P, True)
        s_c, P_c, sc, stc, _ = oracle.esikf_update(prior, P, body, ref, max_iter=3, extrinsic_est_en=ext)
        oracle.map_incremental(s_c, body, sc, ref, True, ds)
        # the two replays agree to ~1e-13 in state; a plane / residual gate sitting exactly on its threshold can flip for
        # a single point, which moves the posterior by ~1e-7 (north_star tolerance: 1e-4 m / rad per frame)
        assert abs(r.update.effct_feat_num - stc[2]) <= 3 and r.update.passes == stc[0]
        assert np.abs(s_g - s_c).max() < 1e-5, (k, np.abs(s_g - s_c).max())
        assert abs(r.map_valid - ref.validnum()) <= 2
        if k == 1:  # recontructIKdTree (laserMapping.cpp:612-669): rebuild from a submap
            sub = t.flatten()[::2].copy()
            t.reconstruct(sub)
            ref.reconstruct(sub)
            assert t.validnum() == ref.validnum() == len(sub)
    a, b = sort_rows(t.flatten()), sort_rows(ref.flatten())
    if len(a) == len(b):
        ok, why = maps_match(a, b)
        assert ok, why
    ses.close()
    t.close()


def test_prefetch_and_split_step_equal_plain_step(oracle):
    """flb_scan_prefetch + flb_scan_step_begin/_finish (double-buffered upload), alternating or with two steps in flight, ==
    flb_scan_step with a host buffer (bit for bit: states, covariances, map contents)."""
    import torch
    scs = [small_scene(seed=s, map_half=25.0, half_extent=80.0) for s in (7, 8, 9)]
    mp = scs[0]["map"]
    outs = []
    for mode in ("plain", "prefetch", "two_in_flight"):
        t = capi.KDTree(voxel_size=0.2, max_points=1 << 19, max_blocks=1 << 16)
        t.Build(mp)
        ses = capi.Session(t, max_scan_points=40000, max_iterations=3)
        res = []
        if mode == "plain":
            for sc in scs:
                s, P, r = ses.scan_step(None, sc["body"], sc["prior"], sc["P"], True)
                res.append((s, P, r.map_valid))
        elif mode == "two_in_flight":
            # replay mode: begin(k+1) before finish(k); finish collects the oldest step; a third begin is refused
            pins = []
            for sc in scs:
                b4 = np.zeros((len(sc["body"]), 4), np.float32)
                b4[:, :3] = sc["body"]
                pins.append(torch.from_numpy(b4).pin_memory())
            sts = [sc["prior"].copy() for sc in scs]
            Ps = [sc["P"].copy() for sc in scs]
            ses.scan_prefetch_ptr(pins[0].data_ptr(), len(scs[0]["body"]), 16)
            ses.scan_step_begin(None, sts[0], Ps[0], True)
            ses.scan_prefetch_ptr(pins[1].data_ptr(), len(scs[1]["body"]), 16)
            for i in range(len(scs)):
                if i + 1 < len(scs):
                    ses.scan_step_begin(None, sts[i + 1], Ps[i + 1], True)
                    if i == 0:
                        with pytest.raises(capi.FlbError, match="two steps are already in flight"):
                            ses.scan_step_begin(None, sts[2], Ps[2], True)
                r = ses.scan_step_finish(None, sts[i], Ps[i])
                if i + 2 < len(scs):
                    ses.scan_prefetch_ptr(pins[i + 2].data_ptr(), len(scs[i + 2]["body"]), 16)
                res.append((sts[i], Ps[i], r.map_valid))
            with pytest.raises(capi.FlbError, match="without flb_scan_step_begin"):
                ses.scan_step_finish(None, sts[0], Ps[0])
        else:
            pins = []
            for sc in scs:
                b4 = np.zeros((len(sc["body"]), 4), np.float32)
                b4[:, :3] = sc["body"]
                pins.append(torch.from_numpy(b4).pin_memory())
            ses.scan_prefetch_ptr(pins[0].data_ptr(), len(scs[0]["body"]), 16)
            for i, sc in enumerate(scs):
                st = sc["prior"].copy()
                P = sc["P"].copy()
                ses.scan_step_begin(None, st, P, True)
                if i + 1 < len(scs):
                    ses.scan_prefetch_ptr(pins[i + 1].data_ptr(), len(scs[i + 1]["body"]), 16)
                r = ses.scan_step_finish(None, st, P)
                res.append((st, P, r.map_valid))
        outs.append((res, sort_rows(t.flatten())))
        ses.close()
        t.close()
    for other in (1, 2):
        for (s0, P0, v0), (s1, P1, v1) in zip(outs[0][0], outs[other][0]):
            assert np.array_equal(s0, s1) and np.array_equal(P0, P1) and v0 == v1, other
        assert np.array_equal(outs[0][1], outs[other][1]), other


def test_map_destroyed_before_session_is_safe(scene):
    """The map is reference counted by its sessions: destroying the KD_TREE handle first must not crash."""
    t = capi.KDTree(voxel_size=0.2, max_points=1 << 19, max_blocks=1 << 16)
    t.Build(scene["map"][:50000])
    ses = capi.Session(t, max_scan_points=1000, max_iterations=3)
    ses.scan_upload(scene["body"][:1000])
    t.close()                       # handle gone, storage kept alive by the session
    s, P, st = ses.update_iterated_dyn_share_modified(scene["prior"], scene["P"])
    assert st["passes"] == 4
    ses.close()


def test_intensity_travels_with_map_points(scene):
    """The reference tree stores whole PointType records (ikd_Tree.h:64-86): intensity comes back from flatten (featsFromMap,
    laserMapping.cpp:2361-2367) and Nearest_Search.  The map operations of intensity_calls return what the reference
    ikd-Tree compiled unmodified returned; then a scan is inserted through map_incremental."""
    m = RecordedMap(capi.KDTree(voxel_size=scene["ds"], max_points=1 << 21, max_blocks=1 << 18))
    intensity_calls(m, scene)
    # Add_Points counts changed voxels here, sequential add operations in the reference
    assert_matches_reference(m, "intensity", ignore_results_of=("Add_Points_xyzi",))
    t = m.tree
    # a scan with intensities through the update + map_incremental: the inserted world points keep the scan's intensity
    body = scene["body"]
    b4 = np.column_stack([body, np.arange(len(body), dtype=np.float32) % 199]).astype(np.float32)
    ses = capi.Session(t, max_scan_points=len(body), max_iterations=3)
    ses.scan_upload_xyzi(b4)
    s, P, st = ses.update_iterated_dyn_share_modified(scene["prior"], scene["P"])
    before = {tuple(r) for r in t.flatten_xyzi().tolist()}
    a, b = ses.map_incremental(s)
    after = t.flatten_xyzi()
    new = np.array([r for r in after.tolist() if tuple(r) not in before], np.float32)
    assert a + b > 0 and len(new) > 0
    world = synth.body_to_world_np(s, body)
    lut = {tuple(w): i for w, i in zip(world.tolist(), b4[:, 3].tolist())}
    hit = [lut.get(tuple(r[:3])) for r in new.tolist()]
    known = [(h, r[3]) for h, r in zip(hit, new.tolist()) if h is not None]
    assert len(known) > 0.9 * len(new) and all(h == v for h, v in known)
    ses.close()
    t.close()


def test_scan_set_device_reads_in_place(oracle):
    """flb_scan_set_device: the scan stays in the caller's device buffer (no copy) — same results as the host upload, also
    with two steps in flight over two different device buffers, and on the host-driven engine."""
    import torch
    scs = [small_scene(seed=s, map_half=25.0, half_extent=80.0) for s in (7, 8, 9)]
    outs = []
    for mode in ("host", "device", "device_two_in_flight", "device_host_engine"):
        t = capi.KDTree(voxel_size=0.2, max_points=1 << 19, max_blocks=1 << 16)
        t.Build(scs[0]["map"])
        ses = capi.Session(t, max_scan_points=40000, max_iterations=3)
        res = []
        devs = []
        for sc in scs:
            b4 = np.zeros((len(sc["body"]), 4), np.float32)
            b4[:, :3] = sc["body"]
            devs.append(torch.from_numpy(b4).cuda())
        torch.cuda.synchronize()
        if mode == "host":
            for sc in scs:
                s, P, r = ses.scan_step(None, sc["body"], sc["prior"], sc["P"], True)
                res.append((s, P, r.map_valid))
        elif mode == "device_two_in_flight":
            sts = [sc["prior"].copy() for sc in scs]
            Ps = [sc["P"].copy() for sc in scs]
            ses.scan_set_device(devs[0].data_ptr(), len(scs[0]["body"]))
            ses.scan_step_begin(None, sts[0], Ps[0], True)
            for i in range(len(scs)):
                if i + 1 < len(scs):
                    ses.scan_set_device(devs[i + 1].data_ptr(), len(scs[i + 1]["body"]))
                    ses.scan_step_begin(None, sts[i + 1], Ps[i + 1], True)
                r = ses.scan_step_finish(None, sts[i], Ps[i])
                res.append((sts[i], Ps[i], r.map_valid))
        else:
            ses.set_update_engine(mode == "device")
            for i, sc in enumerate(scs):
                st, P = sc["prior"].copy(), sc["P"].copy()
                ses.scan_set_device(devs[i].data_ptr(), len(sc["body"]))
                r = ses.scan_step_ptr(None, None, 0, 0, st, P)
                res.append((st, P, r.map_valid))
        outs.append((res, sort_rows(t.flatten())))
        ses.close()
        t.close()
    for other in (1, 2):
        for (s0, P0, v0), (s1, P1, v1) in zip(outs[0][0], outs[other][0]):
            assert np.array_equal(s0, s1) and np.array_equal(P0, P1) and v0 == v1, other
        assert np.array_equal(outs[0][1], outs[other][1]), other
    for (s0, P0, v0), (s1, P1, v1) in zip(outs[0][0], outs[3][0]):     # the host-driven engine agrees to ~1e-13 (other reduction order)
        assert np.abs(s0 - s1).max() < 1e-9 and abs(v0 - v1) <= 2
