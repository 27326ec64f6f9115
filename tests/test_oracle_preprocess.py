"""The reference's own Preprocess::process (src/preprocess.cpp compiled unmodified into oracle/_ref, see oracle/preprocess_ref.mk)
against the recorded fixture tests/golden/preprocess/ref_preprocess.npz and against the documented rules (tests/preprocess_model.py).
Runs on the CPU; the checks that call the reference skip where it was not built."""
import os
import sys

import numpy as np
import pytest

from better_fastlio2_b200 import capi, synth
from tests import preprocess_model as pm

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_preprocess as mg  # noqa: E402


def _need_ref():
    from oracle import preprocess_ref as po
    if not po.available():
        pytest.skip("oracle/_ref/libpreprocess_ref.so not built (reference tree absent at build time)")
    return po.RefPreprocess()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_golden_file_small_and_complete():
    assert os.path.getsize(mg.OUT) < 1 << 20
    cases = {c["name"]: c for c in mg.load()}
    assert set(cases) == {c[0] for c in mg.CASES}
    assert {c["cfg"]["point_filter_num"] for c in cases.values()} >= {1, 3, 4}
    assert cases["velo_time"]["given_offset_time"] == 1 and cases["velo_yaw"]["given_offset_time"] == 0
    last0 = cases["velo_last_time0"]["records"]["time"]
    assert last0[-1] == 0 and (last0[:-1] > 0).any() and cases["velo_last_time0"]["given_offset_time"] == 0
    assert len(cases["velo_empty"]["records"]) == 0 and len(cases["oust_one"]["records"]) == 1


def test_rules_explain_golden_outputs():
    """The NumPy statement of the handlers reproduces every recorded reference output bit for bit."""
    for c in mg.load():
        e = pm.expected(c["records"], c["lidar_type"], **c["cfg"])
        assert e.shape == c["out"].shape, c["name"]
        assert np.array_equal(_bits(e), _bits(c["out"])), c["name"]


def test_golden_contains_quirks():
    cases = {c["name"]: c for c in mg.load()}
    # Velodyne without a time field: the first point of every ring is dropped
    v = cases["velo_yaw"]
    assert len(v["out"]) == len(v["records"]) - len(np.unique(v["records"]["ring"]))
    # several wraps in one ring: times beyond one revolution (100 ms at 10 Hz) occur
    assert cases["velo_multiwrap"]["out"][:, 4].max() > 110.0
    # Livox: point 0 is never used; :197 keeps a point inside the blind range when x or y changed
    lv = cases["livox_pf3_blind"]
    assert len(cases["livox_one"]["out"]) == 0
    r2 = (lv["out"][:, :3].astype(np.float64) ** 2).sum(1)
    assert (r2 <= lv["cfg"]["blind"] ** 2).any()
    keep, _, _ = pm.keep_and_time(lv["records"], capi.LIDAR_LIVOX, **lv["cfg"])
    assert not keep[0]


def test_live_reference_reproduces_golden():
    _need_ref()
    scans = mg.make_scans()
    outs = mg.reference_outputs(scans)
    for c in mg.load():
        assert scans[c["scan"]].tobytes() == mg._clean(c["records"]).tobytes(), c["name"]
        o, g = outs[c["name"]]
        assert np.array_equal(_bits(o), _bits(c["out"])), c["name"]
        assert g == c["given_offset_time"], c["name"]


def test_reference_quirks_on_hand_made_input():
    ref = _need_ref()
    # Velodyne, no time field: 3 rings x 4 columns; the first point of each ring is dropped
    rec = np.zeros(12, capi.VELODYNE_RECORD)
    az = np.deg2rad(-np.repeat(np.arange(4), 3) * 10.0)
    rec["x"], rec["y"], rec["ring"] = 10 * np.cos(az), 10 * np.sin(az), np.tile(np.arange(3), 4)
    out, g = ref.process(rec, capi.LIDAR_VELO16, n_scans=3, scan_rate=10)
    assert g == 0 and len(out) == 9 and np.array_equal(out[:, 0], rec["x"][3:].astype(np.float32))
    assert np.array_equal(_bits(out[:, [0, 1, 2, 8, 9]]), _bits(pm.expected(rec, capi.LIDAR_VELO16, n_scans=3, scan_rate=10)))
    # Livox: point 0 dropped; a z-only change inside the blind range is dropped, an x change inside it is kept
    lv = np.zeros(5, capi.LIVOX_RECORD)
    lv["x"] = [5.0, 5.0, 0.1, 0.1, 0.2]
    lv["z"] = [0.0, 0.0, 0.0, 0.3, 0.3]
    lv["offset_time"] = [0, 1000, 2000, 3000, 4000]
    out, _ = ref.process(lv, capi.LIDAR_LIVOX, n_scans=6, blind=1.0)
    assert np.array_equal(out[:, 0], np.float32([5.0, 0.1, 0.2]))
    assert np.array_equal(_bits(out[:, [0, 1, 2, 8, 9]]), _bits(pm.expected(lv, capi.LIDAR_LIVOX, n_scans=6, blind=1.0)))


@pytest.mark.parametrize("model,lt", [("hdl64", capi.LIDAR_VELO16), ("os64", capi.LIDAR_OUST64), ("hap", capi.LIDAR_LIVOX)])
def test_rules_match_reference_on_random_scans(model, lt):
    ref = _need_ref()
    rng = np.random.default_rng(99)
    n = 3000
    xyz = rng.normal(0, 20, (n, 3)).astype(np.float32)
    ring = rng.integers(0, 16, n)
    if lt == capi.LIDAR_VELO16:
        rec = synth.velodyne_records(xyz, ring, np.zeros(n, np.float32), rng)
    elif lt == capi.LIDAR_OUST64:
        rec = synth.ouster_records(xyz, ring, rng.integers(0, 10**8, n), rng)
    else:
        rec = synth.livox_records(xyz, ring % 8, rng.integers(0, 10**8, n), rng)
    for pf, bl in ((1, 0.01), (3, 15.0)):
        cfg = dict(n_scans=16 if lt != capi.LIDAR_LIVOX else 6, scan_rate=10, point_filter_num=pf, time_unit=3, blind=bl)
        out, _ = ref.process(rec, lt, **cfg)
        assert np.array_equal(_bits(out[:, [0, 1, 2, 8, 9]]), _bits(pm.expected(rec, lt, **cfg))), (model, pf)
