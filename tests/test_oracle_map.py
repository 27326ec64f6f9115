"""CPU tests: the oracle's logical map restatement (port) pinned against the REFERENCE ikd-Tree compiled unmodified
(oracle/_ref/libikd_ref.so) — k-NN, Add_Points with/without downsampling, Delete_Point_Boxes.  The reference's results on
these call sequences are recorded in tests/golden/ref_ikdtree.json (tests/golden/make_golden_ref.py)."""
import numpy as np

from tests.helpers import RecordedMap, assert_matches_reference


def map_points():
    rng = np.random.default_rng(0)
    pts = np.concatenate([rng.uniform(-6, 6, (20000, 2)), rng.normal(0, 0.01, (20000, 1))], 1).astype(np.float32)
    wall = np.stack([np.full(8000, 3.0) + rng.normal(0, 0.01, 8000), rng.uniform(-6, 6, 8000), rng.uniform(0, 4, 8000)], 1)
    return np.concatenate([pts, wall.astype(np.float32)])


def knn_calls(m):
    pts = map_points()
    rng = np.random.default_rng(1)
    m.Build(pts)
    q = np.concatenate([pts[:3000] + rng.normal(0, 0.05, (3000, 3)).astype(np.float32),
                        rng.uniform(-30, 30, (300, 3)).astype(np.float32)]).astype(np.float32)
    for k in (1, 5, 8):
        m.Nearest_Search(q, k)


def add_delete_calls(m):
    pts = map_points()
    rng = np.random.default_rng(2)
    m.Build(pts)
    for it in range(3):
        batch = (pts[rng.integers(0, len(pts), 5000)] + rng.normal(0, 0.15, (5000, 3))).astype(np.float32)
        m.Add_Points(batch, True)
        extra = rng.uniform(-7, 7, (300, 3)).astype(np.float32)
        m.Add_Points(extra, False)
        m.validnum()
        m.flatten()
    boxes = np.array([[-7, -7, -1, -2.0, 7, 5], [0, 0, 1.0, 4, 4, 3.0]], np.float32)
    m.Delete_Point_Boxes(boxes)
    m.flatten()
    q = rng.uniform(-6, 6, (1000, 3)).astype(np.float32)
    m.Nearest_Search(q, 5)


def properties_calls(m):
    """The property harness of tests/helpers.map_properties (used at BASELINE's full size on the GPU) on a small map."""
    from tests.helpers import small_scene, map_properties
    from better_fastlio2_b200 import synth
    sc = small_scene(seed=21, map_half=30.0, half_extent=90.0)
    m.Build(sc["map"][:20000])
    m.Add_Points(sc["map"][20000:], True)
    q = synth.body_to_world_np(sc["st_true"], sc["body"])[::5].astype(np.float32)
    info = map_properties(m, q, np.random.default_rng(2))
    assert info["deleted"] > 0


def test_port_knn_equals_reference(oracle):
    m = RecordedMap(oracle.PortMap(ds=0.2))
    knn_calls(m)
    assert_matches_reference(m, "port_knn")


def test_port_add_delete_equals_reference(oracle):
    m = RecordedMap(oracle.PortMap(ds=0.2))
    add_delete_calls(m)
    assert_matches_reference(m, "port_add_delete")


def test_small_and_empty_maps(oracle):
    port = oracle.PortMap(ds=0.2)
    q = np.zeros((2, 3), np.float32)
    x, d, c = port.Nearest_Search(q, 5)
    assert (c == 0).all()
    port.Build(np.array([[1, 1, 1], [2, 2, 2]], np.float32))
    x, d, c = port.Nearest_Search(q, 5)
    assert (c == 2).all() and np.allclose(d[:, 0], 3.0) and np.isinf(d[:, 2:]).all()


def test_size_independent_properties_on_reference_tree(oracle):
    """The property harness holds for the reference's own ikd-Tree at a small size: it runs on the port, which returns
    what the reference returned on every one of the harness's calls."""
    m = RecordedMap(oracle.PortMap(ds=0.2))
    properties_calls(m)
    assert_matches_reference(m, "properties")
