"""Shared scene builders for the parity tests (seeded, small enough for the CPU oracle to finish in seconds)."""
import hashlib
import json
import os

import numpy as np

from better_fastlio2_b200 import synth


def sort_rows(a):
    a = np.asarray(a)
    if len(a) == 0:
        return a
    idx = np.lexsort((a[:, 2], a[:, 1], a[:, 0]))
    return a[idx]


def small_scene(seed=1, model="vlp16", map_half=50.0, ds=0.2, half_extent=120.0):
    rng = np.random.default_rng(seed)
    world = synth.city_world(half_extent=half_extent, seed=seed)
    st_true = synth.trajectory_state(0)
    body = synth.scan_from_pose(world, st_true, synth.lidar_dirs(model, rng), rng)
    mp = synth.sample_surface_map(world, (0, 0, 0), map_half, ds, rng)
    prior = synth.perturb_state(st_true, rng)
    return dict(rng=rng, world=world, st_true=st_true, body=body, map=mp, prior=prior, P=synth.default_cov(), ds=ds)


def knn_equal(d2_a, xyz_a, cnt_a, d2_b, xyz_b, cnt_b):
    """Exact k-NN agreement: counts and sorted float distances bit-equal; coordinates equal wherever a query has no
    duplicated distance (ties may legitimately be ordered differently, SURVEY.md §7 hard part 1)."""
    assert np.array_equal(cnt_a, cnt_b)
    fin = np.isfinite(d2_a)
    assert np.array_equal(fin, np.isfinite(d2_b))
    assert np.array_equal(d2_a[fin], d2_b[fin]), f"max |dd2| = {np.abs(d2_a[fin] - d2_b[fin]).max()}"
    k = d2_a.shape[1]
    tie = np.zeros(len(d2_a), bool)
    for j in range(k - 1):
        tie |= (d2_a[:, j] == d2_a[:, j + 1]) & np.isfinite(d2_a[:, j])
    ok = ~tie
    xa = np.where(np.isfinite(xyz_a[ok]), xyz_a[ok], 0)
    xb = np.where(np.isfinite(xyz_b[ok]), xyz_b[ok], 0)
    assert np.array_equal(xa, xb)
    return int(tie.sum())


def maps_match(a, b, tol=2e-6):
    """Same point set up to float rounding of individual coordinates: the inserted world points are float roundings
    of a double transform, so two engines whose states agree to ~1e-13 can differ by 1 ulp in a few coordinates."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    if len(a) != len(b):
        return False, f"sizes {len(a)} != {len(b)}"
    va = a.view([("", a.dtype)] * 3).ravel()
    vb = b.view([("", b.dtype)] * 3).ravel()
    only_a = a[~np.isin(va, vb)]
    only_b = b[~np.isin(vb, va)]
    if len(only_a) != len(only_b):
        return False, f"unmatched {len(only_a)} vs {len(only_b)}"
    if len(only_a) > max(20, len(a) // 1000):
        return False, f"too many rounding differences: {len(only_a)}"
    for p in only_a:
        d = np.abs(only_b - p).max(1)
        j = int(np.argmin(d))
        if d[j] > tol * max(1.0, float(np.abs(p).max())):
            return False, f"point {p} has no partner within tolerance (best {d[j]})"
        only_b = np.delete(only_b, j, 0)
    return True, f"{len(only_a)} coordinates differ by rounding"


# ---------------------------------------------------------------------------------------------- size-independent properties
def brute_knn_d2(points, q, k=5):
    """k smallest squared distances from q to points in float32, (dx*dx + dy*dy) + dz*dz like calc_dist (ikd_Tree.cpp:1373)."""
    p = np.asarray(points, np.float32)
    q = np.asarray(q, np.float32)
    d = ((p[:, 0] - q[0]) ** 2 + (p[:, 1] - q[1]) ** 2) + (p[:, 2] - q[2]) ** 2
    k = min(k, len(d))
    return np.sort(np.partition(d, k - 1)[:k])


def map_properties(tree, queries, rng, n_brute=32):
    """Properties every exact k-NN map must satisfy at ANY size (used on the CPU with the reference ikd-Tree at a small
    size and on the GPU at BASELINE's full size): sorted distances, coordinates reproduce distances, agreement with a
    brute-force scan of the map's own content, idempotence of the downsampled insert, box delete bookkeeping."""
    queries = np.ascontiguousarray(queries, np.float32)
    content = tree.flatten()
    assert len(content) == tree.validnum() and len(content) >= 5
    xyz, d2, cnt = tree.Nearest_Search(queries, 5)
    assert (cnt == 5).all()
    assert (np.diff(d2, axis=1) >= 0).all()                                     # ascending
    dd = ((xyz[:, :, 0] - queries[:, None, 0]) ** 2 + (xyz[:, :, 1] - queries[:, None, 1]) ** 2) + \
         (xyz[:, :, 2] - queries[:, None, 2]) ** 2
    assert np.array_equal(dd.astype(np.float32), d2)                            # the returned points ARE at those distances
    pick = rng.choice(len(queries), min(n_brute, len(queries)), replace=False)
    for i in pick:
        assert np.array_equal(brute_knn_d2(content, queries[i]), d2[i]), i      # exact: nothing nearer exists in the map
    # downsampled insert twice = once (each touched voxel already holds its winner)
    X = (queries[::3] + rng.normal(0, 0.03, (len(queries[::3]), 3))).astype(np.float32)
    tree.Add_Points(X, True)
    v1, c1 = tree.validnum(), sort_rows(tree.flatten())
    tree.Add_Points(X, True)
    assert tree.validnum() == v1
    c2 = sort_rows(tree.flatten())
    assert np.array_equal(c1, c2)
    # box delete: count, emptiness of the half-open box, search still exact afterwards
    ctr = np.median(queries, axis=0)
    box = np.array([ctr[0] - 6, ctr[1] - 6, ctr[2] - 3, ctr[0] + 6, ctr[1] + 6, ctr[2] + 30], np.float32)
    inside = ((c2 >= box[:3]) & (c2 < box[3:])).all(1)
    nd = tree.Delete_Point_Boxes(box[None, :])
    assert nd == int(inside.sum()) and nd > 0
    after = tree.flatten()
    assert len(after) == len(c2) - nd == tree.validnum()
    assert not ((after >= box[:3]) & (after < box[3:])).all(1).any()
    near = queries[((queries >= box[:3] - 1) & (queries < box[3:] + 1)).all(1)][:8]
    if len(near):
        _, d3, c3 = tree.Nearest_Search(near, 5)
        for j in range(len(near)):
            assert np.array_equal(brute_knn_d2(after, near[j]), d3[j][:c3[j]])
    return dict(map_points=len(content), queries=len(queries), deleted=nd)


# ---------------------------------------------------------------------------------------------- recorded reference ikd-Tree
# The reference's own ikd-Tree is compiled (oracle/_ref) only where its source is present.  What it returned on the call
# sequences of the tests that compare a map with it is kept in tests/golden/ref_ikdtree.json (tests/golden/make_golden_ref.py),
# so those tests run everywhere: the map under test goes through the same calls and must return the same results.
REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ikdtree.json")


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()[:32]


def knn_digest(d2, pts, cnt):
    """What knn_equal compares, as one digest: counts, which distances are finite, the finite distances bit for bit and the
    neighbour records (xyz, or xyz + intensity) of every query without a tied distance."""
    fin = np.isfinite(d2)
    tie = np.zeros(len(d2), bool)
    for j in range(d2.shape[1] - 1):
        tie |= (d2[:, j] == d2[:, j + 1]) & fin[:, j]
    p = pts[~tie]
    return digest(np.asarray(cnt, np.int32), fin, d2[fin], np.where(np.isfinite(p), p, 0).astype(p.dtype))


def _rows4(a):
    a = np.ascontiguousarray(a, np.float32)
    return a[np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0]))]


class RecordedMap:
    """A map back end (reference ikd-Tree, oracle port or the GPU map) that logs every call as [name, digest of the inputs,
    result]: counts as they are, k-NN results as knn_digest, point sets as the digest of their sorted rows."""

    def __init__(self, tree):
        self.tree, self.calls = tree, []

    def _log(self, name, inputs, result=None):
        self.calls.append([name, digest(*[np.asarray(a) for a in inputs]), result])

    def Build(self, pts):
        self.tree.Build(pts)
        self._log("Build", [pts])

    def Build_xyzi(self, pts4):
        self.tree.Build_xyzi(pts4)
        self._log("Build_xyzi", [pts4])

    def Add_Points(self, pts, downsample_on):
        n = int(self.tree.Add_Points(pts, downsample_on))
        self._log("Add_Points", [pts, downsample_on], n)
        return n

    def Add_Points_xyzi(self, pts4, downsample_on):
        n = int(self.tree.Add_Points_xyzi(pts4, downsample_on))
        self._log("Add_Points_xyzi", [pts4, downsample_on], n)
        return n

    def Delete_Point_Boxes(self, boxes):
        n = int(self.tree.Delete_Point_Boxes(boxes))
        self._log("Delete_Point_Boxes", [boxes], n)
        return n

    def Delete_Points(self, pts):
        n = self.tree.Delete_Points(pts)   # the reference returns nothing
        self._log("Delete_Points", [pts])
        return n

    def Nearest_Search(self, q, k=5, max_dist=0.0):
        if not max_dist:
            out = self.tree.Nearest_Search(q, k)
        elif hasattr(self.tree, "Nearest_Search_md"):
            out = self.tree.Nearest_Search_md(q, k, max_dist)
        else:
            out = self.tree.Nearest_Search(q, k, max_dist=max_dist)
        self._log("Nearest_Search", [q, k, max_dist], knn_digest(out[1], out[0], out[2]))
        return out

    def Nearest_Search_xyzi(self, q, k=5):
        out = self.tree.Nearest_Search_xyzi(q, k)
        self._log("Nearest_Search_xyzi", [q, k], knn_digest(out[1], out[0], out[2]))
        return out

    def flatten(self):
        a = self.tree.flatten()
        self._log("flatten", [], digest(sort_rows(a)))
        return a

    def flatten_xyzi(self):
        a = self.tree.flatten_xyzi()
        self._log("flatten_xyzi", [], digest(_rows4(a)))
        return a

    def validnum(self):
        n = int(self.tree.validnum())
        self._log("validnum", [], n)
        return n

    def close(self):
        self.tree.close()


def assert_matches_reference(rec, case, ignore_results_of=()):
    """The calls logged in `rec` returned what the reference ikd-Tree returned on the same calls (`case` in REF_GOLDEN).
    ignore_results_of: calls whose return value is defined differently by the map under test (e.g. the GPU map's Add_Points
    counts changed voxels, the reference counts sequential add operations); their inputs are still checked."""
    with open(REF_GOLDEN) as f:
        want = json.load(f)[case]
    got = rec.calls
    for i, (g, w) in enumerate(zip(got, want)):
        assert g[0] == w[0] and g[1] == w[1], f"{case}: call {i} {g[0]} differs from the recorded call {w[0]} (inputs changed?)"
        if g[0] not in ignore_results_of:
            assert g[2] == w[2], f"{case}: call {i} {g[0]} returned {g[2]}, the reference ikd-Tree {w[2]}"
    assert len(got) == len(want), f"{case}: {len(got)} calls, {len(want)} recorded"
