"""ctypes view of the C ABI in include/fastlio_b200.h (libfastlio_b200.so, hand-written sm_100a CUDA).

This is plumbing for tests / bench only: the product is the shared library and the C++ facades under
include/fastlio_b200/.  Class and method names mirror the reference interface they stand in for
(KD_TREE: include/ikd-Tree/ikd_Tree.h:225-249; esekf update + h_share_model: esekfom.hpp:1620, laserMapping.cpp:1876).

There is NO CPU fallback: if the CUDA library is missing or no device is visible, calls raise FlbError.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FLB_LIB selects another build of the SAME library (debug/trace or A/B kernel variants); there is still no CPU fallback
LIB_PATH = os.environ.get("FLB_LIB") or os.path.join(_HERE, "libfastlio_b200.so")

NACC_DOF = 23


class FlbError(RuntimeError):
    pass


class MapConfig(C.Structure):
    _fields_ = [("voxel_size", C.c_float), ("max_points", C.c_int), ("max_blocks", C.c_int), ("device", C.c_int)]


class MapStats(C.Structure):
    _fields_ = [("valid_points", C.c_int), ("blocks_in_use", C.c_int), ("block_capacity", C.c_int),
                ("overflow_in_use", C.c_int), ("overflow_capacity", C.c_int), ("hash_capacity", C.c_int),
                ("hash_tombstones", C.c_int), ("coarse_cells", C.c_int), ("rehash_count", C.c_int),
                ("device_bytes", C.c_size_t)]


class SessionConfig(C.Structure):
    _fields_ = [("max_scan_points", C.c_int), ("extrinsic_est_en", C.c_int), ("max_iterations", C.c_int),
                ("laser_point_cov", C.c_double), ("filter_size_map_min", C.c_double), ("limit", C.c_double * 23)]


class PassResult(C.Structure):
    _fields_ = [("valid", C.c_int), ("effct_feat_num", C.c_int), ("total_residual", C.c_double),
                ("HTH", C.c_double * 144), ("HTh", C.c_double * 12)]


class UpdateStats(C.Structure):
    _fields_ = [("passes", C.c_int), ("search_passes", C.c_int), ("effct_feat_num", C.c_int),
                ("converged_count", C.c_int), ("total_residual", C.c_double), ("gpu_ms", C.c_float)]


class FovState(C.Structure):
    _fields_ = [("local_map_min", C.c_float * 3), ("local_map_max", C.c_float * 3), ("initialized", C.c_int),
                ("cube_len", C.c_double), ("det_range", C.c_float), ("pos_lid", C.c_double * 3)]


class ScanResult(C.Structure):
    _fields_ = [("update", UpdateStats), ("n_to_add", C.c_int), ("n_no_downsample", C.c_int), ("n_deleted", C.c_int),
                ("map_valid", C.c_int), ("gpu_ms_total", C.c_float), ("kernel_launches", C.c_int)]


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 8), ("launches", C.c_int * 8), ("regions", C.c_int * 8), ("knn_phase", C.c_longlong * 4),
                ("knn_head_candidates", C.c_longlong), ("knn_chain_nodes", C.c_longlong), ("knn_chain_max", C.c_longlong)]


K_CLASSES = ["transform", "knn", "residual", "reduce", "classify", "insert", "delete"]

class PreprocessCfg(C.Structure):
    _fields_ = [("lidar_type", C.c_int), ("n_scans", C.c_int), ("scan_rate", C.c_int), ("point_filter_num", C.c_int),
                ("time_unit", C.c_int), ("blind", C.c_double), ("feature_enabled", C.c_int)]


class RawLayout(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("stride", "off_x", "off_y", "off_z", "off_intensity", "off_time", "off_ring", "off_tag",
                                       "off_line")]


_lib = None

# every symbol include/fastlio_b200.h declares
EXPORTS = [
    "flb_last_error", "flb_device_count", "flb_version", "flb_map_create", "flb_map_destroy",
    "flb_map_set_downsample_param", "flb_map_has_root", "flb_map_build", "flb_map_reconstruct", "flb_map_add_points",
    "flb_map_delete_boxes", "flb_map_delete_points", "flb_map_nearest_search", "flb_map_box_search",
    "flb_map_radius_search", "flb_map_validnum", "flb_map_size", "flb_map_flatten", "flb_map_range",
    "flb_map_get_stats", "flb_session_default_config", "flb_session_create", "flb_session_destroy", "flb_scan_upload",
    "flb_scan_set_device", "flb_pass", "flb_pass_rows", "flb_esikf_update", "flb_map_incremental",
    "flb_neighbors_download", "flb_fov_segment", "flb_scan_step", "flb_session_stream", "flb_session_sync",
    "flb_map_profile_enable", "flb_map_profile_read", "flb_session_set_update_engine", "flb_scan_prefetch", "flb_scan_step_begin", "flb_scan_step_finish",
    "flb_frontend_create", "flb_frontend_destroy", "flb_frontend_upload", "flb_frontend_undistort",
    "flb_frontend_voxel_filter", "flb_frontend_process", "flb_frontend_download_undistorted", "flb_frontend_download_down",
    "flb_frontend_points_to_world", "flb_voxel_grid_filter", "flb_map_reconstruct_keyframes", "flb_frontend_preprocess",
    "flb_map_build_pt", "flb_map_reconstruct_pt", "flb_map_add_points_pt", "flb_map_nearest_search_xyzi",
    "flb_map_box_search_xyzi", "flb_map_radius_search_xyzi", "flb_map_flatten_xyzi", "flb_scan_upload_pt",
]


def lib():
    """Load the CUDA library. Fails loudly when it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FlbError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, ip, fp, dp = C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p
        L.flb_last_error.restype = C.c_char_p
        L.flb_version.restype = C.c_char_p
        L.flb_map_create.argtypes = [C.POINTER(MapConfig), C.POINTER(vp)]
        L.flb_map_destroy.argtypes = [vp]
        L.flb_map_destroy.restype = None
        L.flb_map_set_downsample_param.argtypes = [vp, C.c_float]
        L.flb_map_has_root.argtypes = [vp]
        L.flb_map_build.argtypes = [vp, fp, C.c_int, C.c_int]
        L.flb_map_reconstruct.argtypes = [vp, fp, C.c_int, C.c_int]
        L.flb_map_add_points.argtypes = [vp, fp, C.c_int, C.c_int, C.c_int, ip]
        L.flb_map_build_pt.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int]
        L.flb_map_reconstruct_pt.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int]
        L.flb_map_add_points_pt.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, ip]
        L.flb_map_nearest_search_xyzi.argtypes = [vp, fp, C.c_int, C.c_int, C.c_int, C.c_float, fp, fp, vp]
        L.flb_map_box_search_xyzi.argtypes = [vp, fp, fp, C.c_int, ip]
        L.flb_map_radius_search_xyzi.argtypes = [vp, fp, C.c_float, fp, C.c_int, ip]
        L.flb_map_flatten_xyzi.argtypes = [vp, fp, C.c_int, ip]
        L.flb_scan_upload_pt.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int]
        L.flb_map_delete_boxes.argtypes = [vp, fp, C.c_int, ip]
        L.flb_map_delete_points.argtypes = [vp, fp, C.c_int, C.c_int, ip]
        L.flb_map_nearest_search.argtypes = [vp, fp, C.c_int, C.c_int, C.c_int, C.c_float, fp, fp, vp]
        L.flb_map_box_search.argtypes = [vp, fp, fp, C.c_int, ip]
        L.flb_map_radius_search.argtypes = [vp, fp, C.c_float, fp, C.c_int, ip]
        L.flb_map_validnum.argtypes = [vp]
        L.flb_map_size.argtypes = [vp]
        L.flb_map_flatten.argtypes = [vp, fp, C.c_int, ip]
        L.flb_map_range.argtypes = [vp, fp]
        L.flb_map_get_stats.argtypes = [vp, C.POINTER(MapStats)]
        L.flb_session_default_config.argtypes = [C.POINTER(SessionConfig)]
        L.flb_session_default_config.restype = None
        L.flb_session_create.argtypes = [vp, C.POINTER(SessionConfig), C.POINTER(vp)]
        L.flb_session_destroy.argtypes = [vp]
        L.flb_session_destroy.restype = None
        L.flb_scan_upload.argtypes = [vp, fp, C.c_int, C.c_int]
        L.flb_scan_set_device.argtypes = [vp, vp, C.c_int]
        L.flb_scan_prefetch.argtypes = [vp, fp, C.c_int, C.c_int]
        L.flb_pass.argtypes = [vp, dp, C.c_int, C.POINTER(PassResult)]
        L.flb_pass_rows.argtypes = [vp, dp, C.c_int, dp, C.c_int, ip]
        L.flb_esikf_update.argtypes = [vp, dp, dp, C.POINTER(UpdateStats)]
        L.flb_map_incremental.argtypes = [vp, dp, C.c_int, ip, ip]
        L.flb_neighbors_download.argtypes = [vp, fp, fp, vp, vp, fp, fp]
        L.flb_fov_segment.argtypes = [vp, C.POINTER(FovState), dp, fp, ip, ip]
        L.flb_scan_step.argtypes = [vp, C.POINTER(FovState), fp, C.c_int, C.c_int, dp, dp, C.c_int, C.POINTER(ScanResult)]
        L.flb_scan_step_begin.argtypes = [vp, C.POINTER(FovState), fp, C.c_int, C.c_int, dp, dp, C.c_int]
        L.flb_scan_step_finish.argtypes = [vp, C.POINTER(FovState), dp, dp, C.POINTER(ScanResult)]
        L.flb_session_stream.argtypes = [vp]
        L.flb_session_stream.restype = vp
        L.flb_session_sync.argtypes = [vp]
        L.flb_session_set_update_engine.argtypes = [vp, C.c_int]
        L.flb_map_profile_enable.argtypes = [vp, C.c_int]
        L.flb_map_profile_read.argtypes = [vp, C.POINTER(Profile), C.c_int]
        L.flb_frontend_create.argtypes = [vp, C.c_int, C.POINTER(vp)]
        L.flb_frontend_destroy.argtypes = [vp]
        L.flb_frontend_destroy.restype = None
        L.flb_frontend_upload.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int]
        L.flb_frontend_preprocess.argtypes = [vp, vp, C.c_int, C.POINTER(RawLayout), C.POINTER(PreprocessCfg), ip,
                                              C.POINTER(C.c_float)]
        L.flb_frontend_undistort.argtypes = [vp, dp, C.c_int, dp]
        L.flb_frontend_voxel_filter.argtypes = [vp, C.c_float, ip]
        L.flb_frontend_process.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, dp, C.c_int, dp, C.c_float, ip]
        L.flb_frontend_download_undistorted.argtypes = [vp, fp, fp, vp, C.c_int, ip]
        L.flb_frontend_download_down.argtypes = [vp, fp, fp, C.c_int, ip]
        L.flb_frontend_points_to_world.argtypes = [vp, C.c_int, dp, fp, C.c_int, ip]
        L.flb_voxel_grid_filter.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_float, fp, C.c_int, ip]
        L.flb_map_reconstruct_keyframes.argtypes = [vp, C.POINTER(vp), ip, C.c_int, C.c_int, C.c_int, fp, C.c_float, fp,
                                                    C.c_int, ip]
        _lib = L
    return _lib


def _chk(rc):
    if rc != 0:
        raise FlbError(lib().flb_last_error().decode())


def _xyz(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("points must be (n,3) or (n,4) float32")
    return a


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class KDTree:
    """Device hashed-voxel map behind the KD_TREE<PointType> API of the reference (ikd_Tree.h:225-249)."""

    def __init__(self, voxel_size=0.2, max_points=1 << 20, max_blocks=0, device=0):
        self.h = C.c_void_p()
        cfg = MapConfig(float(voxel_size), int(max_points), int(max_blocks), int(device))
        _chk(lib().flb_map_create(C.byref(cfg), C.byref(self.h)))
        self.voxel_size = float(voxel_size)
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            lib().flb_map_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_downsample_param(self, v):
        _chk(lib().flb_map_set_downsample_param(self.h, float(v)))

    @property
    def Root_Node(self):
        return True if lib().flb_map_has_root(self.h) else None

    def Build(self, pts):
        pts = _xyz(pts)
        _chk(lib().flb_map_build(self.h, _p(pts), len(pts), pts.strides[0]))

    def reconstruct(self, pts):
        pts = _xyz(pts)
        _chk(lib().flb_map_reconstruct(self.h, _p(pts), len(pts), pts.strides[0]))

    def Add_Points(self, pts, downsample_on):
        pts = _xyz(pts)
        n = C.c_int(0)
        _chk(lib().flb_map_add_points(self.h, _p(pts), len(pts), pts.strides[0], 1 if downsample_on else 0, C.byref(n)))
        return n.value

    # PointType-aware variants: (n, 4) arrays of x, y, z, intensity (ikd_Tree.h:64-86 keeps whole records)
    def Build_xyzi(self, pts4):
        a = np.ascontiguousarray(pts4, np.float32).reshape(-1, 4)
        _chk(lib().flb_map_build_pt(self.h, _p(a), len(a), 16, 12))

    def Add_Points_xyzi(self, pts4, downsample_on):
        a = np.ascontiguousarray(pts4, np.float32).reshape(-1, 4)
        n = C.c_int(0)
        _chk(lib().flb_map_add_points_pt(self.h, _p(a), len(a), 16, 12, 1 if downsample_on else 0, C.byref(n)))
        return n.value

    def Build_pointtype(self, points48):
        a = np.ascontiguousarray(points48, np.float32).reshape(-1, 12)
        _chk(lib().flb_map_build_pt(self.h, _p(a), len(a), POINT_STRIDE, OFF_INTENSITY))

    def Nearest_Search_xyzi(self, q, k=5, max_dist=0.0):
        q = _xyz(q)
        n = len(q)
        out = np.empty((n, k, 4), np.float32)
        d2 = np.empty((n, k), np.float32)
        cnt = np.empty(n, np.int32)
        _chk(lib().flb_map_nearest_search_xyzi(self.h, _p(q), n, q.strides[0], k, float(max_dist), _p(out), _p(d2), _p(cnt)))
        return out, d2, cnt

    def flatten_xyzi(self):
        n = C.c_int(0)
        _chk(lib().flb_map_flatten_xyzi(self.h, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 4), np.float32)
        n2 = C.c_int(0)
        _chk(lib().flb_map_flatten_xyzi(self.h, _p(out), n.value, C.byref(n2)))
        return out[:min(n.value, n2.value)].copy()

    def Box_Search_xyzi(self, box6, cap=1 << 20):
        b = np.ascontiguousarray(box6, np.float32).reshape(6)
        out = np.empty((cap, 4), np.float32)
        n = C.c_int(0)
        _chk(lib().flb_map_box_search_xyzi(self.h, _p(b), _p(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()

    def Delete_Point_Boxes(self, boxes):
        b = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
        n = C.c_int(0)
        _chk(lib().flb_map_delete_boxes(self.h, _p(b), len(b), C.byref(n)))
        return n.value

    def Delete_Points(self, pts):
        pts = _xyz(pts)
        n = C.c_int(0)
        _chk(lib().flb_map_delete_points(self.h, _p(pts), len(pts), pts.strides[0], C.byref(n)))
        return n.value

    def Nearest_Search(self, q, k=5, max_dist=0.0):
        q = _xyz(q)
        n = len(q)
        xyz = np.empty((n, k, 3), np.float32)
        d2 = np.empty((n, k), np.float32)
        cnt = np.empty(n, np.int32)
        _chk(lib().flb_map_nearest_search(self.h, _p(q), n, q.strides[0], k, float(max_dist), _p(xyz), _p(d2), _p(cnt)))
        return xyz, d2, cnt

    def Box_Search(self, box6, cap=1 << 20):
        b = np.ascontiguousarray(box6, np.float32).reshape(6)
        out = np.empty((cap, 3), np.float32)
        n = C.c_int(0)
        _chk(lib().flb_map_box_search(self.h, _p(b), _p(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()

    def Radius_Search(self, center, radius, cap=1 << 20):
        c = np.ascontiguousarray(center, np.float32).reshape(3)
        out = np.empty((cap, 3), np.float32)
        n = C.c_int(0)
        _chk(lib().flb_map_radius_search(self.h, _p(c), float(radius), _p(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()

    def validnum(self):
        v = lib().flb_map_validnum(self.h)
        if v < 0:
            raise FlbError(lib().flb_last_error().decode())
        return v

    def size(self):
        return self.validnum()

    def flatten(self):
        n = C.c_int(0)
        _chk(lib().flb_map_flatten(self.h, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 3), np.float32)
        n2 = C.c_int(0)
        _chk(lib().flb_map_flatten(self.h, _p(out), n.value, C.byref(n2)))
        return out[:min(n.value, n2.value)].copy()

    def tree_range(self):
        b = np.zeros(6, np.float32)
        _chk(lib().flb_map_range(self.h, _p(b)))
        return b

    def profile_enable(self, on=True):
        _chk(lib().flb_map_profile_enable(self.h, 1 if on else 0))

    def profile_read(self, reset=True):
        p = Profile()
        _chk(lib().flb_map_profile_read(self.h, C.byref(p), 1 if reset else 0))
        out = {}
        for i, k in enumerate(K_CLASSES):
            out[k] = {"ms": p.ms[i], "launches": p.launches[i], "regions": p.regions[i]}
        out["knn_phase"] = [int(p.knn_phase[i]) for i in range(4)]
        out["knn_head_candidates"] = int(p.knn_head_candidates)
        out["knn_chain_nodes"] = int(p.knn_chain_nodes)
        out["knn_chain_max"] = int(p.knn_chain_max)
        return out

    def stats(self):
        s = MapStats()
        _chk(lib().flb_map_get_stats(self.h, C.byref(s)))
        return {f[0]: getattr(s, f[0]) for f in MapStats._fields_}


class Session:
    """Per-scan measurement context: h_share_model + update_iterated_dyn_share_modified + map_incremental."""

    def __init__(self, tree, max_scan_points=131072, extrinsic_est_en=False, max_iterations=4, laser_point_cov=0.001,
                 filter_size_map_min=None, limit=None):
        self.tree = tree
        cfg = SessionConfig()
        lib().flb_session_default_config(C.byref(cfg))
        cfg.max_scan_points = int(max_scan_points)
        cfg.extrinsic_est_en = 1 if extrinsic_est_en else 0
        cfg.max_iterations = int(max_iterations)
        cfg.laser_point_cov = float(laser_point_cov)
        cfg.filter_size_map_min = float(filter_size_map_min if filter_size_map_min is not None else tree.voxel_size)
        if limit is not None:
            for i in range(23):
                cfg.limit[i] = float(limit[i])
        self.cfg = cfg
        self.h = C.c_void_p()
        _chk(lib().flb_session_create(tree.h, C.byref(cfg), C.byref(self.h)))
        self.n = 0

    def close(self):
        if getattr(self, "h", None):
            lib().flb_session_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def scan_upload(self, body):
        body = _xyz(body)
        _chk(lib().flb_scan_upload(self.h, _p(body), len(body), body.strides[0]))
        self.n = len(body)

    def scan_upload_xyzi(self, body4):
        """feats_down_body with intensity: (n, 4) float32 x, y, z, intensity (travels into the map, laserMapping.cpp:1101-1110)."""
        a = np.ascontiguousarray(body4, np.float32).reshape(-1, 4)
        self.n = len(a)
        _chk(lib().flb_scan_upload_pt(self.h, _p(a), len(a), 16, 12))

    def scan_prefetch_ptr(self, ptr, n, stride):
        """Start the async upload of the NEXT scan (raw host pointer, pinned recommended)."""
        _chk(lib().flb_scan_prefetch(self.h, C.c_void_p(ptr), int(n), int(stride)))
        self._pending_n = int(n)

    def scan_set_device(self, dev_ptr, n):
        _chk(lib().flb_scan_set_device(self.h, C.c_void_p(dev_ptr), int(n)))
        self.n = int(n)

    def h_share_model(self, state26, converge=True):
        st = np.ascontiguousarray(state26, np.float64)
        r = PassResult()
        _chk(lib().flb_pass(self.h, _p(st), 1 if converge else 0, C.byref(r)))
        return {"valid": bool(r.valid), "effct_feat_num": r.effct_feat_num, "total_residual": r.total_residual,
                "HTH": np.array(r.HTH[:]).reshape(12, 12), "HTh": np.array(r.HTh[:])}

    def pass_rows(self):
        cap = max(self.n, 1)
        hx = np.zeros((12, cap), np.float64)  # column-major M x 12 with ld = cap
        h = np.zeros(cap, np.float64)
        M = C.c_int(0)
        _chk(lib().flb_pass_rows(self.h, _p(hx), cap, _p(h), cap, C.byref(M)))
        return hx[:, :M.value].T.copy(), h[:M.value].copy()

    def update_iterated_dyn_share_modified(self, state26, P):
        st = np.array(state26, np.float64).copy()
        Pm = np.ascontiguousarray(np.array(P, np.float64).reshape(23, 23)).copy()
        us = UpdateStats()
        _chk(lib().flb_esikf_update(self.h, _p(st), _p(Pm), C.byref(us)))
        return st, Pm, {f[0]: getattr(us, f[0]) for f in UpdateStats._fields_}

    def map_incremental(self, state26, flg_EKF_inited=True):
        st = np.ascontiguousarray(state26, np.float64)
        a, b = C.c_int(0), C.c_int(0)
        _chk(lib().flb_map_incremental(self.h, _p(st), 1 if flg_EKF_inited else 0, C.byref(a), C.byref(b)))
        return a.value, b.value

    def neighbors(self):
        n = self.n
        nbr = np.empty((n, 5, 3), np.float32)
        d2 = np.empty((n, 5), np.float32)
        cnt = np.empty(n, np.int32)
        sel = np.empty(n, np.uint8)
        nv = np.empty((n, 4), np.float32)
        world = np.empty((n, 3), np.float32)
        _chk(lib().flb_neighbors_download(self.h, _p(nbr), _p(d2), _p(cnt), _p(sel), _p(nv), _p(world)))
        return {"nbr": nbr, "d2": d2, "cnt": cnt, "sel": sel, "normvec": nv, "world": world}

    def scan_step(self, fov, body, state26, P, flg_EKF_inited=True):
        st = np.array(state26, np.float64).copy()
        Pm = np.ascontiguousarray(np.array(P, np.float64).reshape(23, 23)).copy()
        r = ScanResult()
        if body is not None:
            body = _xyz(body)
            self.n = len(body)
            _chk(lib().flb_scan_step(self.h, C.byref(fov) if fov is not None else None, _p(body), len(body),
                                     body.strides[0], _p(st), _p(Pm), 1 if flg_EKF_inited else 0, C.byref(r)))
        else:
            _chk(lib().flb_scan_step(self.h, C.byref(fov) if fov is not None else None, None, 0, 0, _p(st), _p(Pm),
                                     1 if flg_EKF_inited else 0, C.byref(r)))
        return st, Pm, r

    def scan_step_ptr(self, fov, ptr, n, stride, state26, P, flg_EKF_inited=True):
        """flb_scan_step on a raw host pointer (e.g. pinned memory owned by the caller); state26/P updated in place."""
        r = ScanResult()
        if ptr:
            self.n = int(n)
        elif getattr(self, "_pending_n", None) is not None:
            self.n, self._pending_n = self._pending_n, None
        _chk(lib().flb_scan_step(self.h, C.byref(fov) if fov is not None else None, C.c_void_p(ptr) if ptr else None,
                                 int(n), int(stride), _p(state26), _p(P), 1 if flg_EKF_inited else 0, C.byref(r)))
        return r

    def set_update_engine(self, device_driven=True):
        _chk(lib().flb_session_set_update_engine(self.h, 1 if device_driven else 0))

    def scan_step_begin(self, fov, state26, P, flg_EKF_inited=True):
        """Enqueue the step for the scan made current by scan_upload / scan_set_device / scan_prefetch_ptr."""
        if getattr(self, "_pending_n", None) is not None:
            self.n, self._pending_n = self._pending_n, None
        _chk(lib().flb_scan_step_begin(self.h, C.byref(fov) if fov is not None else None, None, 0, 0, _p(state26), _p(P),
                                       1 if flg_EKF_inited else 0))

    def scan_step_finish(self, fov, state26, P):
        r = ScanResult()
        _chk(lib().flb_scan_step_finish(self.h, C.byref(fov) if fov is not None else None, _p(state26), _p(P), C.byref(r)))
        return r

    def stream_ptr(self):
        return lib().flb_session_stream(self.h)

    def sync(self):
        _chk(lib().flb_session_sync(self.h))


POINT_STRIDE = 48      # pcl::PointXYZINormal (PointType, common_lib.h:161)
OFF_INTENSITY = 32
OFF_CURVATURE = 36


def pack_pointtype(xyz, intensity=None, curvature=None):
    """Host buffer of n reference PointType records (48 B: x,y,z,_, nx,ny,nz,_, intensity,curvature,_,_)."""
    xyz = np.asarray(xyz, np.float32)
    buf = np.zeros((len(xyz), 12), np.float32)
    buf[:, 0:3] = xyz[:, :3]
    if intensity is not None:
        buf[:, 8] = intensity
    if curvature is not None:
        buf[:, 9] = curvature
    return buf


LIDAR_LIVOX, LIDAR_VELO16, LIDAR_OUST64 = 1, 2, 3   # preprocess.h LID_TYPE
# The driver records each handler reads (preprocess.h: velodyne_ros::Point, ouster_ros::Point; livox_ros_driver
# CustomPoint), with the C++ layouts of those structs.
VELODYNE_RECORD = np.dtype({"names": ["x", "y", "z", "intensity", "time", "ring"],
                            "formats": ["<f4", "<f4", "<f4", "<f4", "<f4", "<u2"], "offsets": [0, 4, 8, 16, 20, 24], "itemsize": 32})
OUSTER_RECORD = np.dtype({"names": ["x", "y", "z", "intensity", "t", "reflectivity", "ring", "ambient", "range"],
                          "formats": ["<f4", "<f4", "<f4", "<f4", "<u4", "<u2", "u1", "<u2", "<u4"],
                          "offsets": [0, 4, 8, 16, 20, 24, 26, 28, 32], "itemsize": 48})
LIVOX_RECORD = np.dtype({"names": ["offset_time", "x", "y", "z", "reflectivity", "tag", "line"],
                         "formats": ["<u4", "<f4", "<f4", "<f4", "u1", "u1", "u1"], "offsets": [0, 4, 8, 12, 16, 17, 18],
                         "itemsize": 20})
# field names per lidar type: (intensity, time, ring, tag, line)
_PP_FIELDS = {LIDAR_VELO16: ("intensity", "time", "ring", None, None), LIDAR_OUST64: ("intensity", "t", None, None, None),
              LIDAR_LIVOX: ("reflectivity", "offset_time", None, "tag", "line")}


def raw_layout(dtype, lidar_type):
    """flb_raw_layout of a structured dtype, by field name; missing fields are -1."""
    off = lambda name: dtype.fields[name][1] if name and name in dtype.fields else -1
    fi, ft, fr, fg, fl = _PP_FIELDS.get(int(lidar_type), (None,) * 5)
    return RawLayout(dtype.itemsize, off("x"), off("y"), off("z"), off(fi), off(ft), off(fr), off(fg), off(fl))


class FrontEnd:
    """Device front end of one session: meas.lidar -> UndistortPcl -> VoxelGrid -> feats_down_body (SURVEY.md §8f)."""

    def __init__(self, session, max_raw_points=262144):
        self.session = session
        self.cap = int(max_raw_points)
        self.h = C.c_void_p()
        _chk(lib().flb_frontend_create(session.h, self.cap, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            lib().flb_frontend_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, points48):
        """points48: (n,12) float32 PointType records (see pack_pointtype)."""
        b = np.ascontiguousarray(points48, np.float32)
        assert b.ndim == 2 and b.shape[1] == 12
        _chk(lib().flb_frontend_upload(self.h, _p(b), len(b), POINT_STRIDE, OFF_INTENSITY, OFF_CURVATURE))
        self.n_raw = len(b)

    def upload_ptr(self, ptr, n, stride=POINT_STRIDE, off_i=OFF_INTENSITY, off_c=OFF_CURVATURE):
        _chk(lib().flb_frontend_upload(self.h, C.c_void_p(ptr), int(n), stride, off_i, off_c))
        self.n_raw = int(n)

    def preprocess(self, records, lidar_type, n_scans=16, scan_rate=10, point_filter_num=1, time_unit=2, blind=0.01,
                   feature_enabled=0, layout=None):
        """Preprocess::process on the device: records is a numpy structured array of driver records (e.g. VELODYNE_RECORD,
        OUSTER_RECORD, LIVOX_RECORD); the field layout is taken from its dtype by name unless `layout` is given.
        Returns (n_out, last_curvature); the front end then holds meas.lidar as after upload()."""
        rec = np.ascontiguousarray(records)
        lay = layout if layout is not None else raw_layout(rec.dtype, lidar_type)
        cfg = PreprocessCfg(int(lidar_type), int(n_scans), int(scan_rate), int(point_filter_num), int(time_unit), float(blind),
                            int(feature_enabled))
        n = C.c_int(0)
        last = C.c_float(0.0)
        _chk(lib().flb_frontend_preprocess(self.h, rec.ctypes.data if len(rec) else None, len(rec), C.byref(lay), C.byref(cfg),
                                           C.byref(n), C.byref(last)))
        self.n_raw = n.value
        return n.value, last.value

    def undistort(self, imu_poses, state26_end):
        poses = np.ascontiguousarray(imu_poses, np.float64).reshape(-1, 22)
        st = np.ascontiguousarray(state26_end, np.float64)
        _chk(lib().flb_frontend_undistort(self.h, _p(poses), len(poses), _p(st)))

    def voxel_filter(self, leaf):
        n = C.c_int(0)
        _chk(lib().flb_frontend_voxel_filter(self.h, float(leaf), C.byref(n)))
        self.session.n = n.value
        return n.value

    def process_ptr(self, ptr, n, imu_poses, state26_end, leaf, stride=POINT_STRIDE, off_i=OFF_INTENSITY, off_c=OFF_CURVATURE):
        """flb_frontend_process on a raw host pointer; imu_poses must already be a C-contiguous (k,22) float64 array."""
        cnt = C.c_int(0)
        _chk(lib().flb_frontend_process(self.h, C.c_void_p(ptr), int(n), stride, off_i, off_c, _p(imu_poses), len(imu_poses),
                                        _p(state26_end), float(leaf), C.byref(cnt)))
        self.n_raw = int(n)
        self.session.n = cnt.value
        return cnt.value

    def download_undistorted(self):
        n = self.n_raw
        xyzi = np.empty((max(n, 1), 4), np.float32)
        cur = np.empty(max(n, 1), np.float32)
        perm = np.empty(max(n, 1), np.int32)
        cnt = C.c_int(0)
        _chk(lib().flb_frontend_download_undistorted(self.h, _p(xyzi), _p(cur), _p(perm), n, C.byref(cnt)))
        return xyzi[:n], cur[:n], perm[:n]

    def download_down(self):
        cnt = C.c_int(0)
        _chk(lib().flb_frontend_download_down(self.h, None, None, 0, C.byref(cnt)))
        n = cnt.value
        xyzi = np.empty((max(n, 1), 4), np.float32)
        cur = np.empty(max(n, 1), np.float32)
        _chk(lib().flb_frontend_download_down(self.h, _p(xyzi), _p(cur), n, C.byref(cnt)))
        return xyzi[:n], cur[:n]

    def points_to_world(self, which, state26):
        st = np.ascontiguousarray(state26, np.float64)
        cnt = C.c_int(0)
        out = np.empty((self.cap, 4), np.float32)
        _chk(lib().flb_frontend_points_to_world(self.h, int(which), _p(st), _p(out), self.cap, C.byref(cnt)))
        return out[:cnt.value].copy()


def voxel_grid_filter(tree, points48, leaf):
    """pcl::VoxelGrid centroid filter of a host cloud of PointType records -> (m,4) x,y,z,intensity."""
    b = np.ascontiguousarray(points48, np.float32)
    out = np.empty((max(len(b), 1), 4), np.float32)
    n = C.c_int(0)
    _chk(lib().flb_voxel_grid_filter(tree.h, _p(b), len(b), POINT_STRIDE, OFF_INTENSITY, float(leaf), _p(out), len(out), C.byref(n)))
    return out[:n.value].copy()


def reconstruct_keyframes(tree, clouds48, poses6, leaf):
    """recontructIKdTree's data-parallel part: transform + concatenate + VoxelGrid + reconstruct. Returns featsFromMap."""
    clouds = [np.ascontiguousarray(c, np.float32) for c in clouds48]
    k = len(clouds)
    ptrs = (C.c_void_p * max(k, 1))(*[c.ctypes.data for c in clouds])
    sizes = (C.c_int * max(k, 1))(*[len(c) for c in clouds])
    p6 = np.ascontiguousarray(poses6, np.float32).reshape(-1, 6)
    total = sum(len(c) for c in clouds)
    out = np.empty((max(total, 1), 4), np.float32)
    n = C.c_int(0)
    _chk(lib().flb_map_reconstruct_keyframes(tree.h, ptrs, sizes, k, POINT_STRIDE, OFF_INTENSITY, _p(p6), float(leaf), _p(out),
                                             len(out), C.byref(n)))
    return out[:n.value].copy()


def make_fov(cube_len=200.0, det_range=100.0):
    f = FovState()
    f.cube_len = float(cube_len)
    f.det_range = float(det_range)
    f.initialized = 0
    return f


def fov_segment(tree, fov, pos_lid):
    boxes = np.zeros(18, np.float32)
    nb, nd = C.c_int(0), C.c_int(0)
    p = np.ascontiguousarray(pos_lid, np.float64)
    _chk(lib().flb_fov_segment(tree.h, C.byref(fov), _p(p), _p(boxes), C.byref(nb), C.byref(nd)))
    return boxes.reshape(3, 6)[:nb.value].copy(), nd.value


def device_count():
    return lib().flb_device_count()
