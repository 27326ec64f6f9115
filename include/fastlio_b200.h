/*
 * fastlio_b200.h — C ABI of the B200-native FAST-LIO2 per-scan hot path.
 *
 * This is the drop-in boundary for the path named in BASELINE.json:north_star.  Each entry point states the
 * reference interface it replaces (paths relative to the reference repo Yixin-F/better_fastlio2):
 *
 *   map object       KD_TREE<PointType> ikdtree            include/ikd-Tree/ikd_Tree.h:225-249, src/laserMapping.cpp:116
 *   measurement pass h_share_model(state_ikfom&, dyn_share_datastruct<double>&)      src/laserMapping.cpp:1876-2004
 *   filter update    esekf::update_iterated_dyn_share_modified(R, solve_time)
 *                                                          include/IKFoM_toolkit/esekfom/esekfom.hpp:1620-1938
 *   map insert       map_incremental()                     src/laserMapping.cpp:1440-1496
 *   map delete       lasermap_fov_segment()                src/laserMapping.cpp:1136-1200
 *
 * Conventions
 *   - Plain pointers and sizes only; no C++/torch types.  All functions return 0 on success, non-zero on error
 *     (never throw); flb_last_error() returns a thread-local message.  The reference has no error codes on this
 *     path (SURVEY.md §8b) — the C++ facades in include/fastlio_b200/ map errors to valid=false / ROS_ERROR.
 *   - Points are float xyz with a caller-given byte stride (12 for packed xyz, 16 for float4, 48 for
 *     pcl::PointXYZINormal as used by PointType, common_lib.h:161).  Input buffers are borrowed for the call.
 *   - All *host* pointers unless the name says "_dev".  Calls on one handle must be serialised by the caller (the
 *     reference issues all map/search calls from the main thread); different handles are independent.
 *   - There is NO CPU fallback: every compute entry point fails loudly if no CUDA device is usable.
 *
 * State layout "state26" (doubles), mirrors state_ikfom (include/use-ikfom.hpp:21-30):
 *   [0:3) pos | [3:7) rot quaternion (x,y,z,w = Eigen coeffs order) | [7:11) offset_R_L_I (x,y,z,w) |
 *   [11:14) offset_T_L_I | [14:17) vel | [17:20) bg | [20:23) ba | [23:26) grav (S2, |g| = 9.809)
 * Covariance: 23x23 doubles, row-major, error-state order pos,rot,offR,offT,vel,bg,ba,grav(2).
 */
#ifndef FASTLIO_B200_H_
#define FASTLIO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLB_NUM_MATCH_POINTS 5 /* NUM_MATCH_POINTS, include/common_lib.h:149 */
#define FLB_STATE_DIM 26
#define FLB_STATE_DOF 23

typedef struct flb_map flb_map;         /* device hashed-voxel map; replaces KD_TREE<PointType> */
typedef struct flb_session flb_session; /* per-scan measurement context; replaces h_share_model's file-scope globals */

/* ------------------------------------------------------------------------------------------------ errors / device */
const char* flb_last_error(void);
int flb_device_count(void);          /* number of CUDA devices visible (0 => every compute call fails) */
const char* flb_version(void);

/* ------------------------------------------------------------------------------------------------ map (KD_TREE API) */
typedef struct flb_map_config {
  float voxel_size;        /* downsample_size / filter_size_map_min (KD_TREE ctor box_length, ikd_Tree.h:226) */
  int max_points;          /* capacity in points (valid + overflow chains); 0 -> 8M */
  int max_blocks;          /* capacity in 4x4x4-voxel blocks; 0 -> max_points/4 */
  int device;              /* CUDA device ordinal */
} flb_map_config;

int flb_map_create(const flb_map_config* cfg, flb_map** out);     /* KD_TREE::KD_TREE, ikd_Tree.cpp:9-17 */
void flb_map_destroy(flb_map* m);                                 /* KD_TREE::~KD_TREE, ikd_Tree.cpp:19-27 */
int flb_map_set_downsample_param(flb_map* m, float voxel_size);   /* set_downsample_param, ikd_Tree.cpp:39-42
                                                                     (only legal while the map is empty) */
int flb_map_has_root(const flb_map* m);                           /* Root_Node != nullptr test, laserMapping.cpp:2328 */

/* Build (ikd_Tree.cpp:352-364): replace contents by the cloud, inserted verbatim (no per-voxel dedupe). */
int flb_map_build(flb_map* m, const float* xyz, int n, int stride_bytes);
/* reconstruct (ikd_Tree.cpp:1393-1405): delete everything then Build. */
int flb_map_reconstruct(flb_map* m, const float* xyz, int n, int stride_bytes);
/* Add_Points (ikd_Tree.cpp:413-489). downsample_on!=0: per-voxel winner = closest to the voxel centre (sequential
 * semantics of the reference reproduced for the resulting map).  *n_added = number of voxels whose content changed
 * (the reference returns the number of sequential add operations, which its caller overwrites without reading,
 * laserMapping.cpp:1492-1494; the two differ only when several new points fall into one voxel). */
int flb_map_add_points(flb_map* m, const float* xyz, int n, int stride_bytes, int downsample_on, int* n_added);
/* PointType-aware variants.  The reference tree stores whole pcl::PointXYZINormal records (ikd_Tree.h:64-86) and hands them
 * back from Nearest_Search / flatten (featsFromMap for publishing and saving, laserMapping.cpp:2361-2367); FAST-LIO map
 * points carry x, y, z, intensity (normals and curvature are zero, laserMapping.cpp:1101-1110).  These entry points read the
 * intensity at off_intensity bytes into each record (< 0: none -> 0) and keep it with the map point; the plain xyz entry
 * points above store intensity 0, except that 16-byte records are always taken as (x, y, z, intensity). */
int flb_map_build_pt(flb_map* m, const void* pts, int n, int stride_bytes, int off_intensity);
int flb_map_reconstruct_pt(flb_map* m, const void* pts, int n, int stride_bytes, int off_intensity);
int flb_map_add_points_pt(flb_map* m, const void* pts, int n, int stride_bytes, int off_intensity, int downsample_on, int* n_added);
/* Delete_Point_Boxes (ikd_Tree.cpp:535-556): boxes = nb x {min xyz, max xyz} (BoxPointType, ikd_Tree.h:32-35),
 * half-open test min <= p < max (ikd_Tree.cpp:670); *n_deleted = number of points removed. */
int flb_map_delete_boxes(flb_map* m, const float* boxes6, int nb, int* n_deleted);
/* Delete_Points (ikd_Tree.cpp:513-533): remove points equal to the given ones within 1e-6 per axis (same_point). */
int flb_map_delete_points(flb_map* m, const float* xyz, int n, int stride_bytes, int* n_deleted);
/* Nearest_Search (ikd_Tree.cpp:366-397), batched over nq queries: exact k-NN (k <= 5 on the fast path, <= 20
 * otherwise) among valid points with float squared distances, ascending; max_dist <= 0 means unbounded (the
 * reference default INFINITY).  out_xyz[nq*k*3], out_d2[nq*k] (unfilled = NaN / INF), out_cnt[nq]. */
int flb_map_nearest_search(flb_map* m, const float* q_xyz, int nq, int stride_bytes, int k, float max_dist,
                           float* out_xyz, float* out_d2, int* out_cnt);
/* Box_Search (ikd_Tree.cpp:399-404) / Radius_Search (:406-411): points in a half-open box / within radius.
 * Writes up to cap points; *n_found is the total. */
int flb_map_box_search(flb_map* m, const float* box6, float* out_xyz, int cap, int* n_found);
int flb_map_radius_search(flb_map* m, const float* center_xyz, float radius, float* out_xyz, int cap, int* n_found);
/* the same searches returning (x, y, z, intensity) records: out_xyzi[nq*k*4] resp. out_xyzi[cap*4] */
int flb_map_nearest_search_xyzi(flb_map* m, const float* q_xyz, int nq, int stride_bytes, int k, float max_dist,
                                float* out_xyzi, float* out_d2, int* out_cnt);
int flb_map_box_search_xyzi(flb_map* m, const float* box6, float* out_xyzi, int cap, int* n_found);
int flb_map_radius_search_xyzi(flb_map* m, const float* center_xyz, float radius, float* out_xyzi, int cap, int* n_found);
int flb_map_validnum(flb_map* m);  /* validnum(), ikd_Tree.cpp:128-145 ; -1 on error */
int flb_map_size(flb_map* m);      /* size(), ikd_Tree.cpp:78-96 (== validnum here: no lazy tombstones) */
/* flatten (ikd_Tree.cpp:1325-1352): all valid points, arbitrary order. Writes up to cap; *n = total valid. */
int flb_map_flatten(flb_map* m, float* out_xyz, int cap, int* n);
int flb_map_flatten_xyzi(flb_map* m, float* out_xyzi, int cap, int* n);   /* (x, y, z, intensity) records */
/* tree_range (ikd_Tree.h:245): bounding box of valid points {min xyz, max xyz}. */
int flb_map_range(flb_map* m, float* box6);

typedef struct flb_map_stats {
  int valid_points, blocks_in_use, block_capacity, overflow_in_use, overflow_capacity;
  int hash_capacity, hash_tombstones, coarse_cells, rehash_count;
  size_t device_bytes;
} flb_map_stats;
int flb_map_get_stats(flb_map* m, flb_map_stats* out);

/* Optional per-kernel-class timing with CUDA events on the map's stream (used by bench.py for the roofline figure;
 * no reference counterpart — the reference's own timers are omp_get_wtime marks, laserMapping.cpp:2253-2402). */
enum { FLB_K_TRANSFORM = 0, FLB_K_KNN, FLB_K_RESIDUAL, FLB_K_REDUCE, FLB_K_CLASSIFY, FLB_K_INSERT, FLB_K_DELETE, FLB_K_COUNT = 8 };
typedef struct flb_profile {
  double ms[FLB_K_COUNT];      /* accumulated device time per class */
  int launches[FLB_K_COUNT];   /* kernels launched per class */
  int regions[FLB_K_COUNT];    /* timed regions per class (e.g. one per k-NN pass) */
  long long knn_phase[4];      /* queries resolved by search phase A (5^3 voxel stencil) / B0 (3^3 blocks) /
                                  B (3^3 coarse cells) / C (exhaustive coarse scan) */
  long long knn_head_candidates; /* stencil kernel: occupied stencil voxels visited (one 16-B load each) */
  long long knn_chain_nodes;     /* stencil kernel: overflow-chain nodes visited (voxels holding > 1 point) */
  long long knn_chain_max;       /* largest number of chain nodes visited by a single query */
} flb_profile;
int flb_map_profile_enable(flb_map* m, int on);
int flb_map_profile_read(flb_map* m, flb_profile* out, int reset);

/* ------------------------------------------------------------------------------------------------ session (per scan) */
typedef struct flb_session_config {
  int max_scan_points;      /* capacity N of feats_down_body (the reference caps at 100000, laserMapping.cpp:52) */
  int extrinsic_est_en;     /* mapping/extrinsic_est_en, laserMapping.cpp:44 */
  int max_iterations;       /* NUM_MAX_ITERATIONS (ikdtree/max_iteration), laserMapping.cpp:2064 */
  double laser_point_cov;   /* LASER_POINT_COV, laserMapping.cpp:14 (0.001) */
  double filter_size_map_min; /* ikdtree/filter_size_map_min as the DOUBLE the caller holds, laserMapping.cpp:56 */
  double limit[FLB_STATE_DOF]; /* epsi, laserMapping.cpp:2148-2149 (0.001 each) */
} flb_session_config;

void flb_session_default_config(flb_session_config* cfg);
int flb_session_create(flb_map* m, const flb_session_config* cfg, flb_session** out);
void flb_session_destroy(flb_session* s);

/* feats_down_body (laserMapping.cpp:2322-2325): upload the voxel-downsampled, undistorted scan (LiDAR frame).
 * Resets the per-scan caches (Nearest_Points, point_selected_surf := true, laserMapping.cpp:2131). */
int flb_scan_upload(flb_session* s, const float* body_xyz, int n, int stride_bytes);
/* same for PointType records: the intensity at off_intensity (< 0: none) travels with the point into the map, as
 * pointBodyToWorld copies it (laserMapping.cpp:1101-1110).  16-byte records are (x, y, z, intensity). */
int flb_scan_upload_pt(flb_session* s, const void* body_pts, int n, int stride_bytes, int off_intensity);
/* Asynchronous variant for streaming callers: starts the host->device copy of the NEXT scan on a copy stream into a
 * second buffer and returns immediately, so the transfer overlaps the processing of the current scan.  The scan
 * becomes current at the next flb_scan_step / flb_esikf_update called with body == NULL (which waits for the copy).
 * body_xyz must stay valid (pinned memory recommended) until then; stride 12 or 16 only. */
int flb_scan_prefetch(flb_session* s, const float* body_xyz, int n, int stride_bytes);
/* Same, when the scan already lives in device memory as n float4 (x, y, z, intensity) on the session's device.  The scan is
 * read IN PLACE (no copy; its address travels with the staged inputs of the step): the buffer must stay valid and unmodified
 * until the last call working on this scan (flb_scan_step[_finish], flb_esikf_update, flb_map_incremental, flb_pass...) returned. */
int flb_scan_set_device(flb_session* s, const void* body_xyz4_dev, int n);

typedef struct flb_pass_result {
  int valid;               /* ekfom_data.valid (false when effct_feat_num < 1, laserMapping.cpp:1956-1961) */
  int effct_feat_num;      /* M */
  double total_residual;   /* sum |pd2|, laserMapping.cpp:1951 */
  double HTH[144];         /* h_x^T h_x, 12x12 row-major (esekfom.hpp:1790) */
  double HTh[12];          /* h_x^T h */
} flb_pass_result;

/* One h_share_model call (laserMapping.cpp:1876-2004) for the iterate `state26`; search != 0 == ekfom_data.converge
 * (re-run the 5-NN), else the cached Nearest_Points / point_selected_surf are reused.  Returns the reduced normal
 * equations (boundary B3 of SURVEY.md §8b). */
int flb_pass(flb_session* s, const double* state26, int search, flb_pass_result* out);
/* Exact rows of the last flb_pass (boundary B1): h_x as M x 12 COLUMN-major doubles (Eigen::MatrixXd layout,
 * esekfom.hpp:82) with leading dimension ld >= M, and h[M] (= -pd2, laserMapping.cpp:2001). */
int flb_pass_rows(flb_session* s, double* h_x_colmajor, int ld, double* h, int capacity_rows, int* M);

typedef struct flb_update_stats {
  int passes, search_passes, effct_feat_num, converged_count;
  double total_residual;
  float gpu_ms;            /* device time of all kernels of this update (CUDA events; inside flb_scan_step: %globaltimer span from
                              the sequence's first kernel to just behind its last update kernel) */
} flb_update_stats;

/* update_iterated_dyn_share_modified (esekfom.hpp:1620-1938) with the built-in measurement model: state26 / P23x23
 * hold the propagated state in and the posterior out. */
int flb_esikf_update(flb_session* s, double* state26, double* P, flb_update_stats* stats);

/* Update engine: 1 (default) = device-driven — all passes of the iterated update are enqueued up front and the
 * 23-DOF algebra runs in a device kernel (no host round trip inside a scan); 0 = host-driven — the reference's
 * structure, one synchronisation per pass with the algebra in C++ on the host.  Both give the same result to ~1e-15;
 * the device engine falls back to the host one for the under-determined M < 23 branch (esekfom.hpp:1720-1750). */
int flb_session_set_update_engine(flb_session* s, int device_driven);

/* map_incremental (laserMapping.cpp:1440-1496) with the posterior state: classify every scan point with the cached
 * neighbours, then Add_Points(PointToAdd,true) and Add_Points(PointNoNeedDownsample,false). */
int flb_map_incremental(flb_session* s, const double* state26, int flg_EKF_inited, int* n_to_add, int* n_no_downsample);

/* Debug / parity: the per-scan caches. Any pointer may be NULL. nbr_xyz[N*5*3], nbr_d2[N*5], nbr_cnt[N],
 * selected[N] (point_selected_surf), normvec[N*4] (nx,ny,nz,pd2), world_xyz[N*3] (feats_down_world). */
int flb_neighbors_download(flb_session* s, float* nbr_xyz, float* nbr_d2, int* nbr_cnt, unsigned char* selected,
                           float* normvec, float* world_xyz);

/* ------------------------------------------------------------------------------------------------ fov segment (host) */
typedef struct flb_fov_state {
  float local_map_min[3], local_map_max[3]; /* LocalMap_Points, laserMapping.cpp:1132 */
  int initialized;                          /* Localmap_Initialized, :1133 */
  double cube_len;                          /* mapping/cube_len */
  float det_range;                          /* mapping/det_range (DET_RANGE) */
  double pos_lid[3];                        /* pos_lid, laserMapping.cpp:2383 — LiDAR position of the PREVIOUS
                                               posterior (zero before the first update, as the reference's
                                               zero-initialised global); maintained by flb_scan_step */
} flb_fov_state;
/* lasermap_fov_segment (laserMapping.cpp:1136-1200): moves the local-map cube and deletes the slabs that left it.
 * pos_lid = LiDAR position in world. *n_boxes (<=3) / *n_deleted = kdtree_delete_counter. */
int flb_fov_segment(flb_map* m, flb_fov_state* fov, const double* pos_lid, float* boxes_out18, int* n_boxes,
                    int* n_deleted);

/* ------------------------------------------------------------------------------------------------ whole per-scan step */
typedef struct flb_scan_result {
  flb_update_stats update;
  int n_to_add, n_no_downsample, n_deleted, map_valid;
  float gpu_ms_total;      /* update + insert kernels (+ the on-stream upload and the box deletes when `body` is passed: CUDA
                              events then; otherwise the device-side span of the step's sequence) */
  int kernel_launches;     /* number of kernels launched by this step */
} flb_scan_result;
/* The timed region of SURVEY.md §8d: lasermap_fov_segment -> update_iterated_dyn_share_modified -> map_incremental
 * (laserMapping.cpp:2320, :2380, :2401) for one scan.  body may be NULL if the scan was already set with
 * flb_scan_upload / flb_scan_set_device.  fov may be NULL to skip the fov segment. */
int flb_scan_step(flb_session* s, flb_fov_state* fov, const float* body_xyz, int n, int stride_bytes, double* state26,
                  double* P, int flg_EKF_inited, flb_scan_result* out);

/* The same step split at its single synchronisation point, for streaming callers:
 *   flb_scan_step_begin(...);  flb_scan_prefetch(next scan);  flb_scan_step_finish(...);
 * overlaps the upload of the next scan with the kernels of this one.
 * Replay / batch callers whose next prior does not depend on this posterior may keep TWO steps in flight
 *   begin(k); prefetch(k+1); loop { begin(k+1); finish(k); prefetch(k+2); ... }
 * so that the device never waits for the host between scans (finish always collects the OLDEST step; a third begin is
 * refused).  Results are identical to alternating calls.  Constraints of the two-deep mode: the device-driven engine only; the
 * fov segment of step k+1 sees the lidar position of step k-1; a scan with fewer than 23 effective rows (the explicit-row
 * branch, esekfom.hpp:1720-1750, handled on the host) makes flb_scan_step_finish fail if a younger step is already queued.
 * A live filter (prior k+1 = IMU propagation of posterior k) alternates begin / finish and is unaffected. */
int flb_scan_step_begin(flb_session* s, flb_fov_state* fov, const float* body_xyz, int n, int stride_bytes,
                        const double* state26, const double* P, int flg_EKF_inited);
int flb_scan_step_finish(flb_session* s, flb_fov_state* fov, double* state26, double* P, flb_scan_result* out);

/* ------------------------------------------------------------------------------------------------ front-end rows
 * The callers / data formats either side of the per-scan path (SURVEY.md §8f), so that a raw scan never leaves the
 * GPU between the driver callback and the update:
 *   meas.lidar --UndistortPcl--> feats_undistort --downSizeFilterSurf.filter--> feats_down_body --> flb_scan_step
 * A front end belongs to one session and shares its stream; calls are serialised by the caller like all others.
 * Points are the reference's PointType (pcl::PointXYZINormal, common_lib.h:161): 48-byte stride, x@0 y@4 z@8,
 * intensity@32, curvature@36 (= time offset in ms, preprocess.cpp) — stride and offsets are parameters. */
typedef struct flb_frontend flb_frontend;
#define FLB_IMU_POSE_DOUBLES 22 /* Pose6D (msg/Pose6D.msg, set_pose6d common_lib.h:446-460):
                                   offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9] row-major */
#define FLB_MAX_IMU_POSES 256

int flb_frontend_create(flb_session* s, int max_raw_points, flb_frontend** out);
void flb_frontend_destroy(flb_frontend* f);
/* meas.lidar (IMU_Processing.hpp:242 "pcl_out = *(meas.lidar)"): upload the raw scan. off_intensity / off_curvature are
 * byte offsets of those float fields inside a point, or -1 when absent (treated as 0).  The buffer holds n whole records
 * (n * stride_bytes bytes are copied), as a std::vector<PointType> / pcl::PointCloud does. */
int flb_frontend_upload(flb_frontend* f, const void* pts, int n, int stride_bytes, int off_intensity, int off_curvature);
/* Preprocess::process (src/preprocess.cpp), non-feature branch, on the device: the driver's records -> meas.lidar.
 * Replaces flb_frontend_upload: one copy of n records of layout->stride bytes, then the handler's blind cut,
 * point_filter_num decimation and per-point time offset (curvature, ms) run on the GPU, in input order.
 *   FLB_LIDAR_LIVOX  livox_handler (:178-204): CustomMsg points; x,y,z f32, intensity = reflectivity u8, time =
 *                    offset_time u32 (ns), tag u8, line u8.  Point 0 is never used.
 *   FLB_LIDAR_VELO16 velodyne_handler (:417-473): x,y,z,intensity f32, time f32, ring u16.  When the last point's time
 *                    is not > 0 the times are synthesised per ring from the yaw angle (the first point of each ring is
 *                    dropped) and every ring must be < n_scans.
 *   FLB_LIDAR_OUST64 oust64_handler (:271-297): x,y,z,intensity f32, time = t u32.
 * Offsets of absent fields are -1 (read as 0, as fromROSMsg leaves them); x,y,z are required; f32 / u32 fields must be
 * 4-byte aligned and u16 fields 2-byte aligned inside the record.  *n_out = pl_surf.size() and *last_curvature =
 * pl_surf.back().curvature (0 for an empty cloud), what sync_packages reads.  Afterwards the front end holds the cloud
 * as after flb_frontend_upload of it.  feature_enabled (give_feature) is not supported and is rejected. */
#define FLB_LIDAR_LIVOX 1
#define FLB_LIDAR_VELO16 2
#define FLB_LIDAR_OUST64 3
typedef struct flb_preprocess_cfg {   /* the Preprocess members set at laserMapping.cpp:2034-2041 */
  int lidar_type;        /* FLB_LIDAR_* (preprocess.h LID_TYPE) */
  int n_scans;           /* N_SCANS */
  int scan_rate;         /* SCAN_RATE (Hz), for the synthesised Velodyne times */
  int point_filter_num;  /* keep every point_filter_num-th point, >= 1 */
  int time_unit;         /* 0 s, 1 ms, 2 us, 3 ns (preprocess.h TIME_UNIT; any other value scales by 1) */
  double blind;          /* blind range (m) */
  int feature_enabled;   /* must be 0 */
} flb_preprocess_cfg;
typedef struct flb_raw_layout {   /* byte offsets inside one record of `stride` bytes; -1 = field absent */
  int stride, off_x, off_y, off_z, off_intensity, off_time, off_ring, off_tag, off_line;
} flb_raw_layout;
int flb_frontend_preprocess(flb_frontend* f, const void* records, int n, const flb_raw_layout* layout,
                            const flb_preprocess_cfg* cfg, int* n_out, float* last_curvature);
/* ImuProcess::UndistortPcl, the per-point part (IMU_Processing.hpp:243 sort by time, :334-386 backward compensation).
 * imu_poses = n_poses x 22 doubles = the IMUpose vector built by the forward propagation (:260-322, stays on the host
 * with kf.predict); state26_end = imu_state after the last predict (:329).  Result: feats_undistort in time order
 * (ties keep upload order; the reference's std::sort leaves them unspecified). */
int flb_frontend_undistort(flb_frontend* f, const double* imu_poses, int n_poses, const double* state26_end);
/* downSizeFilterSurf.setInputCloud(feats_undistort); downSizeFilterSurf.filter(*feats_down_body)
 * (laserMapping.cpp:2322-2323, leaf = mappingSurfLeafSize :2135): pcl::VoxelGrid centroid filter (PCL 1.10 semantics:
 * float leaf index relative to the cloud minimum, output ordered by leaf index, centroid of x,y,z,intensity,curvature;
 * PCL's int32 overflow guard returns the input unchanged).  The result becomes the session's current scan
 * (as flb_scan_upload would); *n_out = feats_down_size.  Sums run in time order inside a leaf (PCL: unspecified). */
int flb_frontend_voxel_filter(flb_frontend* f, float leaf_size, int* n_out);
/* The three calls above in one (one synchronisation): raw scan in, feats_down_body left on the device as the session's
 * current scan.  imu_poses == NULL or n_poses == 0 skips the undistortion (no IMU / already compensated). */
int flb_frontend_process(flb_frontend* f, const void* pts, int n, int stride_bytes, int off_intensity, int off_curvature,
                         const double* imu_poses, int n_poses, const double* state26_end, float leaf_size, int* n_out);
/* Read back feats_undistort (x,y,z,intensity per point; curvature; perm[j] = upload index of sorted point j) and
 * feats_down_body.  Any output pointer may be NULL; at most cap points are written, *n = the cloud size. */
int flb_frontend_download_undistorted(flb_frontend* f, float* out_xyzi, float* out_curvature, int* out_perm, int cap, int* n);
int flb_frontend_download_down(flb_frontend* f, float* out_xyzi, float* out_curvature, int cap, int* n);
/* publish_frame_world / map saving (laserMapping.cpp:1502-1540): RGBpointBodyToWorld (:1101-1110) of every point of
 * feats_down_body (which = 0, dense_pub_en false) or feats_undistort (which = 1) with the posterior state. */
int flb_frontend_points_to_world(flb_frontend* f, int which, const double* state26, float* out_xyzi, int cap, int* n);

/* Stand-alone pcl::VoxelGrid centroid filter on a host cloud (the reference's other VoxelGrid call sites, e.g.
 * laserMapping.cpp:640-643, :1780-1789), run on the map's device/stream.  out_xyzi = x,y,z,intensity per point. */
int flb_voxel_grid_filter(flb_map* m, const void* pts, int n, int stride_bytes, int off_intensity, float leaf_size,
                          float* out_xyzi, int cap, int* n_out);
/* recontructIKdTree, the data-parallel part (laserMapping.cpp:632-664): for the selected key frames k (clouds[k] with
 * sizes[k] points in the key frame's own frame, poses6[k] = x,y,z,roll,pitch,yaw of cloudKeyPoses6D) do
 * subMap += transformPointCloud(cloud_k, pose_k) (common_lib.h:711-734), VoxelGrid(leaf), ikdtree.reconstruct(result).
 * The filtered sub-map (featsFromMap, :664) is returned in out_xyzi (up to cap points); *n_points = its size.  The
 * key-frame selection itself (pose radius search, :621-635) is back-end bookkeeping and stays with the caller. */
int flb_map_reconstruct_keyframes(flb_map* m, const void* const* clouds, const int* sizes, int n_keyframes, int stride_bytes,
                                  int off_intensity, const float* poses6, float leaf_size, float* out_xyzi, int cap,
                                  int* n_points);

/* Stream access for callers that overlap work (returns a cudaStream_t as void*). */
void* flb_session_stream(flb_session* s);
int flb_session_sync(flb_session* s);

#ifdef __cplusplus
}
#endif
#endif /* FASTLIO_B200_H_ */
