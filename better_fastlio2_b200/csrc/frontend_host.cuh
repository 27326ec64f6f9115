// frontend_host.cuh — C-ABI entry points of the rows either side of the per-scan path (SURVEY.md §8f ranks 1-4).
// Included at the end of fastlio_b200.cu (uses its flb_map / flb_session definitions and error helpers).
#pragma once
#include "frontend_kernels.cuh"
#include <cub/device/device_radix_sort.cuh>

// ------------------------------------------------------------------------------------------------ voxel-grid workspace
struct VgWork {
  int cap = 0;
  unsigned *keys_a = nullptr, *keys_b = nullptr;
  int *vals_a = nullptr, *vals_b = nullptr, *flags = nullptr, *pos = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
  unsigned* d_mm = nullptr;   // 8 words, see k_vg_init
  unsigned* h_mm = nullptr;   // pinned mirror
};
static void vg_release(VgWork& w) {
  void* ptrs[] = {w.keys_a, w.keys_b, w.vals_a, w.vals_b, w.flags, w.pos, w.tmp, w.d_mm};
  for (void* p : ptrs) if (p) Q(cudaFree(p));
  if (w.h_mm) Q(cudaFreeHost(w.h_mm));
  w = VgWork();
}
static int vg_ensure(VgWork& w, int n) {
  if (n <= w.cap) return 0;
  vg_release(w);
  const int cap = std::max(n, 1 << 12);
  size_t t1 = 0, t2 = 0;
  CU(cub::DeviceRadixSort::SortPairs(nullptr, t1, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr, (int*)nullptr, cap));
  CU(cub::DeviceScan::ExclusiveSum(nullptr, t2, (const int*)nullptr, (int*)nullptr, cap));
  size_t t3 = 0;   // the segmented chain scan of the Velodyne yaw-time preprocess
  CU(cub::DeviceScan::InclusiveScan(nullptr, t3, (const unsigned*)nullptr, (unsigned*)nullptr, flb::PpChainOp(), cap));
  w.tmp_bytes = std::max(std::max(t1, t2), t3) + 256;
  CU(cudaMalloc((void**)&w.keys_a, sizeof(unsigned) * (size_t)cap));
  CU(cudaMalloc((void**)&w.keys_b, sizeof(unsigned) * (size_t)cap));
  CU(cudaMalloc((void**)&w.vals_a, sizeof(int) * (size_t)cap));
  CU(cudaMalloc((void**)&w.vals_b, sizeof(int) * (size_t)cap));
  CU(cudaMalloc((void**)&w.flags, sizeof(int) * (size_t)cap));
  CU(cudaMalloc((void**)&w.pos, sizeof(int) * (size_t)cap));
  CU(cudaMalloc(&w.tmp, w.tmp_bytes));
  CU(cudaMalloc((void**)&w.d_mm, sizeof(unsigned) * 8));
  CU(cudaMallocHost((void**)&w.h_mm, sizeof(unsigned) * 8));
  w.cap = cap;
  return 0;
}

// pcl::VoxelGrid::applyFilter on n device points (x,y,z,intensity [+curvature]) -> out (capacity out_cap points), all on
// `st`.  The output count and PCL's overflow flag are copied to w.h_mm[7] / w.h_mm[6]; valid after the stream drained.
static int vg_enqueue(flb_map* m, VgWork& w, const float4* pts, const float* curv, int n, float leaf, float4* out, float* out_curv,
                      int out_cap, cudaStream_t st) {
  if (vg_ensure(w, n)) return 1;
  const float inv = 1.0f / leaf;   // inverse_leaf_size_
  const int g = grid_for(std::max(n, 1), 256, m->sm_count * 8);
  k_vg_init<<<1, 32, 0, st>>>(w.d_mm);
  m->launches++;
  if (n > 0) {
    k_vg_minmax<<<g, 256, 0, st>>>(pts, n, w.d_mm);
    k_vg_keys<<<g, 256, 0, st>>>(pts, n, inv, w.d_mm, w.keys_a, w.vals_a);
    size_t tb = w.tmp_bytes;
    CU(cub::DeviceRadixSort::SortPairs(w.tmp, tb, (const unsigned*)w.keys_a, w.keys_b, (const int*)w.vals_a, w.vals_b, n, 0, 32, st));
    k_vg_heads<<<g, 256, 0, st>>>(w.keys_b, n, w.flags);
    tb = w.tmp_bytes;
    CU(cub::DeviceScan::ExclusiveSum(w.tmp, tb, (const int*)w.flags, w.pos, n, st));
    k_vg_centroid<<<g, 256, 0, st>>>(pts, curv, w.keys_b, w.vals_b, w.flags, w.pos, n, out, out_curv, out_cap, w.d_mm);
    m->launches += 4 + 6;   // + the radix-sort (histogram, 4 onesweep passes) and scan kernels of CUB
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(w.h_mm, w.d_mm, sizeof(unsigned) * 8, cudaMemcpyDeviceToHost, st));
  return 0;
}

// ------------------------------------------------------------------------------------------------ front end object
struct flb_frontend {
  flb_session* ses = nullptr;
  int cap = 0;
  int n_raw = 0;            // points of the current raw scan (meas.lidar)
  int n_down = -1;          // points of feats_down_body after the last voxel filter (-1: none yet)
  bool sorted = false;      // pts_t holds feats_undistort (time order); else `pts` (upload order) is current
  unsigned char* raw = nullptr;
  size_t raw_cap = 0;
  float4 *pts = nullptr, *pts_t = nullptr;
  float *curv = nullptr, *curv_t = nullptr, *down_curv = nullptr;
  int* perm = nullptr;      // time-sorted position -> upload index
  float4* world = nullptr;  // publish scratch
  double *d_poses = nullptr, *h_poses = nullptr;
  cudaEvent_t ev_poses = nullptr;
  VgWork vg;
  bool holds_ref = false;
  float* pp_t = nullptr;    // preprocess: synthesised Velodyne times by raw index (allocated on first use)
  int* pp_ring = nullptr;   // preprocess: sorted position of each ring's first point, n_scans + 1 entries
  int pp_ring_cap = 0;
};

extern "C" int flb_frontend_create(flb_session* s, int max_raw_points, flb_frontend** out) {
  if (!s || !out) return set_err("flb_frontend_create: null argument");
  if (max_raw_points <= 0) return set_err("max_raw_points must be > 0");
  CU(cudaSetDevice(s->map->cfg.device));
  flb_frontend* f = new (std::nothrow) flb_frontend();
  if (!f) return set_err("out of host memory");
  f->ses = s;
  f->cap = max_raw_points;
  const size_t N = (size_t)max_raw_points;
  cudaError_t e = cudaSuccess;
  auto A = [&](void** p, size_t b) { if (e == cudaSuccess) e = cudaMalloc(p, b); };
  A((void**)&f->pts, sizeof(float4) * N);
  A((void**)&f->pts_t, sizeof(float4) * N);
  A((void**)&f->world, sizeof(float4) * N);
  A((void**)&f->curv, sizeof(float) * N);
  A((void**)&f->curv_t, sizeof(float) * N);
  A((void**)&f->down_curv, sizeof(float) * N);
  A((void**)&f->perm, sizeof(int) * N);
  A((void**)&f->d_poses, sizeof(double) * IMU_POSE_DOUBLES * MAX_IMU_POSES);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&f->h_poses, sizeof(double) * IMU_POSE_DOUBLES * MAX_IMU_POSES);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ev_poses, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    cudaGetLastError();
    flb_frontend_destroy(f);
    return set_err("flb_frontend_create: %s", cudaGetErrorString(e));
  }
  if (vg_ensure(f->vg, max_raw_points)) { flb_frontend_destroy(f); return 1; }
  s->map->refs++;   // keeps the map (and its stream) alive
  f->holds_ref = true;
  *out = f;
  return 0;
}

extern "C" void flb_frontend_destroy(flb_frontend* f) {
  if (!f) return;
  flb_map* m = f->ses ? f->ses->map : nullptr;
  if (m) { Q(cudaSetDevice(m->cfg.device)); Q(cudaStreamSynchronize(m->stream)); }
  void* ptrs[] = {f->raw, f->pts, f->pts_t, f->world, f->curv, f->curv_t, f->down_curv, f->perm, f->d_poses, f->pp_t, f->pp_ring};
  for (void* p : ptrs) if (p) Q(cudaFree(p));
  if (f->h_poses) Q(cudaFreeHost(f->h_poses));
  if (f->ev_poses) Q(cudaEventDestroy(f->ev_poses));
  const bool counted = f->holds_ref;
  vg_release(f->vg);
  delete f;
  if (m && counted) map_release(m);
}

static inline const float4* fe_cloud(const flb_frontend* f) { return f->sorted ? f->pts_t : f->pts; }
static inline const float* fe_curv(const flb_frontend* f) { return f->sorted ? f->curv_t : f->curv; }

extern "C" int flb_frontend_upload(flb_frontend* f, const void* pts, int n, int stride, int off_intensity, int off_curvature) {
  if (!f) return set_err("null front end");
  if (n < 0 || n > f->cap) return set_err("raw scan of %d points exceeds max_raw_points=%d", n, f->cap);
  if (n > 0 && (!pts || stride < 12)) return set_err("bad raw scan buffer");
  if ((off_intensity >= 0 && off_intensity + 4 > stride) || (off_curvature >= 0 && off_curvature + 4 > stride))
    return set_err("field offset outside the point stride");
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  f->n_raw = n;
  f->sorted = false;
  f->n_down = -1;
  if (n == 0) return 0;
  const size_t bytes = (size_t)n * stride;
  if (bytes > f->raw_cap) {
    if (f->raw) cudaFree(f->raw);
    f->raw = nullptr; f->raw_cap = 0;
    const size_t cap = std::max(bytes, (size_t)f->cap * (size_t)stride);   // sized once for the capacity: scans vary in size
    CU(cudaMalloc((void**)&f->raw, cap));
    f->raw_cap = cap;
  }
  CU(cudaMemcpyAsync(f->raw, pts, bytes, cudaMemcpyHostToDevice, m->stream));
  k_pack_xyzic<<<grid_for(n, 256, m->sm_count * 8), 256, 0, m->stream>>>(f->raw, stride, off_intensity, off_curvature, f->pts, f->curv, n);
  m->launches++;
  CU(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------ preprocess
static int pp_check_field(int off, int size, int stride, const char* name) {
  if (off < 0) return 0;
  if (off + size > stride) return set_err("flb_frontend_preprocess: field %s at byte %d lies outside the %d-byte record", name, off, stride);
  if (off % size) return set_err("flb_frontend_preprocess: field %s at byte %d is not %d-byte aligned", name, off, size);
  return 0;
}

extern "C" int flb_frontend_preprocess(flb_frontend* f, const void* records, int n, const flb_raw_layout* layout,
                                       const flb_preprocess_cfg* cfg, int* n_out, float* last_curvature) {
  if (!f || !layout || !cfg) return set_err("flb_frontend_preprocess: null argument");
  if (n < 0 || n > f->cap) return set_err("raw scan of %d points exceeds max_raw_points=%d", n, f->cap);
  if (n > 0 && !records) return set_err("flb_frontend_preprocess: null records");
  const int lt = cfg->lidar_type;
  if (lt != FLB_LIDAR_LIVOX && lt != FLB_LIDAR_VELO16 && lt != FLB_LIDAR_OUST64)
    return set_err("flb_frontend_preprocess: unsupported lidar_type %d (1 LIVOX, 2 VELO16, 3 OUST64)", lt);
  if (cfg->feature_enabled) return set_err("flb_frontend_preprocess: feature extraction (feature_enabled) is not supported");
  if (cfg->point_filter_num < 1) return set_err("point_filter_num must be >= 1 (got %d)", cfg->point_filter_num);
  if (cfg->n_scans < 1 || cfg->n_scans > 65535) return set_err("n_scans must be in [1, 65535] (got %d)", cfg->n_scans);
  if (lt == FLB_LIDAR_VELO16 && cfg->scan_rate < 1) return set_err("scan_rate must be >= 1 (got %d)", cfg->scan_rate);
  const flb_raw_layout& L = *layout;
  if (L.stride < 1) return set_err("flb_frontend_preprocess: bad record stride %d", L.stride);
  if (L.off_x < 0 || L.off_y < 0 || L.off_z < 0) return set_err("flb_frontend_preprocess: the x, y and z fields are required");
  const bool livox = lt == FLB_LIDAR_LIVOX;
  if (pp_check_field(L.off_x, 4, L.stride, "x") || pp_check_field(L.off_y, 4, L.stride, "y") || pp_check_field(L.off_z, 4, L.stride, "z") ||
      pp_check_field(L.off_intensity, livox ? 1 : 4, L.stride, livox ? "reflectivity" : "intensity") ||
      pp_check_field(L.off_time, 4, L.stride, livox ? "offset_time" : "time") ||
      (lt == FLB_LIDAR_VELO16 && pp_check_field(L.off_ring, 2, L.stride, "ring")) ||
      (livox && (pp_check_field(L.off_tag, 1, L.stride, "tag") || pp_check_field(L.off_line, 1, L.stride, "line"))))
    return 1;
  if (L.stride % 4) return set_err("flb_frontend_preprocess: record stride %d is not a multiple of 4", L.stride);
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  f->n_raw = 0;
  f->sorted = false;
  f->n_down = -1;
  if (n_out) *n_out = 0;
  if (last_curvature) *last_curvature = 0.f;
  // velodyne_handler returns at once on an empty cloud; the others produce nothing from it either
  if (n == 0) return 0;
  cudaStream_t st = m->stream;
  const size_t bytes = (size_t)n * L.stride;
  if (bytes > f->raw_cap) {
    if (f->raw) Q(cudaFree(f->raw));
    f->raw = nullptr; f->raw_cap = 0;
    const size_t cap = std::max(bytes, (size_t)f->cap * (size_t)L.stride);
    CU(cudaMalloc((void**)&f->raw, cap));
    f->raw_cap = cap;
  }
  CU(cudaMemcpyAsync(f->raw, records, bytes, cudaMemcpyHostToDevice, st));

  PpArgs a;
  a.rec = f->raw;
  a.stride = L.stride; a.off_x = L.off_x; a.off_y = L.off_y; a.off_z = L.off_z; a.off_i = L.off_intensity; a.off_t = L.off_time;
  a.off_ring = L.off_ring; a.off_tag = L.off_tag; a.off_line = L.off_line;
  a.n = n; a.n_scans = cfg->n_scans; a.pfn = cfg->point_filter_num;
  const int tu = cfg->time_unit;
  a.time_scale = tu == 0 ? 1.e3f : tu == 1 ? 1.f : tu == 2 ? 1.e-3f : tu == 3 ? 1.e-6f : 1.f;
  a.blind2 = cfg->blind * cfg->blind;
  a.omega = 0.361 * cfg->scan_rate;
  int mode = lt == FLB_LIDAR_OUST64 ? PP_OUSTER : livox ? PP_LIVOX : PP_VELO_TIME;
  if (mode == PP_VELO_TIME) {   // given_offset_time is decided by the last point (:322)
    float t_last = 0.f;
    if (L.off_time >= 0) memcpy(&t_last, (const unsigned char*)records + (size_t)(n - 1) * L.stride + L.off_time, sizeof(float));
    if (!(t_last > 0.f)) mode = PP_VELO_YAW;
  }

  VgWork& w = f->vg;
  const int g = grid_for(n, 256, m->sm_count * 8);
  int* keep = w.flags;
  int* pos = w.pos;
  k_vg_init<<<1, 32, 0, st>>>(w.d_mm);   // d_mm[2] = first raw index with ring >= n_scans (none: 0xFFFFFFFF)
  m->launches++;
  size_t tb = w.tmp_bytes;
  if (mode == PP_VELO_YAW) {
    if (!f->pp_t) CU(cudaMalloc((void**)&f->pp_t, sizeof(float) * (size_t)f->cap));
    if (cfg->n_scans + 1 > f->pp_ring_cap) {
      if (f->pp_ring) Q(cudaFree(f->pp_ring));
      f->pp_ring = nullptr; f->pp_ring_cap = 0;
      CU(cudaMalloc((void**)&f->pp_ring, sizeof(int) * (size_t)(cfg->n_scans + 1)));
      f->pp_ring_cap = cfg->n_scans + 1;
    }
    int bits = 1;
    while ((1u << bits) <= (unsigned)cfg->n_scans) ++bits;
    float* c0 = f->curv_t;   // scratch: undistort rewrites it before anything reads it
    k_pp_ring_keys<<<g, 256, 0, st>>>(a, w.keys_a, w.vals_a, w.d_mm);
    CU(cub::DeviceRadixSort::SortPairs(w.tmp, tb, (const unsigned*)w.keys_a, w.keys_b, (const int*)w.vals_a, w.vals_b, n, 0, bits, st));
    k_pp_ring_start<<<g, 256, 0, st>>>(w.keys_b, n, f->pp_ring);
    k_pp_yaw_c0<<<g, 256, 0, st>>>(a, w.keys_b, w.vals_b, f->pp_ring, c0);
    k_pp_yaw_codes<<<g, 256, 0, st>>>(w.keys_b, f->pp_ring, c0, n, a.omega, w.keys_a);
    tb = w.tmp_bytes;
    CU(cub::DeviceScan::InclusiveScan(w.tmp, tb, (const unsigned*)w.keys_a, (unsigned*)pos, flb::PpChainOp(), n, st));
    k_pp_yaw_apply<<<g, 256, 0, st>>>(w.vals_b, c0, (const unsigned*)pos, n, a.omega, f->pp_t);
    k_pp_keep<PP_VELO_YAW><<<g, 256, 0, st>>>(a, f->pp_ring, w.vals_b, keep);
    m->launches += 6 + 5 + 1;   // + the radix-sort and scan kernels of CUB
  } else if (mode == PP_LIVOX) {
    int* valid = (int*)w.keys_a;
    int* valid_excl = (int*)w.keys_b;
    k_pp_livox_valid<<<g, 256, 0, st>>>(a, valid);
    CU(cub::DeviceScan::ExclusiveSum(w.tmp, tb, (const int*)valid, valid_excl, n, st));
    k_pp_keep<PP_LIVOX><<<g, 256, 0, st>>>(a, valid, valid_excl, keep);
    m->launches += 2 + 1;
  } else if (mode == PP_OUSTER) {
    k_pp_keep<PP_OUSTER><<<g, 256, 0, st>>>(a, nullptr, nullptr, keep);
    m->launches++;
  } else {
    k_pp_keep<PP_VELO_TIME><<<g, 256, 0, st>>>(a, nullptr, nullptr, keep);
    m->launches++;
  }
  tb = w.tmp_bytes;
  CU(cub::DeviceScan::ExclusiveSum(w.tmp, tb, (const int*)keep, pos, n, st));
  switch (mode) {
    case PP_OUSTER: k_pp_scatter<PP_OUSTER><<<g, 256, 0, st>>>(a, keep, pos, nullptr, f->pts, f->curv, w.d_mm); break;
    case PP_VELO_TIME: k_pp_scatter<PP_VELO_TIME><<<g, 256, 0, st>>>(a, keep, pos, nullptr, f->pts, f->curv, w.d_mm); break;
    case PP_VELO_YAW: k_pp_scatter<PP_VELO_YAW><<<g, 256, 0, st>>>(a, keep, pos, f->pp_t, f->pts, f->curv, w.d_mm); break;
    default: k_pp_scatter<PP_LIVOX><<<g, 256, 0, st>>>(a, keep, pos, nullptr, f->pts, f->curv, w.d_mm); break;
  }
  k_pp_last<<<1, 1, 0, st>>>(f->curv, w.d_mm);
  m->launches += 1 + 2;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(w.h_mm, w.d_mm, sizeof(unsigned) * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (mode == PP_VELO_YAW && w.h_mm[2] != 0xFFFFFFFFu) {
    const unsigned i = w.h_mm[2];
    unsigned short ring = 0;
    memcpy(&ring, (const unsigned char*)records + (size_t)i * L.stride + L.off_ring, sizeof(ring));
    return set_err("flb_frontend_preprocess: point %u has ring %u >= n_scans=%d (times are synthesised per ring)", i, (unsigned)ring,
                   cfg->n_scans);
  }
  f->n_raw = (int)w.h_mm[0];
  if (n_out) *n_out = f->n_raw;
  if (last_curvature) memcpy(last_curvature, &w.h_mm[1], sizeof(float));
  return 0;
}

extern "C" int flb_frontend_undistort(flb_frontend* f, const double* imu_poses22, int n_poses, const double* state26_end) {
  if (!f) return set_err("null front end");
  if (!imu_poses22 || !state26_end) return set_err("flb_frontend_undistort: null argument");
  if (n_poses < 1 || n_poses > MAX_IMU_POSES) return set_err("n_poses must be in [1, %d]", MAX_IMU_POSES);
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  const int n = f->n_raw;
  if (n == 0) { f->sorted = true; return 0; }
  cudaStream_t st = m->stream;
  // pinned staging (a pageable cudaMemcpyAsync measured ~7 ms per call here); the event guards its reuse
  CU(cudaEventSynchronize(f->ev_poses));
  memcpy(f->h_poses, imu_poses22, sizeof(double) * IMU_POSE_DOUBLES * (size_t)n_poses);
  CU(cudaMemcpyAsync(f->d_poses, f->h_poses, sizeof(double) * IMU_POSE_DOUBLES * (size_t)n_poses, cudaMemcpyHostToDevice, st));
  CU(cudaEventRecord(f->ev_poses, st));
  const int g = grid_for(n, 256, m->sm_count * 8);
  // sort(pcl_out.points.begin(), pcl_out.points.end(), time_list)  (IMU_Processing.hpp:243) — stable here
  k_time_keys<<<g, 256, 0, st>>>(f->curv, f->vg.keys_a, f->vg.vals_a, n);
  size_t tb = f->vg.tmp_bytes;
  CU(cub::DeviceRadixSort::SortPairs(f->vg.tmp, tb, (const unsigned*)f->vg.keys_a, f->vg.keys_b, (const int*)f->vg.vals_a, f->perm, n, 0, 32, st));
  UndistortEnd e;
  for (int k = 0; k < 4; ++k) { e.rot[k] = state26_end[3 + k]; e.offR[k] = state26_end[7 + k]; }
  for (int k = 0; k < 3; ++k) { e.pos[k] = state26_end[k]; e.offT[k] = state26_end[11 + k]; }
  k_undistort<<<g, 256, sizeof(double) * IMU_POSE_DOUBLES * (size_t)n_poses, st>>>(f->pts, f->curv, f->perm, n, f->d_poses, n_poses, e,
                                                                                  f->pts_t, f->curv_t);
  m->launches += 2 + 5;
  CU(cudaGetLastError());
  f->sorted = true;
  return 0;
}

extern "C" int flb_frontend_voxel_filter(flb_frontend* f, float leaf, int* n_out) {
  if (!f) return set_err("null front end");
  if (!(leaf > 0.f)) return set_err("leaf size must be > 0");
  flb_session* s = f->ses;
  flb_map* m = s->map;
  CU(cudaSetDevice(m->cfg.device));
  if (s->pending_n >= 0) return set_err("flb_frontend_voxel_filter: a prefetched scan is pending on this session");
  const int n = f->n_raw;
  // the centroids are written straight into the session's feats_down_body buffer
  if (vg_enqueue(m, f->vg, fe_cloud(f), fe_curv(f), n, leaf, s->body, f->down_curv, s->cap, m->stream)) return 1;
  CU(cudaStreamSynchronize(m->stream));
  int nd = (int)f->vg.h_mm[7];
  if (f->vg.h_mm[6]) {
    // PCL: "Leaf size is too small for the input dataset. Integer indices would overflow." -> output = input
    if (n > s->cap) return set_err("voxel filter overflow guard: unfiltered scan of %d points exceeds max_scan_points=%d", n, s->cap);
    CU(cudaMemcpyAsync(s->body, fe_cloud(f), sizeof(float4) * (size_t)n, cudaMemcpyDeviceToDevice, m->stream));
    CU(cudaMemcpyAsync(f->down_curv, fe_curv(f), sizeof(float) * (size_t)n, cudaMemcpyDeviceToDevice, m->stream));
    nd = n;
  }
  if (nd > s->cap) return set_err("filtered scan of %d points exceeds max_scan_points=%d", nd, s->cap);
  f->n_down = nd;
  if (n_out) *n_out = nd;
  return scan_reset(s, nd);
}

// upload + undistort + voxel filter in one call (one synchronisation): meas.lidar -> feats_down_body on the device
extern "C" int flb_frontend_process(flb_frontend* f, const void* pts, int n, int stride, int off_intensity, int off_curvature,
                                    const double* imu_poses22, int n_poses, const double* state26_end, float leaf, int* n_out) {
  if (flb_frontend_upload(f, pts, n, stride, off_intensity, off_curvature)) return 1;
  if (imu_poses22 && n_poses > 0 && flb_frontend_undistort(f, imu_poses22, n_poses, state26_end)) return 1;
  return flb_frontend_voxel_filter(f, leaf, n_out);
}

static int fe_download(flb_map* m, const float4* src, const float* src_curv, int n, float* out_xyzi, float* out_curv, int cap) {
  const int c = std::min(n, cap);
  if (c > 0 && out_xyzi) CU(cudaMemcpyAsync(out_xyzi, src, sizeof(float4) * (size_t)c, cudaMemcpyDeviceToHost, m->stream));
  if (c > 0 && out_curv && src_curv) CU(cudaMemcpyAsync(out_curv, src_curv, sizeof(float) * (size_t)c, cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return 0;
}

extern "C" int flb_frontend_download_undistorted(flb_frontend* f, float* out_xyzi, float* out_curv, int* out_perm, int cap, int* n) {
  if (!f) return set_err("null front end");
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  if (n) *n = f->n_raw;
  const int c = std::min(f->n_raw, cap);
  if (c > 0 && out_perm) {
    if (f->sorted) CU(cudaMemcpyAsync(out_perm, f->perm, sizeof(int) * (size_t)c, cudaMemcpyDeviceToHost, m->stream));
    else for (int i = 0; i < c; ++i) out_perm[i] = i;
  }
  return fe_download(m, fe_cloud(f), fe_curv(f), f->n_raw, out_xyzi, out_curv, cap);
}

extern "C" int flb_frontend_download_down(flb_frontend* f, float* out_xyzi, float* out_curv, int cap, int* n) {
  if (!f) return set_err("null front end");
  if (f->n_down < 0) return set_err("flb_frontend_download_down: no filtered scan yet");
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  if (n) *n = f->n_down;
  return fe_download(m, f->ses->body, f->down_curv, f->n_down, out_xyzi, out_curv, cap);
}

extern "C" int flb_frontend_points_to_world(flb_frontend* f, int which, const double* state26, float* out_xyzi, int cap, int* n) {
  if (!f) return set_err("null front end");
  if (!state26) return set_err("null state");
  flb_map* m = f->ses->map;
  CU(cudaSetDevice(m->cfg.device));
  const float4* src;
  int cnt;
  if (which == 0) {   // feats_down_body (dense_pub_en == false)
    src = f->ses->body;
    cnt = f->ses->n;
  } else if (which == 1) {   // feats_undistort (dense_pub_en == true, map_save_en)
    src = fe_cloud(f);
    cnt = f->n_raw;
  } else {
    return set_err("which must be 0 (feats_down_body) or 1 (feats_undistort)");
  }
  if (n) *n = cnt;
  if (cnt > f->cap) return set_err("cloud of %d points exceeds the front end capacity %d", cnt, f->cap);
  if (cnt > 0) {
    k_transform<<<grid_for(cnt, 256, m->sm_count * 8), 256, 0, m->stream>>>(pose_from(state26), src, f->world, cnt);
    m->launches++;
    CU(cudaGetLastError());
  }
  return fe_download(m, f->world, nullptr, cnt, out_xyzi, nullptr, cap);
}

// ------------------------------------------------------------------------------------------------ stand-alone filters
static int upload_xyzi(flb_map* m, const void* pts, int n, int stride, int off_intensity, unsigned char** raw, float4* dst) {
  const size_t bytes = (size_t)n * stride;
  CU(cudaMalloc((void**)raw, bytes));
  CU(cudaMemcpyAsync(*raw, pts, bytes, cudaMemcpyHostToDevice, m->stream));
  k_pack_xyzic<<<grid_for(n, 256, m->sm_count * 8), 256, 0, m->stream>>>(*raw, stride, off_intensity, -1, dst, nullptr, n);
  m->launches++;
  CU(cudaGetLastError());
  return 0;
}

extern "C" int flb_voxel_grid_filter(flb_map* m, const void* pts, int n, int stride, int off_intensity, float leaf, float* out_xyzi,
                                     int cap, int* n_out) {
  if (!m) return set_err("null map");
  if (n_out) *n_out = 0;
  if (n < 0) return set_err("negative point count");
  if (!(leaf > 0.f)) return set_err("leaf size must be > 0");
  if (n == 0) return 0;
  if (!pts || stride < 12) return set_err("bad point buffer");
  if (off_intensity >= 0 && off_intensity + 4 > stride) return set_err("field offset outside the point stride");
  CU(cudaSetDevice(m->cfg.device));
  VgWork w;
  unsigned char* raw = nullptr;
  float4 *in = nullptr, *out = nullptr;
  int rc = 0;
  auto body = [&]() -> int {
    CU(cudaMalloc((void**)&in, sizeof(float4) * (size_t)n));
    CU(cudaMalloc((void**)&out, sizeof(float4) * (size_t)n));
    if (upload_xyzi(m, pts, n, stride, off_intensity, &raw, in)) return 1;
    if (vg_enqueue(m, w, in, nullptr, n, leaf, out, nullptr, n, m->stream)) return 1;
    CU(cudaStreamSynchronize(m->stream));
    const bool ovf = w.h_mm[6] != 0;
    const int nd = ovf ? n : (int)w.h_mm[7];
    if (n_out) *n_out = nd;
    const int c = std::min(nd, cap);
    if (c > 0 && out_xyzi) CU(cudaMemcpy(out_xyzi, ovf ? in : out, sizeof(float4) * (size_t)c, cudaMemcpyDeviceToHost));
    return 0;
  };
  rc = body();
  if (raw) Q(cudaFree(raw));
  if (in) Q(cudaFree(in));
  if (out) Q(cudaFree(out));
  vg_release(w);
  return rc;
}

// pcl::getTransformation(x, y, z, roll, pitch, yaw) (PCL 1.10 common/impl/eigen.hpp), float, as transformPointCloud
// uses it (common_lib.h:720-721)
static Affine12 affine_from_rpy(const float* p6) {
  Affine12 a;
  const float x = p6[0], y = p6[1], z = p6[2], roll = p6[3], pitch = p6[4], yaw = p6[5];
  const float A = std::cos(yaw), B = std::sin(yaw), C = std::cos(pitch), D = std::sin(pitch);
  const float E = std::cos(roll), F = std::sin(roll), DE = D * E, DF = D * F;
  a.t[0] = A * C; a.t[1] = A * DF - B * E; a.t[2] = B * F + A * DE; a.t[3] = x;
  a.t[4] = B * C; a.t[5] = A * E + B * DF; a.t[6] = B * DE - A * F; a.t[7] = y;
  a.t[8] = -D;    a.t[9] = C * F;          a.t[10] = C * E;         a.t[11] = z;
  return a;
}

extern "C" int flb_map_reconstruct_keyframes(flb_map* m, const void* const* clouds, const int* sizes, int n_kf, int stride,
                                             int off_intensity, const float* poses6, float leaf, float* out_xyzi, int cap,
                                             int* n_points) {
  if (!m) return set_err("null map");
  if (n_points) *n_points = 0;
  if (n_kf < 0 || (n_kf > 0 && (!clouds || !sizes || !poses6))) return set_err("flb_map_reconstruct_keyframes: bad arguments");
  if (!(leaf > 0.f)) return set_err("leaf size must be > 0");
  if (stride < 12) return set_err("stride_bytes must be >= 12");
  if (off_intensity >= 0 && off_intensity + 4 > stride) return set_err("field offset outside the point stride");
  long long total = 0;
  for (int k = 0; k < n_kf; ++k) {
    if (sizes[k] < 0 || (sizes[k] > 0 && !clouds[k])) return set_err("key frame %d: bad cloud", k);
    total += sizes[k];
  }
  if (total > INT_MAX) return set_err("sub-map of %lld points is too large", total);
  CU(cudaSetDevice(m->cfg.device));
  const int n = (int)total;
  VgWork w;
  unsigned char* raw = nullptr;
  float4 *in = nullptr, *out = nullptr;
  auto body = [&]() -> int {
    if (n == 0) return map_reset_storage(m);   // reconstruct with an empty cloud: everything deleted
    // scratch of the sub-map assembly: kept with the map and only ever grown (recontructIKdTree runs every kd_step key frames
    // with clouds of similar size; cudaMalloc / cudaFree of ~200 MB per call cost more than the kernels)
    const size_t need_raw = (size_t)n * stride, need_pts = sizeof(float4) * (size_t)n;
    if (need_raw > m->kf_raw_cap) {
      if (m->kf_raw) Q(cudaFree(m->kf_raw));
      m->kf_raw = nullptr; m->kf_raw_cap = 0;
      CU(cudaMalloc((void**)&m->kf_raw, need_raw + need_raw / 4));
      m->kf_raw_cap = need_raw + need_raw / 4;
    }
    if (need_pts > m->kf_pts_cap) {
      if (m->kf_in) Q(cudaFree(m->kf_in));
      if (m->kf_out) Q(cudaFree(m->kf_out));
      m->kf_in = m->kf_out = nullptr; m->kf_pts_cap = 0;
      CU(cudaMalloc((void**)&m->kf_in, need_pts + need_pts / 4));
      CU(cudaMalloc((void**)&m->kf_out, need_pts + need_pts / 4));
      m->kf_pts_cap = need_pts + need_pts / 4;
    }
    raw = m->kf_raw; in = m->kf_in; out = m->kf_out;
    // *subMapKeyFrames += *transformPointCloud(surfCloudKeyFrames[k], &cloudKeyPoses6D->points[k])  (laserMapping.cpp:636)
    size_t off = 0;
    for (int k = 0; k < n_kf; ++k) {
      const int c = sizes[k];
      if (c == 0) continue;
      unsigned char* r = raw + off * stride;
      CU(cudaMemcpyAsync(r, clouds[k], (size_t)c * stride, cudaMemcpyHostToDevice, m->stream));
      const int g = grid_for(c, 256, m->sm_count * 8);
      k_pack_xyzic<<<g, 256, 0, m->stream>>>(r, stride, off_intensity, -1, out + off, nullptr, c);
      k_transform_affine<<<g, 256, 0, m->stream>>>(affine_from_rpy(poses6 + 6 * k), out + off, in + off, c);
      m->launches += 2;
      off += c;
    }
    CU(cudaGetLastError());
    // downSizeFilterGlobalMapKeyFrames.filter(*subMapKeyFramesDS)  (laserMapping.cpp:640-643)
    if (vg_enqueue(m, w, in, nullptr, n, leaf, out, nullptr, n, m->stream)) return 1;
    CU(cudaStreamSynchronize(m->stream));
    const bool ovf = w.h_mm[6] != 0;
    const int nd = ovf ? n : (int)w.h_mm[7];
    const float4* ds = ovf ? in : out;
    if (n_points) *n_points = nd;
    // ikdtree.reconstruct(subMapKeyFramesDS->points)  (laserMapping.cpp:656)
    if (map_reset_storage(m)) return 1;
    if (nd > 0 && insert_device(m, ds, nullptr, nd, 0)) return 1;
    if (fetch_counters(m)) return 1;
    // featsFromMap->points = subMapKeyFramesDS->points  (laserMapping.cpp:664)
    const int c = std::min(nd, cap);
    if (c > 0 && out_xyzi) CU(cudaMemcpy(out_xyzi, ds, sizeof(float4) * (size_t)c, cudaMemcpyDeviceToHost));
    return 0;
  };
  const int rc = body();
  vg_release(w);
  return rc;
}
