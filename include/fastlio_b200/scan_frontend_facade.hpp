// scan_frontend_facade.hpp — drop-in C++ shapes for the two steps immediately before the per-scan update, so that the raw
// scan stays on the GPU from the driver callback to the posterior (SURVEY.md §8f ranks 1, 2 and 4):
//
//   * flb::ScanFrontEnd::undistort(...)  replaces the per-point backward pass of ImuProcess::UndistortPcl
//     (src/IMU_Processing.hpp:243 sort, :334-386); the forward propagation (:260-329, kf_state.predict per IMU sample)
//     stays where it is and hands over its IMUpose vector and imu_state;
//   * flb::VoxelGridGpu<PointT>          keeps the pcl::VoxelGrid call shape used at src/laserMapping.cpp:2135 and
//     :2322-2323:   downSizeFilterSurf.setLeafSize(l, l, l);  .setInputCloud(feats_undistort);  .filter(*feats_down_body);
//     its result is ALSO the session's current scan, so LioGpu::begin_scan (the upload) is no longer needed;
//   * flb::ScanFrontEnd::to_world(...)   replaces the RGBpointBodyToWorld loops of publish_frame_world
//     (src/laserMapping.cpp:1502-1540).
//
//   flb::ScanFrontEnd fe;  fe.attach(gpu.handle(), 300000);        // next to `flb::LioGpu gpu;`
//   // in ImuProcess::UndistortPcl, instead of lines 334-386:
//   fe.undistort(*meas.lidar, IMUpose, imu_state, pcl_out);        // pcl_out = time-sorted, compensated cloud
//   // in main(), instead of lines 2322-2323:
//   flb::VoxelGridGpu<PointType> downSizeFilterSurf(&fe);  ...  downSizeFilterSurf.filter(*feats_down_body);
//
// Only member names of the reference types are needed (Pose6D: offset_time, acc, gyr, vel, pos, rot —
// msg/Pose6D.msg; pcl::PointCloud: points; PointType: x,y,z,intensity,curvature), so the header compiles without ROS/PCL.
#pragma once
#include <cstddef>
#include <cstdio>
#include <type_traits>
#include <vector>

#include "../fastlio_b200.h"
#include "lio_gpu_frontend.hpp"

namespace flb {

class ScanFrontEnd {
 public:
  ~ScanFrontEnd() { if (fe_) flb_frontend_destroy(fe_); }
  bool attach(flb_session* ses, int max_raw_points) {
    if (flb_frontend_create(ses, max_raw_points, &fe_)) { std::fprintf(stderr, "[fastlio_b200] %s\n", flb_last_error()); fe_ = nullptr; return false; }
    return true;
  }
  flb_frontend* handle() { return fe_; }

  // meas.lidar -> device (IMU_Processing.hpp:242 "pcl_out = *(meas.lidar)")
  template <class Cloud>
  bool upload(const Cloud& cloud) {
    ++gen_;
    typedef typename std::remove_reference<decltype(cloud.points[0])>::type P;
    const int n = (int)cloud.points.size();
    const P* p0 = n ? &cloud.points[0] : nullptr;
    const int off_i = n ? (int)((const char*)&p0->intensity - (const char*)p0) : -1;
    const int off_c = n ? (int)((const char*)&p0->curvature - (const char*)p0) : -1;
    return ok(flb_frontend_upload(fe_, p0, n, (int)sizeof(P), off_i, off_c), "upload");
  }

  // The backward pass of UndistortPcl.  poses = IMUpose (vector<Pose6D>), imu_state = kf_state.get_x() after the last
  // predict.  When `out` is given it receives the time-sorted compensated cloud (x,y,z,intensity,curvature), i.e. pcl_out.
  template <class Cloud, class PoseVec, class State>
  bool undistort(const Cloud& lidar, const PoseVec& poses, const State& imu_state, Cloud* out = nullptr) {
    if (!on_device(lidar) && !upload(lidar)) return false;
    std::vector<double> pz(poses.size() * FLB_IMU_POSE_DOUBLES);
    for (size_t k = 0; k < poses.size(); ++k) {
      double* o = &pz[k * FLB_IMU_POSE_DOUBLES];
      o[0] = poses[k].offset_time;
      for (int i = 0; i < 3; ++i) { o[1 + i] = poses[k].acc[i]; o[4 + i] = poses[k].gyr[i]; o[7 + i] = poses[k].vel[i]; o[10 + i] = poses[k].pos[i]; }
      for (int i = 0; i < 9; ++i) o[13 + i] = poses[k].rot[i];
    }
    double st[FLB_STATE_DIM];
    pack_state26(imu_state, st);
    if (!ok(flb_frontend_undistort(fe_, pz.data(), (int)poses.size(), st), "undistort")) return false;
    if (out) {
      const int n = (int)lidar.points.size();
      xyzi_.resize((size_t)n * 4);
      curv_.resize(n);
      int m = 0;
      if (!ok(flb_frontend_download_undistorted(fe_, xyzi_.data(), curv_.data(), nullptr, n, &m), "download")) return false;
      out->points.resize(m);
      for (int i = 0; i < m; ++i) fill(out->points[i], &xyzi_[4 * (size_t)i], curv_[i]);
    }
    return true;
  }

  // downSizeFilterSurf.filter(*feats_down_body): leaves feats_down_body as the session's current scan; returns
  // feats_down_size (or -1).  `out` (optional) receives the centroids on the host as well.
  template <class Cloud>
  int voxel_filter(float leaf, Cloud* out) {
    int n = 0;
    if (!ok(flb_frontend_voxel_filter(fe_, leaf, &n), "voxel_filter")) return -1;
    if (out) {
      xyzi_.resize((size_t)n * 4 + 4);
      curv_.resize(n + 1);
      int m = 0;
      if (!ok(flb_frontend_download_down(fe_, xyzi_.data(), curv_.data(), n, &m), "download")) return -1;
      out->points.resize(n);
      for (int i = 0; i < n; ++i) fill(out->points[i], &xyzi_[4 * (size_t)i], curv_[i]);
    }
    return n;
  }

  // publish_frame_world (laserMapping.cpp:1506-1514, :1529-1536): dense = feats_undistort, else feats_down_body
  template <class State, class Cloud>
  bool to_world(const State& state_point, bool dense, Cloud& laserCloudWorld, int capacity) {
    double st[FLB_STATE_DIM];
    pack_state26(state_point, st);
    xyzi_.resize((size_t)capacity * 4 + 4);
    int n = 0;
    if (!ok(flb_frontend_points_to_world(fe_, dense ? 1 : 0, st, xyzi_.data(), capacity, &n), "to_world")) return false;
    if (n > capacity) n = capacity;
    laserCloudWorld.points.resize(n);
    for (int i = 0; i < n; ++i) fill(laserCloudWorld.points[i], &xyzi_[4 * (size_t)i], 0.f);
    return true;
  }

  // Called by PreprocessGpu after it left `cloud` on the device: until the next upload or preprocess, undistort()
  // of this very cloud (same object, same point storage and size) uses the device copy instead of uploading it.
  void device_cloud_replaced() { ++gen_; }
  template <class Cloud>
  void mark_on_device(const Cloud& cloud) {
    dev_gen_ = ++gen_;
    dev_cloud_ = &cloud;
    dev_points_ = cloud.points.empty() ? nullptr : (const void*)&cloud.points[0];
    dev_n_ = cloud.points.size();
  }

 private:
  template <class P>
  static void fill(P& p, const float* v, float curvature) {
    p = P();
    p.x = v[0]; p.y = v[1]; p.z = v[2]; p.intensity = v[3]; p.curvature = curvature;
  }
  template <class Cloud>
  bool on_device(const Cloud& c) const {
    return dev_gen_ == gen_ && dev_cloud_ == (const void*)&c && dev_n_ == c.points.size() &&
           dev_points_ == (c.points.empty() ? nullptr : (const void*)&c.points[0]);
  }
  static bool ok(int rc, const char* what) {
    if (rc) std::fprintf(stderr, "[fastlio_b200] %s: %s\n", what, flb_last_error());
    return rc == 0;
  }
  flb_frontend* fe_ = nullptr;
  std::vector<float> xyzi_, curv_;
  unsigned long long gen_ = 0, dev_gen_ = 0;   // bumped by every upload / preprocess
  const void* dev_cloud_ = nullptr;
  const void* dev_points_ = nullptr;
  size_t dev_n_ = 0;
};

// pcl::VoxelGrid<PointT> call shape on top of a ScanFrontEnd.  setInputCloud() is accepted for source compatibility: the
// cloud that is filtered is the one the front end already holds on the device (the output of undistort(), or of an
// explicit ScanFrontEnd::upload() when the caller has no IMU step).
template <class PointT>
class VoxelGridGpu {
 public:
  explicit VoxelGridGpu(ScanFrontEnd* fe = nullptr) : fe_(fe) {}
  void attach(ScanFrontEnd* fe) { fe_ = fe; }
  void setLeafSize(float lx, float ly, float lz) {
    if (lx != ly || lx != lz) std::fprintf(stderr, "[fastlio_b200] VoxelGridGpu: anisotropic leaves are not supported (the reference never uses them)\n");
    leaf_ = lx;
  }
  template <class CloudPtr>
  void setInputCloud(const CloudPtr&) {}
  template <class Cloud>
  void filter(Cloud& output) {
    const int n = fe_ ? fe_->voxel_filter(leaf_, &output) : -1;
    if (n < 0) output.points.clear();
  }

 private:
  ScanFrontEnd* fe_;
  float leaf_ = 0.5f;
};

}  // namespace flb
