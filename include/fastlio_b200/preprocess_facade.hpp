// preprocess_facade.hpp — flb::PreprocessGpu, the call shape of the reference's Preprocess (src/preprocess.h) with the
// non-feature branch of its handlers running on the GPU (flb_frontend_preprocess).  In src/laserMapping.cpp:
//
//   shared_ptr<Preprocess> p_pre(new Preprocess());                 // :113
//   ->  shared_ptr<flb::PreprocessGpu> p_pre(new flb::PreprocessGpu());   p_pre->attach(&fe);   // fe: flb::ScanFrontEnd
//
// The members set at :2034-2041 (lidar_type, N_SCANS, SCAN_RATE, point_filter_num, time_unit, blind, feature_enabled)
// and both process() overloads keep their names, so standard_pcl_cbk / livox_pcl_cbk stay as they are.  process()
// leaves pcl_out filled on the host (lidar_buffer / sync_packages read points.size() and points.back().curvature) AND
// on the device: a following ScanFrontEnd::undistort(*meas.lidar, ...) of that same cloud skips its upload, so the
// driver's records cross PCIe once and the 48-byte cloud is never sent back.
//
// Only member names are used: PointCloud2 (fields[].name/offset/datatype, data, point_step, width, height), CustomMsg
// (point_num, points[] with offset_time, x, y, z, reflectivity, tag, line), PointType (x, y, z, intensity, curvature),
// so the header compiles without ROS or PCL.  Like fromROSMsg, which copies bytes and does not convert, a field whose
// datatype differs from the one the handler's point struct declares is rejected; a missing field reads as 0.
#pragma once
#include <cstdio>
#include <cstring>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../fastlio_b200.h"
#include "scan_frontend_facade.hpp"

namespace flb {

class PreprocessGpu {
 public:
  // the public members of Preprocess that laserMapping.cpp sets (preprocess.h)
  int lidar_type = FLB_LIDAR_LIVOX, N_SCANS = 6, SCAN_RATE = 10, point_filter_num = 1, time_unit = 2;
  double blind = 0.01;
  bool feature_enabled = false;
  bool given_offset_time = false;   // Velodyne: whether the last scan carried per-point times (:322-325)

  explicit PreprocessGpu(ScanFrontEnd* fe = nullptr) : fe_(fe) {}
  void attach(ScanFrontEnd* fe) { fe_ = fe; }
  void set(bool feat_en, int lid_type, double bld, int pfilt_num) {
    feature_enabled = feat_en; lidar_type = lid_type; blind = bld; point_filter_num = pfilt_num;
  }

  // process(const CustomMsg::ConstPtr&, PointCloud::Ptr&) and process(const PointCloud2::ConstPtr&, PointCloud::Ptr&).
  // Returns false (and leaves pcl_out empty) on an error, which is also printed.
  template <class MsgPtr, class CloudPtr>
  bool process(const MsgPtr& msg, CloudPtr& pcl_out) {
    pcl_out->points.clear();
    flb_raw_layout L;
    const void* rec = nullptr;
    int n = 0;
    if (!layout(*msg, L, rec, n)) return false;
    return run(rec, n, L, *pcl_out);
  }

  // Field layout of a PointCloud2 for the configured handler, by field name (as fromROSMsg maps them).
  template <class PC2>
  bool pc2_layout(const PC2& m, flb_raw_layout& L) const {
    L = flb_raw_layout{(int)m.point_step, -1, -1, -1, -1, -1, -1, -1, -1};
    const bool velo = lidar_type == FLB_LIDAR_VELO16;
    if (!velo && lidar_type != FLB_LIDAR_OUST64) return fail("lidar_type %d takes a CustomMsg, not a PointCloud2", lidar_type);
    struct Want { const char* name; int datatype; int* off; };
    const Want want[] = {{"x", 7, &L.off_x}, {"y", 7, &L.off_y}, {"z", 7, &L.off_z}, {"intensity", 7, &L.off_intensity},
                         {velo ? "time" : "t", velo ? 7 : 6, &L.off_time}, {"ring", 4, velo ? &L.off_ring : nullptr}};
    for (const auto& f : m.fields) {
      for (const Want& w : want) {
        if (!w.off || std::string(f.name) != w.name) continue;
        if ((int)f.datatype != w.datatype)
          return fail("PointCloud2 field '%s' has datatype %d; the handler's point struct declares %d", w.name, (int)f.datatype, w.datatype);
        *w.off = (int)f.offset;
      }
    }
    return true;
  }

 private:
  template <class T, class = void>
  struct is_pc2 : std::false_type {};
  template <class T>
  struct is_pc2<T, decltype((void)std::declval<const T&>().fields, void())> : std::true_type {};

  template <class Msg>
  bool layout(const Msg& m, flb_raw_layout& L, const void*& rec, int& n) const {
    if constexpr (is_pc2<Msg>::value) {
      if (!pc2_layout(m, L)) return false;
      n = (int)(m.width * m.height);
      if ((size_t)n * m.point_step > m.data.size()) return fail("PointCloud2 holds %zu bytes, fewer than width*height records", m.data.size());
      rec = n ? (const void*)m.data.data() : nullptr;
    } else {   // livox_ros_driver::CustomMsg
      if (lidar_type != FLB_LIDAR_LIVOX) return fail("a CustomMsg needs lidar_type %d (LIVOX)", FLB_LIDAR_LIVOX);
      typedef typename std::decay<decltype(m.points[0])>::type P;
      n = (int)m.point_num;
      if ((size_t)n > m.points.size()) return fail("CustomMsg point_num %d exceeds its %zu points", n, m.points.size());
      const P* p0 = m.points.empty() ? nullptr : &m.points[0];
      static const P probe{};
      const char* b = (const char*)&probe;
      L = flb_raw_layout{(int)sizeof(P), (int)((const char*)&probe.x - b), (int)((const char*)&probe.y - b), (int)((const char*)&probe.z - b),
                         (int)((const char*)&probe.reflectivity - b), (int)((const char*)&probe.offset_time - b), -1,
                         (int)((const char*)&probe.tag - b), (int)((const char*)&probe.line - b)};
      rec = n ? (const void*)p0 : nullptr;
    }
    return true;
  }

  template <class Cloud>
  bool run(const void* rec, int n, const flb_raw_layout& L, Cloud& out) {
    if (!fe_ || !fe_->handle()) return fail("PreprocessGpu is not attached to a ScanFrontEnd");
    const flb_preprocess_cfg cfg{lidar_type, N_SCANS, SCAN_RATE, point_filter_num, time_unit, blind, feature_enabled ? 1 : 0};
    int m = 0;
    float last = 0.f;
    fe_->device_cloud_replaced();
    if (flb_frontend_preprocess(fe_->handle(), rec, n, &L, &cfg, &m, &last)) return fail("%s", flb_last_error());
    if (lidar_type == FLB_LIDAR_VELO16 && n > 0) given_offset_time = last_time_positive(rec, n, L);
    xyzi_.resize((size_t)m * 4 + 4);
    curv_.resize((size_t)m + 1);
    int got = 0;
    if (flb_frontend_download_undistorted(fe_->handle(), xyzi_.data(), curv_.data(), nullptr, m, &got)) return fail("%s", flb_last_error());
    out.points.resize(m);
    for (int i = 0; i < m; ++i) {
      auto& p = out.points[i];
      p = typename std::decay<decltype(p)>::type();
      p.x = xyzi_[4 * (size_t)i]; p.y = xyzi_[4 * (size_t)i + 1]; p.z = xyzi_[4 * (size_t)i + 2];
      p.intensity = xyzi_[4 * (size_t)i + 3]; p.curvature = curv_[i];
    }
    fe_->mark_on_device(out);
    return true;
  }
  static bool last_time_positive(const void* rec, int n, const flb_raw_layout& L) {
    if (L.off_time < 0) return false;
    float t;
    std::memcpy(&t, (const char*)rec + (size_t)(n - 1) * L.stride + L.off_time, sizeof(t));
    return t > 0.f;
  }
  template <class... A>
  static bool fail(const char* fmt, A... a) {
    std::fprintf(stderr, "[fastlio_b200] PreprocessGpu: ");
    std::fprintf(stderr, fmt, a...);
    std::fprintf(stderr, "\n");
    return false;
  }

  ScanFrontEnd* fe_;
  std::vector<float> xyzi_, curv_;
};

}  // namespace flb
