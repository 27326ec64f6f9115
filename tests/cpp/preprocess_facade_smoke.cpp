// Compile-and-run check of flb::PreprocessGpu (include/fastlio_b200/preprocess_facade.hpp) with message types shaped
// like sensor_msgs::PointCloud2 and livox_ros_driver::CustomMsg.  The PointCloud2 uses a field order unlike the
// reference's point struct; the result must equal flb_frontend_preprocess on the same points in the reference layout.
// Built by tests/test_preprocess_facade_cpp.py:  g++ -Ioracle/shim -Iinclude ... -lfastlio_b200
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <random>
#include <string>
#include <vector>

#include <fastlio_b200/lio_gpu_frontend.hpp>
#include <fastlio_b200/preprocess_facade.hpp>
#include <fastlio_b200/scan_frontend_facade.hpp>
#include <pcl/point_types.h>

typedef pcl::PointXYZINormal PointType;
struct Cloud {
  typedef std::shared_ptr<Cloud> Ptr;
  std::vector<PointType> points;
};
struct PointField { std::string name; uint32_t offset; uint8_t datatype; uint32_t count; };
struct PointCloud2 {
  typedef std::shared_ptr<const PointCloud2> ConstPtr;
  uint32_t height = 1, width = 0, point_step = 0;
  std::vector<PointField> fields;
  std::vector<uint8_t> data;
};
struct CustomPoint { uint32_t offset_time; float x, y, z; uint8_t reflectivity, tag, line; };
struct CustomMsg {
  typedef std::shared_ptr<const CustomMsg> ConstPtr;
  uint32_t point_num = 0;
  std::vector<CustomPoint> points;
};

template <class T> static void put(std::vector<uint8_t>& d, size_t at, T v) { std::memcpy(d.data() + at, &v, sizeof(T)); }

static int compare(const Cloud& a, flb_frontend* fe, const void* rec, int n, const flb_raw_layout& L, const flb_preprocess_cfg& cfg,
                   int code) {
  int m = 0;
  float last = 0.f;
  if (flb_frontend_preprocess(fe, rec, n, &L, &cfg, &m, &last)) { std::printf("abi: %s\n", flb_last_error()); return code; }
  std::vector<float> xyzi((size_t)m * 4 + 4), cur((size_t)m + 1);
  int got = 0;
  if (flb_frontend_download_undistorted(fe, xyzi.data(), cur.data(), nullptr, m, &got)) return code + 1;
  if (m != (int)a.points.size() || m == 0) { std::printf("count %d vs %zu\n", m, a.points.size()); return code + 2; }
  for (int i = 0; i < m; ++i) {
    const PointType& p = a.points[i];
    const float v[5] = {p.x, p.y, p.z, p.intensity, p.curvature};
    const float w[5] = {xyzi[4 * i], xyzi[4 * i + 1], xyzi[4 * i + 2], xyzi[4 * i + 3], cur[i]};
    if (std::memcmp(v, w, sizeof(v))) { std::printf("point %d differs\n", i); return code + 3; }
  }
  if (std::memcmp(&last, &a.points.back().curvature, sizeof(float))) return code + 4;
  return 0;
}

int main() {
  if (flb_device_count() <= 0) { std::printf("NO_GPU compile-only ok\n"); return 0; }
  flb_map_config mc{0.5f, 1 << 16, 1 << 12, 0};
  flb_map* map = nullptr;
  if (flb_map_create(&mc, &map)) { std::printf("%s\n", flb_last_error()); return 2; }
  flb_session_config sc;
  flb_session_default_config(&sc);
  flb_session* ses = nullptr;
  if (flb_session_create(map, &sc, &ses)) { std::printf("%s\n", flb_last_error()); return 3; }
  flb::ScanFrontEnd fe;
  if (!fe.attach(ses, 1 << 16)) return 4;
  flb::PreprocessGpu pre(&fe);

  // Velodyne-like cloud, 32 rings column-major, shuffled fields: ring@0 time@4 z@8 intensity@12 x@16 y@20, 24 bytes
  std::mt19937 rng(3);
  std::uniform_real_distribution<float> U(2.f, 40.f);
  const int cols = 400, rings = 32, n = cols * rings;
  for (int timed = 0; timed < 2; ++timed) {
    PointCloud2 pc;
    pc.width = n;
    pc.point_step = 24;
    pc.fields = {{"ring", 0, 4, 1}, {"time", 4, 7, 1}, {"z", 8, 7, 1}, {"intensity", 12, 7, 1}, {"x", 16, 7, 1}, {"y", 20, 7, 1}};
    pc.data.assign((size_t)n * 24, 0);
    std::vector<uint8_t> ref((size_t)n * 32, 0);   // velodyne_ros::Point layout: x y z _ intensity time ring
    for (int c = 0; c < cols; ++c)
      for (int r = 0; r < rings; ++r) {
        const int i = c * rings + r;
        const float az = -6.2831853f * c / cols, d = U(rng);
        const float x = d * std::cos(az), y = d * std::sin(az), z = 0.05f * r - 1.f, in = (float)(i % 255);
        const float t = timed ? 0.1f * (c + 1) / cols : 0.f;
        const uint16_t ring = (uint16_t)r;
        put(pc.data, i * 24 + 0, ring); put(pc.data, i * 24 + 4, t); put(pc.data, i * 24 + 8, z);
        put(pc.data, i * 24 + 12, in); put(pc.data, i * 24 + 16, x); put(pc.data, i * 24 + 20, y);
        put(ref, i * 32 + 0, x); put(ref, i * 32 + 4, y); put(ref, i * 32 + 8, z);
        put(ref, i * 32 + 16, in); put(ref, i * 32 + 20, t); put(ref, i * 32 + 24, ring);
      }
    pre.lidar_type = FLB_LIDAR_VELO16; pre.N_SCANS = rings; pre.SCAN_RATE = 10; pre.point_filter_num = 2; pre.time_unit = 0;
    pre.blind = 5.0;
    Cloud::Ptr out(new Cloud());
    if (!pre.process(PointCloud2::ConstPtr(new PointCloud2(pc)), out)) return 10;
    if (pre.given_offset_time != (timed == 1)) return 11;
    const flb_raw_layout L{32, 0, 4, 8, 16, 20, 24, -1, -1};
    const flb_preprocess_cfg cfg{FLB_LIDAR_VELO16, rings, 10, 2, 0, 5.0, 0};
    if (int rc = compare(*out, fe.handle(), ref.data(), n, L, cfg, 20 + 10 * timed)) return rc;
    // a field with another datatype than velodyne_ros::Point declares is rejected, as fromROSMsg would not convert it
    pc.fields[0].datatype = 5;
    if (pre.process(PointCloud2::ConstPtr(new PointCloud2(pc)), out) || !out->points.empty()) return 40;
  }

  // Livox CustomMsg
  CustomMsg lm;
  lm.point_num = 3000;
  for (int i = 0; i < 3000; ++i) {
    CustomPoint p{};
    p.offset_time = (uint32_t)(i * 33333);
    p.x = U(rng); p.y = U(rng) - 20.f; p.z = 0.1f * (i % 7);
    if (i % 11 == 0 && i) p = lm.points.back();   // consecutive duplicate
    p.reflectivity = (uint8_t)(i % 256); p.tag = (uint8_t)((i % 5) * 0x10); p.line = (uint8_t)(i % 8);
    lm.points.push_back(p);
  }
  pre.lidar_type = FLB_LIDAR_LIVOX; pre.N_SCANS = 6; pre.point_filter_num = 3; pre.blind = 0.5;
  Cloud::Ptr lout(new Cloud());
  if (!pre.process(CustomMsg::ConstPtr(new CustomMsg(lm)), lout)) return 50;
  const flb_raw_layout LL{(int)sizeof(CustomPoint), 4, 8, 12, 16, 0, -1, 17, 18};
  const flb_preprocess_cfg lcfg{FLB_LIDAR_LIVOX, 6, 10, 3, 2, 0.5, 0};
  if (int rc = compare(*lout, fe.handle(), lm.points.data(), 3000, LL, lcfg, 60)) return rc;
  // feature extraction is not supported: reported, nothing produced
  pre.feature_enabled = true;
  if (pre.process(CustomMsg::ConstPtr(new CustomMsg(lm)), lout) || !lout->points.empty()) return 70;
  std::printf("PREPROCESS_FACADE_OK\n");
  return 0;
}
