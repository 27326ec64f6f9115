// TEST INFRASTRUCTURE ONLY. C entry points around the REFERENCE's own Preprocess (src/preprocess.cpp, compiled unmodified
// next to this file by oracle/preprocess_ref.mk against the stand-in headers in shim/preprocess/).
// Records go in with the layouts of the reference's point structs (velodyne_ros::Point, ouster_ros::Point,
// livox_ros_driver::CustomPoint) -- the same bytes better_fastlio2_b200.capi's *_RECORD dtypes describe -- and
// pl_surf comes out as 48-byte PointType records.
#include <cstddef>
#include <cstring>

#include "preprocess.h"

static_assert(sizeof(velodyne_ros::Point) == 32 && offsetof(velodyne_ros::Point, intensity) == 16 &&
                  offsetof(velodyne_ros::Point, time) == 20 && offsetof(velodyne_ros::Point, ring) == 24,
              "velodyne_ros::Point layout");
static_assert(sizeof(ouster_ros::Point) == 48 && offsetof(ouster_ros::Point, intensity) == 16 && offsetof(ouster_ros::Point, t) == 20 &&
                  offsetof(ouster_ros::Point, ring) == 26,
              "ouster_ros::Point layout");
static_assert(sizeof(livox_ros_driver::CustomPoint) == 20 && offsetof(livox_ros_driver::CustomPoint, x) == 4 &&
                  offsetof(livox_ros_driver::CustomPoint, reflectivity) == 16 && offsetof(livox_ros_driver::CustomPoint, line) == 18,
              "CustomPoint layout");
static_assert(sizeof(PointType) == 48, "PointType layout");

extern "C" {

void* ppref_create() { return new Preprocess(); }
void ppref_destroy(void* h) { delete static_cast<Preprocess*>(h); }

// One Preprocess::process call with the public members set as laserMapping.cpp:2034-2041 does.  Returns pl_surf.size()
// (at most cap records are written to out48) or -1 for an unknown lidar_type.
int ppref_process(void* h, int lidar_type, int n_scans, int scan_rate, int point_filter_num, int time_unit, double blind,
                  const void* records, int n, float* out48, int cap, int* given_offset_time) {
  Preprocess& p = *static_cast<Preprocess*>(h);
  p.lidar_type = lidar_type;
  p.N_SCANS = n_scans;
  p.SCAN_RATE = scan_rate;
  p.point_filter_num = point_filter_num;
  p.time_unit = time_unit;
  p.blind = blind;
  p.feature_enabled = false;
  pcl::PointCloud<PointType>::Ptr out(new pcl::PointCloud<PointType>());
  if (lidar_type == LIVOX) {
    livox_ros_driver::CustomMsg::Ptr msg(new livox_ros_driver::CustomMsg());
    msg->point_num = (uint32_t)n;
    msg->points.resize(n);
    if (n) std::memcpy(msg->points.data(), records, sizeof(livox_ros_driver::CustomPoint) * (size_t)n);
    p.process(livox_ros_driver::CustomMsg::ConstPtr(msg), out);
  } else if (lidar_type == VELO16 || lidar_type == OUST64) {
    sensor_msgs::PointCloud2::Ptr msg(new sensor_msgs::PointCloud2());
    const size_t stride = lidar_type == VELO16 ? sizeof(velodyne_ros::Point) : sizeof(ouster_ros::Point);
    msg->width = (uint32_t)n;
    msg->point_step = (uint32_t)stride;
    msg->data.assign((const uint8_t*)records, (const uint8_t*)records + stride * (size_t)n);
    p.process(sensor_msgs::PointCloud2::ConstPtr(msg), out);
  } else {
    return -1;
  }
  if (given_offset_time) *given_offset_time = p.given_offset_time ? 1 : 0;
  const int m = (int)out->points.size();
  for (int i = 0; i < m && i < cap; ++i) std::memcpy(out48 + 12 * (size_t)i, &out->points[i], sizeof(PointType));
  return m;
}

}  // extern "C"
