// TEST INFRASTRUCTURE ONLY (oracle). Stand-in for livox_ros_driver's generated message headers (msg/CustomPoint.msg,
// msg/CustomMsg.msg): the members preprocess.cpp reads, in the message's field order.
#pragma once
#include <cstdint>
#include <memory>
#include <vector>

#include "../common_lib.h"

namespace livox_ros_driver {
struct CustomPoint {
  uint32_t offset_time;   // ns, relative to timebase
  float x, y, z;
  uint8_t reflectivity, tag, line;
};
struct CustomMsg {
  typedef std::shared_ptr<CustomMsg> Ptr;
  typedef std::shared_ptr<const CustomMsg> ConstPtr;
  std_msgs::Header header;
  uint64_t timebase = 0;
  uint32_t point_num = 0;
  uint8_t lidar_id = 0;
  std::vector<CustomPoint> points;
};
}  // namespace livox_ros_driver
