// TEST INFRASTRUCTURE ONLY (oracle). Stand-in for the reference's include/common_lib.h, so that its src/preprocess.cpp
// compiles unmodified without ROS, PCL or Eigen (see oracle/preprocess_ref.mk: -I shim/preprocess, NOT -I$(REF)/include).
// Only what preprocess.{h,cpp} touch: PointType (pcl::PointXYZINormal), pcl::PointCloud, the PCL / Eigen point macros,
// a 3-vector with the Eigen::Vector3d operations give_feature uses, sensor_msgs::PointCloud2 with a record-copy
// fromROSMsg, and ros::Time / Publisher.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#define PCL_ADD_POINT4D float x, y, z, data_pad_
#define PCL_ADD_RGB float rgb
#define EIGEN_ALIGN16 alignas(16)
#define EIGEN_MAKE_ALIGNED_OPERATOR_NEW
#define POINT_CLOUD_REGISTER_POINT_STRUCT(...)

namespace ros {
struct Time {
  double t = 0.0;
  double toSec() const { return t; }
};
struct Publisher {};
}  // namespace ros

namespace std_msgs {
struct Header {
  ros::Time stamp;
  std::string frame_id;
};
}  // namespace std_msgs

namespace Eigen {
struct Vector3d;
struct RowVector3d {
  double v[3];
  double operator*(const Vector3d& o) const;
};
struct Vector3d {
  double v[3] = {0.0, 0.0, 0.0};
  Vector3d() = default;
  Vector3d(double a, double b, double c) : v{a, b, c} {}
  static Vector3d Zero() { return Vector3d(); }
  double dot(const Vector3d& o) const { return v[0] * o.v[0] + v[1] * o.v[1] + v[2] * o.v[2]; }
  double norm() const { return std::sqrt(dot(*this)); }
  void setZero() { v[0] = v[1] = v[2] = 0.0; }
  void normalize() {
    const double n = norm();
    if (n > 0.0) { v[0] /= n; v[1] /= n; v[2] /= n; }
  }
  Vector3d operator-(const Vector3d& o) const { return Vector3d(v[0] - o.v[0], v[1] - o.v[1], v[2] - o.v[2]); }
  RowVector3d transpose() const { return RowVector3d{{v[0], v[1], v[2]}}; }
  struct Comma {
    Vector3d* d;
    int k;
    Comma& operator,(double a) { d->v[k++] = a; return *this; }
  };
  Comma operator<<(double a) { v[0] = a; return Comma{this, 1}; }
};
inline double RowVector3d::operator*(const Vector3d& o) const { return v[0] * o.v[0] + v[1] * o.v[1] + v[2] * o.v[2]; }
}  // namespace Eigen

namespace pcl {
struct PointXYZINormal {   // 48 bytes, default-constructed as PCL does (xyz 0, data[3] = 1, the rest 0)
  float x = 0.f, y = 0.f, z = 0.f, data_pad_ = 1.f;
  float normal_x = 0.f, normal_y = 0.f, normal_z = 0.f, data_n_pad_ = 0.f;
  float intensity = 0.f, curvature = 0.f, pad_[2] = {0.f, 0.f};
};
template <class T>
struct PointCloud {
  typedef std::shared_ptr<PointCloud<T>> Ptr;
  typedef std::shared_ptr<const PointCloud<T>> ConstPtr;
  std::vector<T> points;
  uint32_t width = 0, height = 1;
  size_t size() const { return points.size(); }
  bool empty() const { return points.empty(); }
  void clear() { points.clear(); width = 0; }
  void reserve(size_t n) { points.reserve(n); }
  void resize(size_t n) { points.resize(n); width = (uint32_t)n; }
  void push_back(const T& p) { points.push_back(p); width = (uint32_t)points.size(); }
  T& operator[](size_t i) { return points[i]; }
  const T& operator[](size_t i) const { return points[i]; }
};
}  // namespace pcl

typedef pcl::PointXYZINormal PointType;

namespace sensor_msgs {
struct PointCloud2 {
  typedef std::shared_ptr<PointCloud2> Ptr;
  typedef std::shared_ptr<const PointCloud2> ConstPtr;
  std_msgs::Header header;
  uint32_t height = 1, width = 0, point_step = 0;
  std::vector<uint8_t> data;   // width * height records of the driver's point struct
};
}  // namespace sensor_msgs

namespace pcl {
// pcl::fromROSMsg with a message whose fields are laid out as T: a plain record copy
template <class T>
void fromROSMsg(const sensor_msgs::PointCloud2& msg, PointCloud<T>& cloud) {
  const size_t n = (size_t)msg.width * msg.height;
  cloud.points.resize(n);
  for (size_t i = 0; i < n; ++i) std::memcpy((void*)&cloud.points[i], msg.data.data() + i * msg.point_step, sizeof(T));
  cloud.width = (uint32_t)n;
  cloud.height = 1;
}
template <class T>
void toROSMsg(const PointCloud<T>&, sensor_msgs::PointCloud2&) {}
}  // namespace pcl
