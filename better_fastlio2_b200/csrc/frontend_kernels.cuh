// frontend_kernels.cuh — the rows either side of the per-scan path (SURVEY.md §8f), as sm_100a kernels:
//   rank 2  UndistortPcl backward pass          src/IMU_Processing.hpp:241-243 (time sort), :334-386 (compensation)
//   rank 1  pcl::VoxelGrid centroid filter      src/laserMapping.cpp:2322-2323 (leaf :2135); PCL 1.10 voxel_grid.hpp
//   rank 3  transformPointCloud (key frames)    include/common_lib.h:711-734, used by recontructIKdTree laserMapping.cpp:636
//   rank 4  pointBodyToWorld / RGBpointBodyToWorld for publishing   src/laserMapping.cpp:1077-1110, :1502-1540
// All of it is per-point streaming work (HBM bound, a few dozen bytes per point); sorting is cub::DeviceRadixSort.
// The TU is compiled with -fmad=false: the reference is built without FMA contraction (CMakeLists.txt:9, no -march).
#pragma once
#include "knn_kernels.cuh"

namespace flb {

// monotone float -> uint map (radix-sortable; -0.0 < +0.0 as for the total order, NaN sorts last for positive NaN)
__device__ __forceinline__ unsigned f2ordu(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordu2f(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
}

// strided host-layout points (e.g. 48-byte pcl::PointXYZINormal: x@0 y@4 z@8 intensity@32 curvature@36) -> float4
// (x,y,z,intensity) + curvature; a negative offset means "field absent" (0).
__global__ void k_pack_xyzic(const unsigned char* __restrict__ src, int stride, int off_i, int off_c, float4* __restrict__ dst,
                             float* __restrict__ curv, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned char* b = src + (size_t)i * stride;
    const float* p = reinterpret_cast<const float*>(b);
    const float in = off_i >= 0 ? *reinterpret_cast<const float*>(b + off_i) : 0.f;
    dst[i] = make_float4(p[0], p[1], p[2], in);
    if (curv) curv[i] = off_c >= 0 ? *reinterpret_cast<const float*>(b + off_c) : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------ undistortion
constexpr int IMU_POSE_DOUBLES = 22;   // Pose6D: offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9] (msg/Pose6D.msg)
constexpr int MAX_IMU_POSES = 256;     // 22*8*256 = 44 KB staged in shared memory (typical scans: 20-100 IMU samples)

struct UndistortEnd {   // imu_state after the forward propagation (IMU_Processing.hpp:329)
  double rot[4], offR[4], pos[3], offT[3];
};

__global__ void k_time_keys(const float* __restrict__ curv, unsigned* __restrict__ keys, int* __restrict__ vals, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    keys[i] = f2ordu(curv[i]);
    vals[i] = i;
  }
}

__device__ __forceinline__ void exp_so3_d(const double* w, double dt, double* R) {   // Exp(ang_vel, dt), math_tools.h:39-61
  const double n = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  R[0] = 1.0; R[1] = 0.0; R[2] = 0.0; R[3] = 0.0; R[4] = 1.0; R[5] = 0.0; R[6] = 0.0; R[7] = 0.0; R[8] = 1.0;
  if (!(n > 0.0000001)) return;
  const double a0 = w[0] / n, a1 = w[1] / n, a2 = w[2] / n;
  const double K[9] = {0.0, -a2, a1, a2, 0.0, -a0, -a1, a0, 0.0};
  const double r = n * dt;
  double s, c;
  sincos(r, &s, &c);
  const double c1 = 1.0 - c;
  double cK[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) cK[i] = c1 * K[i];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double kk = cK[i * 3 + 0] * K[j] + cK[i * 3 + 1] * K[3 + j] + cK[i * 3 + 2] * K[6 + j];
      R[i * 3 + j] = (R[i * 3 + j] + s * K[i * 3 + j]) + kk;
    }
}

// one compensation with segment (head, tail) (IMU_Processing.hpp:353-378)
__device__ __forceinline__ void undistort_point(float& px, float& py, float& pz, double t, const double* head, const double* tail,
                                                const UndistortEnd& e) {
  const double dt = t - head[0];
  double E[9], Ri[9];
  exp_so3_d(tail + 4, dt, E);
  const double* Rm = head + 13;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Ri[i * 3 + j] = Rm[i * 3] * E[j] + Rm[i * 3 + 1] * E[3 + j] + Rm[i * 3 + 2] * E[6 + j];
  double T[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) T[k] = ((head[10 + k] + head[7 + k] * dt) + ((0.5 * tail[1 + k]) * dt) * dt) - e.pos[k];
  double ax, ay, az;
  qrot_d(e.offR, (double)px, (double)py, (double)pz, ax, ay, az);
  ax += e.offT[0]; ay += e.offT[1]; az += e.offT[2];
  double bx = (Ri[0] * ax + Ri[1] * ay + Ri[2] * az) + T[0];
  double by = (Ri[3] * ax + Ri[4] * ay + Ri[5] * az) + T[1];
  double bz = (Ri[6] * ax + Ri[7] * ay + Ri[8] * az) + T[2];
  const double rc[4] = {-e.rot[0], -e.rot[1], -e.rot[2], e.rot[3]};
  const double oc[4] = {-e.offR[0], -e.offR[1], -e.offR[2], e.offR[3]};
  double cx, cy, cz, dx, dy, dz;
  qrot_d(rc, bx, by, bz, cx, cy, cz);
  cx -= e.offT[0]; cy -= e.offT[1]; cz -= e.offT[2];
  qrot_d(oc, cx, cy, cz, dx, dy, dz);
  px = (float)dx; py = (float)dy; pz = (float)dz;
}

// Thread j handles the j-th point in time order (perm from the stable radix sort by curvature).  A point belongs to
// the LAST segment whose head time it exceeds (what the reference's backward double sweep computes for time-sorted
// points); points not later than IMUpose[0] stay untouched.  Quirk kept: the first sorted point is compensated again by
// every earlier segment whose head time it exceeds (the `break` at begin() leaves the iterator on it, :382-383).
__global__ void k_undistort(const float4* __restrict__ pts, const float* __restrict__ curv, const int* __restrict__ perm, int n,
                            const double* __restrict__ poses, int np, UndistortEnd e, float4* __restrict__ out,
                            float* __restrict__ out_curv) {
  extern __shared__ double sp[];
  for (int k = threadIdx.x; k < np * IMU_POSE_DOUBLES; k += blockDim.x) sp[k] = poses[k];
  __syncthreads();
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const int i = perm[j];
    float4 p = pts[i];
    const float cf = curv[i];
    const double t = (double)cf / double(1000);
    int h = np - 2;
    while (h >= 0 && !(t > sp[h * IMU_POSE_DOUBLES])) --h;
    if (h >= 0) {
      undistort_point(p.x, p.y, p.z, t, sp + h * IMU_POSE_DOUBLES, sp + (h + 1) * IMU_POSE_DOUBLES, e);
      if (j == 0) {
        for (int g = h - 1; g >= 0; --g)
          if (t > sp[g * IMU_POSE_DOUBLES])
            undistort_point(p.x, p.y, p.z, t, sp + g * IMU_POSE_DOUBLES, sp + (g + 1) * IMU_POSE_DOUBLES, e);
      }
    }
    out[j] = p;
    out_curv[j] = cf;
  }
}

// ------------------------------------------------------------------------------------------------ voxel grid
// d_mm[0..2] = ordered-uint min x,y,z ; d_mm[3..5] = ordered-uint max ; d_mm[6] = overflow flag ; d_mm[7] = #outputs
__global__ void k_vg_init(unsigned* mm) {
  if (threadIdx.x < 3) mm[threadIdx.x] = 0xFFFFFFFFu;
  else if (threadIdx.x < 8) mm[threadIdx.x] = 0u;
}
__global__ void k_vg_minmax(const float4* __restrict__ pts, int n, unsigned* __restrict__ mm) {   // getMinMax3D
  unsigned lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) continue;
    const unsigned ox = f2ordu(p.x), oy = f2ordu(p.y), oz = f2ordu(p.z);
    lo[0] = min(lo[0], ox); lo[1] = min(lo[1], oy); lo[2] = min(lo[2], oz);
    hi[0] = max(hi[0], ox); hi[1] = max(hi[1], oy); hi[2] = max(hi[2], oz);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    lo[k] = __reduce_min_sync(FULL, lo[k]);
    hi[k] = __reduce_max_sync(FULL, hi[k]);
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      atomicMin(&mm[k], lo[k]);
      atomicMax(&mm[3 + k], hi[k]);
    }
  }
}

struct VgGrid { int min_b[3]; int mul[3]; bool overflow; };
// min_b_, div_b_, divb_mul_ and the overflow guard of applyFilter, recomputed per thread from the 6 extrema (cheap)
__device__ __forceinline__ VgGrid vg_grid(const unsigned* mm, float inv) {
  VgGrid g;
  float mn[3], mx[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { mn[k] = ordu2f(mm[k]); mx[k] = ordu2f(mm[3 + k]); }
  const long long dx = (long long)((mx[0] - mn[0]) * inv) + 1;
  const long long dy = (long long)((mx[1] - mn[1]) * inv) + 1;
  const long long dz = (long long)((mx[2] - mn[2]) * inv) + 1;
  g.overflow = (dx * dy * dz) > (long long)INT_MAX;
  int div[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    g.min_b[k] = (int)floorf(mn[k] * inv);
    div[k] = (int)floorf(mx[k] * inv) - g.min_b[k] + 1;
  }
  g.mul[0] = 1; g.mul[1] = div[0]; g.mul[2] = div[0] * div[1];
  return g;
}

__global__ void k_vg_keys(const float4* __restrict__ pts, int n, float inv, unsigned* __restrict__ mm, unsigned* __restrict__ keys,
                          int* __restrict__ vals) {
  const VgGrid g = vg_grid(mm, inv);
  if (blockIdx.x == 0 && threadIdx.x == 0) mm[6] = g.overflow ? 1u : 0u;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    unsigned key = 0xFFFFFFFFu;   // non-finite points are dropped (PCL does so for non-dense clouds)
    if (!g.overflow && isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
      const int i0 = (int)(floorf(p.x * inv) - (float)g.min_b[0]);
      const int i1 = (int)(floorf(p.y * inv) - (float)g.min_b[1]);
      const int i2 = (int)(floorf(p.z * inv) - (float)g.min_b[2]);
      key = (unsigned)(i0 * g.mul[0] + i1 * g.mul[1] + i2 * g.mul[2]);
    }
    keys[i] = key;
    vals[i] = i;
  }
}

__global__ void k_vg_heads(const unsigned* __restrict__ keys, int n, int* __restrict__ flags) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned k = keys[i];
    flags[i] = (k != 0xFFFFFFFFu && (i == 0 || keys[i - 1] != k)) ? 1 : 0;
  }
}

// The thread of each leaf's first sorted point sums the leaf sequentially in sorted order (stable sort => ascending
// input index, a fixed order) exactly as CentroidPoint does: float sums, then division by the count as a float.
__global__ void k_vg_centroid(const float4* __restrict__ pts, const float* __restrict__ curv, const unsigned* __restrict__ keys,
                              const int* __restrict__ vals, const int* __restrict__ flags, const int* __restrict__ pos, int n,
                              float4* __restrict__ out, float* __restrict__ out_curv, int out_cap, unsigned* __restrict__ mm) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (!flags[i]) continue;
    const unsigned k = keys[i];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f, sc = 0.f;
    int j = i;
    for (; j < n && keys[j] == k; ++j) {
      const int src = vals[j];
      const float4 p = pts[src];
      sx += p.x; sy += p.y; sz += p.z; si += p.w;
      if (curv) sc += curv[src];
    }
    const float cnt = (float)(j - i);
    const int o = pos[i];
    if (o < out_cap) {
      out[o] = make_float4(sx / cnt, sy / cnt, sz / cnt, si / cnt);
      if (out_curv) out_curv[o] = sc / cnt;
    }
    if (j == n || keys[j] == 0xFFFFFFFFu) mm[7] = (unsigned)(o + 1);   // the last leaf publishes the output count
  }
}

// ------------------------------------------------------------------------------------------------ transforms
// transformPointCloud (common_lib.h:711-734): float affine "t00*x + t01*y + t02*z + t03", intensity copied
struct Affine12 { float t[12]; };
__global__ void k_transform_affine(Affine12 a, const float4* __restrict__ in, float4* __restrict__ out, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    out[i] = make_float4(a.t[0] * p.x + a.t[1] * p.y + a.t[2] * p.z + a.t[3], a.t[4] * p.x + a.t[5] * p.y + a.t[6] * p.z + a.t[7],
                         a.t[8] * p.x + a.t[9] * p.y + a.t[10] * p.z + a.t[11], p.w);
  }
}

// ------------------------------------------------------------------------------------------------ LiDAR preprocessing
// Preprocess::process, non-feature branch (src/preprocess.cpp): driver records -> meas.lidar (pts / curv, input order).
//   PP_OUSTER     oust64_handler   :271-297
//   PP_VELO_TIME  velodyne_handler :417-473 with a time field (last point's time > 0, :322)
//   PP_VELO_YAW   velodyne_handler :417-473 without one: per-ring times synthesised from the yaw angle
//   PP_LIVOX      livox_handler    :178-204
// Every kernel writes a keep flag per raw point; an exclusive scan of the flags gives the output slot (order preserved).
enum PpMode { PP_OUSTER = 0, PP_VELO_TIME = 1, PP_VELO_YAW = 2, PP_LIVOX = 3 };

struct PpArgs {
  const unsigned char* rec;
  int stride, off_x, off_y, off_z, off_i, off_t, off_ring, off_tag, off_line;
  int n, n_scans, pfn;
  float time_scale;   // time_unit_scale (:65-82)
  double blind2;      // blind * blind
  double omega;       // omega_l = 0.361 * SCAN_RATE (:315)
};

__device__ __forceinline__ float pp_f32(const PpArgs& a, int i, int off) {
  return off >= 0 ? *reinterpret_cast<const float*>(a.rec + (size_t)i * a.stride + off) : 0.f;
}
__device__ __forceinline__ unsigned pp_u32(const PpArgs& a, int i, int off) {
  return off >= 0 ? *reinterpret_cast<const unsigned*>(a.rec + (size_t)i * a.stride + off) : 0u;
}
__device__ __forceinline__ unsigned pp_u16(const PpArgs& a, int i, int off) {
  return off >= 0 ? (unsigned)*reinterpret_cast<const unsigned short*>(a.rec + (size_t)i * a.stride + off) : 0u;
}
__device__ __forceinline__ unsigned pp_u8(const PpArgs& a, int i, int off) {
  return off >= 0 ? (unsigned)a.rec[(size_t)i * a.stride + off] : 0u;
}
__device__ __forceinline__ float3 pp_xyz(const PpArgs& a, int i) {
  return make_float3(pp_f32(a, i, a.off_x), pp_f32(a, i, a.off_y), pp_f32(a, i, a.off_z));
}
// x*x+y*y+z*z summed in float (the TU has no FMA contraction), compared in double with blind*blind
__device__ __forceinline__ float pp_r2(float3 p) { return p.x * p.x + p.y * p.y + p.z * p.z; }

// atan2f as glibc's libm computes it (the fdlibm single-precision algorithm: e_atan2f.c / s_atanf.c, 11-term
// polynomial), in IEEE float arithmetic (this TU has no FMA contraction; '/' is correctly rounded).  The reference
// calls the float overload (atan2(float, float) -> atan2f), so this reproduces its yaw angles bit for bit where the
// host libm is that implementation; a correctly rounded atan2 differs from it in the last bit for ~16 % of inputs.
__device__ __forceinline__ float pp_atanf_core(float x, unsigned hx) {
  const float atanhi[4] = {4.6364760399e-01f, 7.8539812565e-01f, 9.8279368877e-01f, 1.5707962513e+00f};
  const float atanlo[4] = {5.0121582440e-09f, 3.7748947079e-08f, 3.4473217170e-08f, 7.5497894159e-08f};
  const unsigned ix = hx & 0x7fffffffu;
  if (ix >= 0x4c000000u) {   // |x| >= 2^25
    if (ix > 0x7f800000u) return x + x;
    return (int)hx > 0 ? atanhi[3] + atanlo[3] : -atanhi[3] - atanlo[3];
  }
  int id;
  if (ix < 0x3ee00000u) {   // |x| < 0.4375
    if (ix < 0x31000000u) return x;
    id = -1;
  } else {
    x = fabsf(x);
    if (ix < 0x3f980000u) {
      if (ix < 0x3f300000u) { id = 0; x = (2.0f * x - 1.0f) / (2.0f + x); }
      else { id = 1; x = (x - 1.0f) / (x + 1.0f); }
    } else {
      if (ix < 0x401c0000u) { id = 2; x = (x - 1.5f) / (1.0f + 1.5f * x); }
      else { id = 3; x = -1.0f / x; }
    }
  }
  const float z = x * x, w = z * z;
  const float s1 = z * (3.3333334327e-01f + w * (1.4285714924e-01f + w * (9.0908870101e-02f + w * (6.6610731184e-02f +
                   w * (4.9768779427e-02f + w * 1.6285819933e-02f)))));
  const float s2 = w * (-2.0000000298e-01f + w * (-1.1111110449e-01f + w * (-7.6918758452e-02f + w * (-5.8335702866e-02f +
                   w * -3.6531571299e-02f))));
  if (id < 0) return x - x * (s1 + s2);
  const float r = atanhi[id] - ((x * (s1 + s2) - atanlo[id]) - x);
  return (int)hx < 0 ? -r : r;
}
__device__ __forceinline__ float pp_atan2f(float y, float x) {
  const float pi_o_4 = 7.8539818525e-01f, pi_o_2 = 1.5707963705e+00f, pi = 3.1415927410e+00f, pi_lo = -8.7422776573e-08f;
  const unsigned hx = __float_as_uint(x), hy = __float_as_uint(y), ix = hx & 0x7fffffffu, iy = hy & 0x7fffffffu;
  if (ix > 0x7f800000u || iy > 0x7f800000u) return x + y;
  if (hx == 0x3f800000u) return pp_atanf_core(y, hy);
  const int m = (int)(((hy >> 31) & 1u) | ((hx >> 30) & 2u));
  if (iy == 0) return m == 0 || m == 1 ? y : m == 2 ? pi : -pi;
  if (ix == 0) return (int)hy < 0 ? -pi_o_2 : pi_o_2;
  if (ix == 0x7f800000u) {
    if (iy == 0x7f800000u) return m == 0 ? pi_o_4 : m == 1 ? -pi_o_4 : m == 2 ? 3.0f * pi_o_4 : -3.0f * pi_o_4;
    return m == 0 ? 0.0f : m == 1 ? -0.0f : m == 2 ? pi : -pi;
  }
  if (iy == 0x7f800000u) return (int)hy < 0 ? -pi_o_2 : pi_o_2;
  const int k = ((int)iy - (int)ix) >> 23;
  float z;
  if (k > 60) z = pi_o_2 + 0.5f * pi_lo;
  else if ((int)hx < 0 && k < -60) z = 0.0f;
  else { const float q = fabsf(y / x); z = pp_atanf_core(q, __float_as_uint(q)); }
  switch (m) {
    case 0: return z;
    case 1: return -z;
    case 2: return pi - (z - pi_lo);
    default: return (z - pi_lo) - pi;
  }
}
// yaw_angle = atan2(added_pt.y, added_pt.x) * 57.2957 (:436): the float result widened to double
__device__ __forceinline__ double pp_yaw(float3 p) { return (double)pp_atan2f(p.y, p.x) * 57.2957; }

// ---- Velodyne without a time field.  Rings are grouped by a stable radix sort on the ring (keys = ring clamped to
// n_scans, vals = raw index), so a ring's points appear in raw order and its first sorted point is its first point.
__global__ void k_pp_ring_keys(PpArgs a, unsigned* __restrict__ keys, int* __restrict__ vals, unsigned* __restrict__ mm) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) {
    const unsigned r = pp_u16(a, i, a.off_ring);
    if (r >= (unsigned)a.n_scans) atomicMin(&mm[2], (unsigned)i);   // is_first[layer] out of bounds in the reference
    keys[i] = min(r, (unsigned)a.n_scans);
    vals[i] = i;
  }
}
__global__ void k_pp_ring_start(const unsigned* __restrict__ keys, int n, int* __restrict__ ring_start) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
    if (j == 0 || keys[j - 1] != keys[j]) ring_start[keys[j]] = j;
}
// c0[j] = the offset time before the wrap correction (:450-457) of sorted point j, rounded to float
__global__ void k_pp_yaw_c0(PpArgs a, const unsigned* __restrict__ keys, const int* __restrict__ vals,
                            const int* __restrict__ ring_start, float* __restrict__ c0) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
    const int h = ring_start[keys[j]];
    if (h == j) { c0[j] = 0.f; continue; }
    const double yaw = pp_yaw(pp_xyz(a, vals[j]));
    const double yaw_fp = pp_yaw(pp_xyz(a, vals[h]));
    c0[j] = yaw <= yaw_fp ? (float)((yaw_fp - yaw) / a.omega) : (float)((yaw_fp - yaw + 360.0) / a.omega);
  }
}

// The wrap rule (:459) "if (c < time_last) c += 360/omega" chains through a ring: time_last is the previous point's
// ADJUSTED value.  Point j's bump bit is a function of point j-1's bump bit, one of the four maps {0,1} -> {0,1},
// coded as bit0 = f(0), bit1 = f(1); bit2 marks a ring's first point, which restarts the chain (segmented scan).
__device__ __forceinline__ float pp_bump(float c, double omega) { return (float)((double)c + 360.0 / omega); }
__global__ void k_pp_yaw_codes(const unsigned* __restrict__ keys, const int* __restrict__ ring_start, const float* __restrict__ c0,
                               int n, double omega, unsigned* __restrict__ codes) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const int h = ring_start[keys[j]];
    unsigned code;
    if (h == j) {
      code = 4u;   // first point: time_last = 0, the point itself is dropped (:438-446)
    } else if (h == j - 1) {
      const unsigned b = c0[j] < 0.f ? 1u : 0u;   // compared with time_last = 0
      code = b | (b << 1);
    } else {
      const float p = c0[j - 1];
      code = (c0[j] < p ? 1u : 0u) | (c0[j] < pp_bump(p, omega) ? 2u : 0u);
    }
    codes[j] = code;
  }
}
struct PpChainOp {   // (earlier a) then (later b); a segment head in b discards a
  __host__ __device__ __forceinline__ unsigned operator()(unsigned a, unsigned b) const {
    if (b & 4u) return b;
    const unsigned f0 = (b >> (a & 1u)) & 1u, f1 = (b >> ((a >> 1) & 1u)) & 1u;
    return f0 | (f1 << 1) | (a & 4u);
  }
};
// t_raw[i] = the final offset time of raw point i (ring heads are dropped later and get 0)
__global__ void k_pp_yaw_apply(const int* __restrict__ vals, const float* __restrict__ c0, const unsigned* __restrict__ chain, int n,
                               double omega, float* __restrict__ t_raw) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
    t_raw[vals[j]] = (chain[j] & 1u) ? pp_bump(c0[j], omega) : c0[j];
}
__device__ __forceinline__ bool pp_is_ring_head(const PpArgs& a, int i, const int* ring_start, const int* vals) {
  const unsigned r = min(pp_u16(a, i, a.off_ring), (unsigned)a.n_scans);
  return vals[ring_start[r]] == i;
}

// ---- Livox: a point is valid when line < N_SCANS and the return tag is 0x00 / 0x10 (:184); points start at 1
__device__ __forceinline__ int pp_livox_valid(const PpArgs& a, int i) {
  if (i < 1) return 0;
  const unsigned tag = pp_u8(a, i, a.off_tag) & 0x30u;
  return (pp_u8(a, i, a.off_line) < (unsigned)a.n_scans && (tag == 0x10u || tag == 0x00u)) ? 1 : 0;
}
__global__ void k_pp_livox_valid(PpArgs a, int* __restrict__ valid) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) valid[i] = pp_livox_valid(a, i);
}
// selected: ++valid_num % point_filter_num == 0 (:186-188); valid_excl = exclusive scan of the valid flags
__device__ __forceinline__ bool pp_livox_selected(const PpArgs& a, int i, const int* valid, const int* valid_excl) {
  return i >= 1 && valid[i] && ((unsigned)(valid_excl[i] + 1) % (unsigned)a.pfn) == 0u;
}

// ---- keep flags, per mode
template <int MODE>
__global__ void k_pp_keep(PpArgs a, const int* __restrict__ aux0, const int* __restrict__ aux1, int* __restrict__ keep) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) {
    const float3 p = pp_xyz(a, i);
    bool k;
    if (MODE == PP_OUSTER) {
      k = (i % a.pfn == 0) && !((double)pp_r2(p) < a.blind2);
    } else if (MODE == PP_VELO_TIME) {
      k = (i % a.pfn == 0) && (double)pp_r2(p) > a.blind2;
    } else if (MODE == PP_VELO_YAW) {   // aux0 = ring_start, aux1 = vals (sorted position -> raw index)
      k = (i % a.pfn == 0) && !pp_is_ring_head(a, i, aux0, aux1) && (double)pp_r2(p) > a.blind2;
    } else {   // PP_LIVOX: aux0 = valid flags, aux1 = their exclusive scan
      k = pp_livox_selected(a, i, aux0, aux1);
      if (k) {
        // pl_full[i-1] is the previous raw point when it was selected, else the zero point of resize() (:190-197)
        float3 q = make_float3(0.f, 0.f, 0.f);
        if (pp_livox_selected(a, i - 1, aux0, aux1)) q = pp_xyz(a, i - 1);
        // :197 parses as  dx || dy || (dz && r2 > blind2)  -- kept literally; abs is the float overload
        k = ((double)fabsf(p.x - q.x) > 1e-7) || ((double)fabsf(p.y - q.y) > 1e-7) ||
            (((double)fabsf(p.z - q.z) > 1e-7) && ((double)pp_r2(p) > a.blind2));
      }
    }
    keep[i] = k ? 1 : 0;
  }
}

// ---- order-preserving compaction into the front end's (x,y,z,intensity) / curvature arrays
template <int MODE>
__global__ void k_pp_scatter(PpArgs a, const int* __restrict__ keep, const int* __restrict__ pos, const float* __restrict__ t_raw,
                             float4* __restrict__ out, float* __restrict__ out_curv, unsigned* __restrict__ mm) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += gridDim.x * blockDim.x) {
    const bool k = keep[i] != 0;
    if (i == a.n - 1) mm[0] = (unsigned)(pos[i] + (k ? 1 : 0));   // the output count
    if (!k) continue;
    const float3 p = pp_xyz(a, i);
    float in, c;
    if (MODE == PP_LIVOX) {
      in = (float)pp_u8(a, i, a.off_i);                    // intensity = reflectivity
      c = (float)pp_u32(a, i, a.off_t) / float(1000000);   // offset_time / float(1000000)
    } else {
      in = pp_f32(a, i, a.off_i);
      if (MODE == PP_OUSTER) c = (float)pp_u32(a, i, a.off_t) * a.time_scale;   // t * time_unit_scale
      else if (MODE == PP_VELO_TIME) c = pp_f32(a, i, a.off_t) * a.time_scale;  // time * time_unit_scale
      else c = t_raw[i];
    }
    out[pos[i]] = make_float4(p.x, p.y, p.z, in);
    out_curv[pos[i]] = c;
  }
}
// mm[1] = points.back().curvature (what sync_packages reads), float bits; 0 for an empty cloud
__global__ void k_pp_last(const float* __restrict__ out_curv, unsigned* __restrict__ mm) {
  const int cnt = (int)mm[0];
  mm[1] = cnt > 0 ? __float_as_uint(out_curv[cnt - 1]) : 0u;
}

}  // namespace flb
