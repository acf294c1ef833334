// lvo_handlers.hpp — header-only C++ adaptor over the C ABI (include/lvo.h) with the shapes of the reference's three
// per-frame bodies, so that each of them can be replaced by one call:
//
//   lvo::ScanRegistration::laserCloudHandler   <- laserCloudHandler body      src/scanRegistration.cpp:127-411
//   lvo::LaserOdometry::process                <- odometry frame body         src/laserOdometry.cpp:353-641
//   lvo::LaserMapping::process                 <- mapping process() body      src/laserMapping.cpp:307-848
//
// `Cloud` is any type shaped like pcl::PointCloud<pcl::PointXYZI>: a public `points` container with data() / size() /
// resize() whose elements expose float x, y, z, intensity at fixed offsets (pcl::PointXYZI: stride 32, intensity at 16;
// lvo_point: stride 16, intensity at 12).  No PCL / ROS / Eigen header is needed here.
// Errors: negative liblvo codes become std::runtime_error (message from lvo_last_error); the reference's soft
// conditions (first frame, few correspondences, map too small) are returned as the positive LVO_W_* codes.
#pragma once
#include <cstddef>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/lvo.h"

namespace lvo {

struct Pose {  // quaternion (x, y, z, w) + translation, the layout of para_q/para_t and parameters[7]
  double q[4] = {0, 0, 0, 1};
  double t[3] = {0, 0, 0};
};

template <class Cloud>
inline lvo_cloud_view view_of(const Cloud& c) {
  typedef typename std::remove_reference<decltype(c.points[0])>::type P;
  lvo_cloud_view v;
  v.data = c.points.empty() ? nullptr : static_cast<const void*>(c.points.data());
  v.n = c.points.size();
  v.stride = sizeof(P);
  v.off_xyz = offsetof(P, x);
  v.off_intensity = offsetof(P, intensity);
  return v;
}

class Context {
 public:
  explicit Context(const lvo_config& cfg) {
    int r = lvo_create(&cfg, &ctx_);
    if (r != LVO_OK) {
      std::string msg = ctx_ ? lvo_last_error(ctx_) : "bad configuration";
      if (ctx_) lvo_destroy(ctx_);
      ctx_ = nullptr;
      throw std::runtime_error("lvo_create failed (" + std::to_string(r) + "): " + msg);
    }
    cap_ = cfg.max_points > 0 ? (size_t)cfg.max_points : 262144;
  }
  ~Context() { if (ctx_) lvo_destroy(ctx_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  lvo_ctx* get() const { return ctx_; }
  size_t capacity() const { return cap_; }
  int check(int r) const {
    if (r < 0) throw std::runtime_error(std::string("liblvo error ") + std::to_string(r) + ": " + lvo_last_error(ctx_));
    return r;
  }
  // HDL-64 / VLP-16 launch-file parameter sets (launch/aloam_velodyne_HDL_64.launch:3-13, _VLP_16.launch:3-13)
  static lvo_config hdl64() { lvo_config c; lvo_default_config(&c); return c; }
  static lvo_config vlp16() { lvo_config c; lvo_default_config(&c); c.n_scans = 16; c.minimum_range = 0.3; c.line_res = 0.2; c.plane_res = 0.4; return c; }

 private:
  lvo_ctx* ctx_ = nullptr;
  size_t cap_ = 0;
};

namespace detail {
// receive a packed lvo_point cloud into a Cloud with arbitrary point stride
template <class Cloud>
inline void store(const std::vector<lvo_point>& src, size_t n, Cloud& dst) {
  dst.points.resize(n);
  for (size_t i = 0; i < n; ++i) { dst.points[i].x = src[i].x; dst.points[i].y = src[i].y; dst.points[i].z = src[i].z; dst.points[i].intensity = src[i].intensity; }
}
}  // namespace detail

class ScanRegistration {
 public:
  explicit ScanRegistration(Context& c) : c_(c) { for (auto& b : buf_) b.resize(c.capacity()); }
  // in = /velodyne_points ; outputs = /velodyne_cloud_2, /laser_cloud_sharp, _less_sharp, _flat, _less_flat
  template <class Cloud>
  int laserCloudHandler(const Cloud& in, Cloud& laserCloud, Cloud& cornerPointsSharp, Cloud& cornerPointsLessSharp, Cloud& surfPointsFlat,
                        Cloud& surfPointsLessFlat) {
    lvo_cloud_out o[5];
    for (int k = 0; k < 5; ++k) { o[k].data = buf_[k].data(); o[k].cap = buf_[k].size(); o[k].n = 0; }
    int r = c_.check(lvo_extract_features(c_.get(), view_of(in), &o[0], &o[1], &o[2], &o[3], &o[4]));
    detail::store(buf_[0], o[0].n, laserCloud); detail::store(buf_[1], o[1].n, cornerPointsSharp); detail::store(buf_[2], o[2].n, cornerPointsLessSharp);
    detail::store(buf_[3], o[3].n, surfPointsFlat); detail::store(buf_[4], o[4].n, surfPointsLessFlat);
    return r;
  }

 private:
  Context& c_;
  std::vector<lvo_point> buf_[5];
};

namespace detail {
inline bool covariance(Context& c, int probe, double covariance[36]) {
  lvo_pose_uncertainty u;
  c.check(lvo_probe_fetch(c.get(), 0, probe, &u, sizeof(u), nullptr));
  for (int k = 0; k < 36; ++k) covariance[k] = u.covariance[k];
  return u.positive_definite != 0;
}
}  // namespace detail

class LaserOdometry {
 public:
  explicit LaserOdometry(Context& c) : c_(c) {}
  // returns LVO_W_FIRST_FRAME on the initialising frame; q_last_curr / q_w_curr as in laserOdometry.cpp:126-137
  template <class Cloud>
  int process(const Cloud& cornerPointsSharp, const Cloud& cornerPointsLessSharp, const Cloud& surfPointsFlat, const Cloud& surfPointsLessFlat,
              Pose& T_last_curr, Pose& T_w_curr) {
    lvo_pose a, b;
    int r = c_.check(lvo_scan_to_scan(c_.get(), view_of(cornerPointsSharp), view_of(cornerPointsLessSharp), view_of(surfPointsFlat),
                                      view_of(surfPointsLessFlat), &a, &b));
    for (int k = 0; k < 4; ++k) { T_last_curr.q[k] = a.q[k]; T_w_curr.q[k] = b.q[k]; }
    for (int k = 0; k < 3; ++k) { T_last_curr.t[k] = a.t[k]; T_w_curr.t[k] = b.t[k]; }
    return r;
  }
  // Distortion mode 2 only (lvo_config::distortion): the clouds that laserOdometry.cpp:646-662 would publish after the
  // TransformToEnd block :610-625 — call after process() and hand the results to LaserMapping::process.
  // cornerLast / surfLast were transformed on the device by process(); the full-resolution cloud is transformed here.
  template <class Cloud>
  void publishedClouds(Cloud& laserCloudCornerLast, Cloud& laserCloudSurfLast, Cloud& laserCloudFullRes) {
    if (buf_.size() < c_.capacity()) buf_.resize(c_.capacity());
    const int what[2] = {LVO_P_LESS_SHARP, LVO_P_LESS_FLAT};
    Cloud* dst[2] = {&laserCloudCornerLast, &laserCloudSurfLast};
    for (int k = 0; k < 2; ++k) {
      size_t bytes = 0;
      c_.check(lvo_probe_fetch(c_.get(), 0, what[k], buf_.data(), buf_.size() * sizeof(lvo_point), &bytes));
      detail::store(buf_, bytes / sizeof(lvo_point), *dst[k]);
    }
    lvo_cloud_out o;
    o.data = buf_.data(); o.cap = buf_.size(); o.n = 0;
    c_.check(lvo_transform_cloud(c_.get(), view_of(laserCloudFullRes), nullptr, 1, &o));
    detail::store(buf_, o.n, laserCloudFullRes);
  }
  // Covariance of T_last_curr from the last process() (lvo_pose_uncertainty::covariance, row-major 6 x 6 in (tx, ty, tz, rx, ry, rz),
  // the layout of nav_msgs::Odometry::pose.covariance): all zeros, and false, on the first frame or when the problem does not constrain
  // every direction (lvo_pose_uncertainty::positive_definite).
  bool motionCovariance(double covariance[36]) { return detail::covariance(c_, LVO_P_ODO_UNCERTAINTY, covariance); }

 private:
  Context& c_;
  std::vector<lvo_point> buf_;
};

class LaserMapping {
 public:
  explicit LaserMapping(Context& c) : c_(c), reg_(c.capacity()) {}
  // laserCloudFullRes is transformed in place into the map frame, as laserMapping.cpp:838-842 does
  template <class Cloud>
  int process(const Cloud& laserCloudCornerLast, const Cloud& laserCloudSurfLast, Cloud& laserCloudFullRes, const Pose& T_wodom_curr, Pose& T_w_curr) {
    lvo_pose in, out;
    for (int k = 0; k < 4; ++k) in.q[k] = T_wodom_curr.q[k];
    for (int k = 0; k < 3; ++k) in.t[k] = T_wodom_curr.t[k];
    lvo_cloud_out reg;
    reg.data = reg_.data(); reg.cap = reg_.size(); reg.n = 0;
    int r = c_.check(lvo_scan_to_map(c_.get(), view_of(laserCloudCornerLast), view_of(laserCloudSurfLast), view_of(laserCloudFullRes), &in, &out, &reg));
    for (int k = 0; k < 4; ++k) T_w_curr.q[k] = out.q[k];
    for (int k = 0; k < 3; ++k) T_w_curr.t[k] = out.t[k];
    detail::store(reg_, reg.n, laserCloudFullRes);
    frameCount_++;
    return r;
  }
  // The publication schedule of laserMapping.cpp:806-836 (frameCount is incremented at the end of process(), :854):
  // true when the frame just processed is one on which the reference publishes /laser_cloud_surround (every 5th)
  // or /laser_cloud_map (every 20th).
  bool surroundDue() const { return frameCount_ > 0 && (frameCount_ - 1) % 5 == 0; }
  bool mapDue() const { return frameCount_ > 0 && (frameCount_ - 1) % 20 == 0; }
  template <class Cloud>
  void laserCloudSurround(Cloud& out) { fetch(0, out); }   // :806-815
  template <class Cloud>
  void laserCloudMap(Cloud& out) { fetch(1, out); }        // :823-836
  // Localisation in a fixed prior map (lvo_set_lane_map_update): false skips the insertion and re-filter of :737-801 on the
  // following frames, so an imported map is registered against but not changed; true (the default) maps as the reference does.
  void setMapUpdate(bool update) { c_.check(lvo_set_lane_map_update(c_.get(), 0, update ? 1 : 0)); }
  // Covariance of T_w_curr from the last process(), for the pose.covariance of /aft_mapped_to_init (the reference leaves it zero);
  // same layout and return value as LaserOdometry::motionCovariance.
  bool poseCovariance(double covariance[36]) { return detail::covariance(c_, LVO_P_MAP_UNCERTAINTY, covariance); }

 private:
  template <class Cloud>
  void fetch(int which, Cloud& out) {
    lvo_cloud_out o;
    o.data = map_.data(); o.cap = map_.size(); o.n = 0;
    int r = lvo_map_cloud(c_.get(), 0, which, &o);
    if (r == LVO_E_CAPACITY) { map_.resize(o.n); o.data = map_.data(); o.cap = map_.size(); r = lvo_map_cloud(c_.get(), 0, which, &o); }
    c_.check(r);
    detail::store(map_, o.n, out);
  }
  Context& c_;
  std::vector<lvo_point> reg_, map_;
  long frameCount_ = 0;
};

}  // namespace lvo
