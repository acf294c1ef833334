// lvo_synth.cpp — deterministic synthetic lidar sweeps (SURVEY §8d).  Host-only helper for tests and bench.py;
// it replaces the reference's KITTI feeder (src/kittiHelper.cpp, out of scope) with a procedural scene so that
// the hot path can be exercised without datasets.
//
// Sensor models
//   64 : HDL-64-shaped.  64 beams, elevations 1.95 - i/3 deg (i < 32) and -8.88 - 0.5 i deg (i < 32), chosen to sit
//        inside the ring bins of reference src/scanRegistration.cpp:189-192; 1875 azimuth steps => 120 000 rays.
//   16 : VLP-16-shaped.  16 beams -15..+15 deg step 2 (:171); 1800 azimuth steps => 28 800 rays.
// Rays are emitted azimuth-major and clockwise (ori = -atan2(y, x) increasing, as :208 expects) and cast from the
// sensor pose into an endless procedural street: ground plane, two facades with hashed recesses (vertical edges),
// poles, boxes.  Range noise N(0, 0.01 m); rays without a return inside 120 m are dropped.
// The trajectory is KITTI-00-shaped: `speed` m/frame forward with an S-curve yaw and a small roll/pitch/z wobble,
// applied rigidly per sweep (no intra-sweep distortion, consistent with DISTORTION 0, laserOdometry.cpp:67) by
// lvo_synth_sweep; lvo_synth_sweep_moving casts every azimuth column from the pose interpolated between frame and frame + 1
// (a spinning sensor on a moving platform: the input DISTORTION 1 is written for).
#include <cmath>
#include <cstdint>
#include <cstring>

namespace {

struct P4 { float x, y, z, i; };

inline uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
inline double u01(uint64_t h) { return ((h >> 11) + 0.5) * (1.0 / 9007199254740992.0); }
inline uint64_t hash3(uint64_t a, uint64_t b, uint64_t c) { return mix64(mix64(mix64(a) ^ b) ^ c); }

struct Scene {
  uint64_t seed;
  double ground_z = -1.73;
  double wall_y = 8.0, seg_len = 4.0;
  bool features = true;   // false: ground and two flat facades only (a tunnel: translation along x is unobservable)
  double recess(long k, int side) const {
    if (!features) return 0.0;
    uint64_t h = hash3(seed, (uint64_t)(k + (1l << 40)), (uint64_t)(side + 7));
    int r = (int)(h % 5);
    return r == 0 ? 1.2 : (r == 1 ? 0.6 : 0.0);
  }
  // first hit of a ray with one facade (side = +1: y > 0, -1: y < 0)
  double hit_facade(const double o[3], const double d[3], int side) const {
    double oy = side * o[1], dy = side * d[1];
    if (dy <= 1e-12) return INFINITY;
    double t = (wall_y - oy) / dy;
    if (t < 0) t = 0;
    for (int it = 0; it < 200; ++it) {
      double x = o[0] + t * d[0];
      long k = (long)std::floor(x / seg_len);
      double Yk = wall_y + recess(k, side);
      double tw = (Yk - oy) / dy;
      double xw = o[0] + tw * d[0];
      if (xw >= k * seg_len && xw <= (k + 1) * seg_len) return tw;
      if (std::fabs(d[0]) < 1e-12) return tw;
      // leave the segment through a side boundary
      double xb = d[0] > 0 ? (k + 1) * seg_len : k * seg_len;
      long kn = d[0] > 0 ? k + 1 : k - 1;
      double tb = (xb - o[0]) / d[0];
      double yb = oy + tb * dy;
      double Yn = wall_y + recess(kn, side);
      if (yb >= Yn) return tb;  // side wall between a deeper and a shallower segment
      t = tb + 1e-9;
      if (t > 400.0) return INFINITY;
    }
    return INFINITY;
  }
  double hit_poles(const double o[3], const double d[3], double tmax) const {
    double best = INFINITY;
    const double R = 0.15, spacing = 10.0, top = 6.0;
    double dd = d[0] * d[0] + d[1] * d[1];
    if (dd < 1e-14) return best;
    double xr = std::fabs(d[0]) * tmax;
    long m0 = (long)std::floor((o[0] - xr) / spacing) - 1, m1 = (long)std::ceil((o[0] + xr) / spacing) + 1;
    if (m1 - m0 > 40) { m0 = (long)std::floor(o[0] / spacing) - 20; m1 = m0 + 40; }
    for (long m = m0; m <= m1; ++m)
      for (int side = -1; side <= 1; side += 2) {
        uint64_t h = hash3(seed ^ 0x51, (uint64_t)(m + (1l << 40)), (uint64_t)(side + 3));
        double cx = m * spacing + (u01(h) - 0.5) * 4.0;
        double cy = side * (5.2 + u01(mix64(h)) * 0.8);
        double fx = o[0] - cx, fy = o[1] - cy;
        double b = fx * d[0] + fy * d[1];
        double c = fx * fx + fy * fy - R * R;
        double disc = b * b - dd * c;
        if (disc < 0) continue;
        double t = (-b - std::sqrt(disc)) / dd;
        if (t <= 0 || t >= best) continue;
        double z = o[2] + t * d[2];
        if (z < ground_z || z > top) continue;
        best = t;
      }
    return best;
  }
  double hit_boxes(const double o[3], const double d[3], double tmax) const {
    double best = INFINITY;
    const double spacing = 25.0;
    double xr = std::fabs(d[0]) * tmax;
    long m0 = (long)std::floor((o[0] - xr) / spacing) - 1, m1 = (long)std::ceil((o[0] + xr) / spacing) + 1;
    if (m1 - m0 > 16) { m0 = (long)std::floor(o[0] / spacing) - 8; m1 = m0 + 16; }
    for (long m = m0; m <= m1; ++m)
      for (int side = -1; side <= 1; side += 2) {
        uint64_t h = hash3(seed ^ 0xB0, (uint64_t)(m + (1l << 40)), (uint64_t)(side + 3));
        double cx = m * spacing + (u01(h) - 0.5) * 10.0;
        double cy = side * (6.3 + u01(mix64(h)) * 0.6);
        double lo[3] = {cx - 2.1, cy - 0.9, ground_z}, hi[3] = {cx + 2.1, cy + 0.9, ground_z + 1.5};
        double t0 = 0, t1 = best;
        bool ok = true;
        for (int a = 0; a < 3 && ok; ++a) {
          if (std::fabs(d[a]) < 1e-14) { if (o[a] < lo[a] || o[a] > hi[a]) ok = false; continue; }
          double ta = (lo[a] - o[a]) / d[a], tb = (hi[a] - o[a]) / d[a];
          if (ta > tb) { double s = ta; ta = tb; tb = s; }
          if (ta > t0) t0 = ta;
          if (tb < t1) t1 = tb;
          if (t0 > t1) ok = false;
        }
        if (ok && t0 > 0 && t0 < best) best = t0;
      }
    return best;
  }
  double cast(const double o[3], const double d[3]) const {
    double t = INFINITY;
    if (d[2] < -1e-12) t = (ground_z - o[2]) / d[2];
    double tf = hit_facade(o, d, +1); if (tf < t) t = tf;
    tf = hit_facade(o, d, -1); if (tf < t) t = tf;
    if (!features) return t;
    double lim = t < 130.0 ? t : 130.0;
    double tp = hit_poles(o, d, lim); if (tp < t) t = tp;
    double tb = hit_boxes(o, d, lim); if (tb < t) t = tb;
    return t;
  }
};

struct Pose { double R[9]; double t[3]; double q[4]; };

// x, y, z, yaw, pitch, roll of the sensor at an integer frame
void pose_params(int seq, int frame, double speed, double p[6]) {
  // integrate the planar path
  double x = 0, y = 0;
  const double A = 10.0 * M_PI / 180.0, T = 80.0;
  double phase = 0.37 * seq;
  for (int k = 0; k < frame; ++k) {
    double yaw = A * std::sin(2 * M_PI * k / T + phase);
    x += speed * std::cos(yaw); y += speed * std::sin(yaw);
  }
  p[0] = x; p[1] = y;
  p[2] = 0.05 * std::sin(frame / 13.0 + 0.5 * seq);
  p[3] = A * std::sin(2 * M_PI * frame / T + phase);
  p[4] = 0.3 * M_PI / 180.0 * std::sin(frame / 11.0 + 2.0 * seq);
  p[5] = 0.5 * M_PI / 180.0 * std::sin(frame / 7.0 + seq);
}
void pose_from_params(const double p[6], Pose& P) {
  const double x = p[0], y = p[1], z = p[2], yaw = p[3], pitch = p[4], roll = p[5];
  double cy = std::cos(yaw), sy = std::sin(yaw), cp = std::cos(pitch), sp = std::sin(pitch), cr = std::cos(roll), sr = std::sin(roll);
  // R = Rz(yaw) Ry(pitch) Rx(roll)
  double R[9] = {cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                 sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                 -sp,     cp * sr,                cp * cr};
  std::memcpy(P.R, R, sizeof(R));
  P.t[0] = x; P.t[1] = y; P.t[2] = z;
  // quaternion (x,y,z,w) from yaw/pitch/roll
  double hy = yaw / 2, hp = pitch / 2, hr = roll / 2;
  double cyh = std::cos(hy), syh = std::sin(hy), cph = std::cos(hp), sph = std::sin(hp), crh = std::cos(hr), srh = std::sin(hr);
  P.q[3] = crh * cph * cyh + srh * sph * syh;
  P.q[0] = srh * cph * cyh - crh * sph * syh;
  P.q[1] = crh * sph * cyh + srh * cph * syh;
  P.q[2] = crh * cph * syh - srh * sph * cyh;
}
void pose_of(int seq, int frame, double speed, Pose& P) {
  double p[6];
  pose_params(seq, frame, speed, p);
  pose_from_params(p, P);
}

}  // namespace

extern "C" {

// Number of rays of a sensor model (upper bound of the points a sweep can contain).
long lvo_synth_rays(int model) { return model == 16 ? 16L * 1800 : 64L * 1875; }

}  // extern "C"

// Generates sweep `frame` of sequence `seq` into out[cap] (packed x,y,z,intensity=0).  gt_pose7 (optional) gets the
// ground-truth sensor pose (q xyzw, t) in the frame of sweep 0 of the same sequence.  Returns the number of points,
// or -1 if cap is too small / the model is unknown.
// naz = azimuth columns per sweep (0: the model's default).
static long synth_sweep(int model, int seq, int frame, double speed, float* out_xyzi, long cap, double* gt_pose7, bool moving, int naz = 0,
                        bool features = true) {
  if (model != 16 && model != 64) return -1;
  const int beams = model;
  if (naz == 0) naz = model == 16 ? 1800 : 1875;
  if (naz < 1 || cap < (long)beams * naz) return -1;
  Scene sc;
  sc.seed = 1000ull * (uint64_t)model + 10ull * (uint64_t)seq;
  sc.features = features;
  Pose P, P0;
  double pa[6], pb[6];
  pose_params(seq, frame, speed, pa);
  pose_params(seq, frame + 1, speed, pb);
  // ground truth: rigid sweeps -> pose at `frame` relative to frame 0; moving sensor -> pose at the END of the sweep relative to
  // the end of sweep 0 (what q_w_curr / t_w_curr accumulate when the clouds are moved to the sweep end, laserOdometry.cpp:176-191)
  pose_of(seq, moving ? frame + 1 : frame, speed, P);
  pose_of(seq, moving ? 1 : 0, speed, P0);
  if (gt_pose7) {
    // relative pose T0^-1 * T  (frame 0 is the odometry / map origin, laserOdometry.cpp:126-128)
    double Rr[9], tr[3], dt[3] = {P.t[0] - P0.t[0], P.t[1] - P0.t[1], P.t[2] - P0.t[2]};
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += P0.R[k * 3 + r] * P.R[k * 3 + c]; Rr[r * 3 + c] = s; }
      tr[r] = P0.R[0 * 3 + r] * dt[0] + P0.R[1 * 3 + r] * dt[1] + P0.R[2 * 3 + r] * dt[2];
    }
    // rotation matrix -> quaternion
    double tr_ = Rr[0] + Rr[4] + Rr[8], qw, qx, qy, qz;
    if (tr_ > 0) { double s = std::sqrt(tr_ + 1.0) * 2; qw = 0.25 * s; qx = (Rr[7] - Rr[5]) / s; qy = (Rr[2] - Rr[6]) / s; qz = (Rr[3] - Rr[1]) / s; }
    else if (Rr[0] > Rr[4] && Rr[0] > Rr[8]) { double s = std::sqrt(1.0 + Rr[0] - Rr[4] - Rr[8]) * 2; qw = (Rr[7] - Rr[5]) / s; qx = 0.25 * s; qy = (Rr[1] + Rr[3]) / s; qz = (Rr[2] + Rr[6]) / s; }
    else if (Rr[4] > Rr[8]) { double s = std::sqrt(1.0 + Rr[4] - Rr[0] - Rr[8]) * 2; qw = (Rr[2] - Rr[6]) / s; qx = (Rr[1] + Rr[3]) / s; qy = 0.25 * s; qz = (Rr[5] + Rr[7]) / s; }
    else { double s = std::sqrt(1.0 + Rr[8] - Rr[0] - Rr[4]) * 2; qw = (Rr[3] - Rr[1]) / s; qx = (Rr[2] + Rr[6]) / s; qy = (Rr[5] + Rr[7]) / s; qz = 0.25 * s; }
    gt_pose7[0] = qx; gt_pose7[1] = qy; gt_pose7[2] = qz; gt_pose7[3] = qw;
    gt_pose7[4] = tr[0]; gt_pose7[5] = tr[1]; gt_pose7[6] = tr[2];
  }
  const double step = 2 * M_PI / naz;
  // start azimuth differs per sequence so that the halfPassed state machine (:209-236) sees different phases
  const double az0 = M_PI - 0.5 * step - (seq % 4) * (M_PI / 2.0) * 0.97;
  const double min_keep = 0.05, max_range = 120.0, sigma = 0.01;
  long n = 0;
  P4* out = reinterpret_cast<P4*>(out_xyzi);
  if (!moving) pose_from_params(pa, P);
  for (int j = 0; j < naz; ++j) {
    if (moving) {
      const double tau = (double)j / naz;
      double pi[6];
      for (int k = 0; k < 6; ++k) pi[k] = pa[k] + tau * (pb[k] - pa[k]);
      pose_from_params(pi, P);
    }
    double az = az0 - j * step;
    double ca = std::cos(az), sa = std::sin(az);
    for (int b = 0; b < beams; ++b) {
      double el_deg = model == 16 ? (-15.0 + 2.0 * b) : (b < 32 ? 1.95 - b / 3.0 : -8.88 - 0.5 * (b - 32));
      double el = el_deg * M_PI / 180.0;
      double ce = std::cos(el), se = std::sin(el);
      double ds[3] = {ce * ca, ce * sa, se};
      double dw[3] = {P.R[0] * ds[0] + P.R[1] * ds[1] + P.R[2] * ds[2], P.R[3] * ds[0] + P.R[4] * ds[1] + P.R[5] * ds[2],
                      P.R[6] * ds[0] + P.R[7] * ds[1] + P.R[8] * ds[2]};
      double t = sc.cast(P.t, dw);
      if (!(t < max_range) || t < min_keep) continue;
      uint64_t h = hash3(sc.seed ^ 0xABCDEF, (uint64_t)frame, (uint64_t)j * 64 + (uint64_t)b);
      double u1 = u01(h), u2 = u01(mix64(h));
      double g = std::sqrt(-2.0 * std::log(u1)) * std::cos(2 * M_PI * u2);
      double r = t + sigma * g;
      out[n].x = (float)(r * ds[0]); out[n].y = (float)(r * ds[1]); out[n].z = (float)(r * ds[2]); out[n].i = 0.f;
      ++n;
    }
  }
  return n;
}

extern "C" {
long lvo_synth_sweep(int model, int seq, int frame, double speed, float* out_xyzi, long cap, double* gt_pose7) {
  return synth_sweep(model, seq, frame, speed, out_xyzi, cap, gt_pose7, false);
}
// Same scene and trajectory, but the sensor keeps moving while it spins: column j of the sweep is cast from the pose at time
// frame + j / naz.  gt_pose7 = pose at the end of the sweep relative to the end of sweep 0.
long lvo_synth_sweep_moving(int model, int seq, int frame, double speed, float* out_xyzi, long cap, double* gt_pose7) {
  return synth_sweep(model, seq, frame, speed, out_xyzi, cap, gt_pose7, true);
}
// Same scene and trajectory as lvo_synth_sweep with `naz` azimuth columns per ring (0: the model's default): dense rings of sensors
// that spin slower or fire faster, e.g. a VLP-16 at 5 Hz (~3600 columns).  out[cap] needs model * naz entries.
long lvo_synth_sweep_res(int model, int seq, int frame, double speed, int naz, float* out_xyzi, long cap, double* gt_pose7) {
  return synth_sweep(model, seq, frame, speed, out_xyzi, cap, gt_pose7, false, naz);
}
// Same beam pattern, trajectory and noise as lvo_synth_sweep, cast into the same street with its recesses, poles and boxes removed:
// the ground plane and two flat facades, parallel to the world x axis.  Translation along the street is unobservable there, the
// degenerate case of a straight tunnel or corridor.  street_axis3 (optional) gets the world x axis in the sensor frame of sweep 0 (the
// odometry and map origin).
long lvo_synth_sweep_tunnel(int model, int seq, int frame, double speed, float* out_xyzi, long cap, double* gt_pose7, double* street_axis3) {
  if (street_axis3) {
    Pose P0;
    pose_of(seq, 0, speed, P0);
    for (int r = 0; r < 3; ++r) street_axis3[r] = P0.R[0 * 3 + r];   // R0^T e_x
  }
  return synth_sweep(model, seq, frame, speed, out_xyzi, cap, gt_pose7, false, 0, false);
}

}  // extern "C"
