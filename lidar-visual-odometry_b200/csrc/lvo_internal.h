// lvo_internal.h — context layout and helpers shared by the .cu translation units of liblvo.so.
//
// Data layout in HBM (DESIGN.md §3): every per-lane array lives at `base + lane * cap` inside one arena owned by
// the context; clouds are AoS float4 (x, y, z, intensity) so that one 128-bit load fetches a point.  All counts
// that depend on the data (n_kept, feature counts, map sizes, ...) stay on the device in `LaneState`; kernels are
// launched with capacity-derived grids and grid-stride over the device-side counts, so a whole frame is enqueued
// without a host round trip.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/lvo.h"
#include "lvo_math.h"

#define LVO_MAX_RINGS 64
#define LVO_SECTORS 6
#define LVO_MAX_OUTER 16
#define LVO_MAX_LM 8
#define LVO_TRACE_W 10
#define LVO_CUBE_W 21
#define LVO_CUBE_H 21
#define LVO_CUBE_D 11
#define LVO_NCUBES (LVO_CUBE_W * LVO_CUBE_H * LVO_CUBE_D)  // 4851, laserMapping.cpp:82
#define LVO_MAX_VALID 75                                     // 5 x 5 x 3, laserMapping.cpp:512-516
#define LVO_VSEGS (LVO_MAX_VALID + 1)                        // + one pseudo segment for inserts into non-valid cubes

// One residual block, the parameters of the reference functors (lidarFactor.hpp):
//   type 0 LidarEdgeFactor      : c = curr_point, a = last_point_a, b = (last_point_a - last_point_b) / |last_point_a - last_point_b| (the unit
//                                 direction of the edge, taken once when the record is written: the functor's residual
//                                 (lp - a) x (lp - b) / |a - b| equals (lp - a) x b' exactly, and its Jacobian with respect to lp is -[b']x,
//                                 so an evaluation needs no square root and no division), d = s (interpolation ratio; 1 unless DISTORTION)
//   type 1 LidarPlaneFactor     : c = curr_point, a = last_point_j, b = ljm_norm (unit normal, built at construction), d = s
//   type 2 LidarPlaneNormFactor : c = curr_point, a = plane_unit_norm, d = negative_OA_dot_norm
//   type -1 : no factor for this feature
struct __align__(16) LvoFactor {
  double c[3], a[3], b[3], d;
  int type, pad;
};
#ifdef __CUDACC__
// b slot of a type-0 record from the two line points (lidarFactor.hpp:36-37: de = lpa - lpb, de.norm())
__device__ __forceinline__ void lvo_edge_direction(const double* a, const double* b, double* e) {
  const double dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
  const double den = sqrt(dx * dx + dy * dy + dz * dz);
  e[0] = dx / den; e[1] = dy / den; e[2] = dz / den;
}
#endif

// Scalars of one lane that live on the device.
struct LaneState {
  // ---- extract
  int n_in, first_kept, last_kept, switch_idx, n_kept;
  float start_ori, end_ori;
  int ring_count[LVO_MAX_RINGS], ring_start[LVO_MAX_RINGS + 1];
  int scan_start[LVO_MAX_RINGS], scan_end[LVO_MAX_RINGS];
  int n_sharp, n_less_sharp, n_flat, n_less_flat;
  int n_lf_cand;                       // less-flat candidates before the per-ring voxel filter
  int lf_ring_off[LVO_MAX_RINGS + 1];  // offsets of the per-ring less-flat output
  // ---- odometry
  int odo_inited;
  double para_q[4], para_t[3];  // laserOdometry.cpp:131-133
  double q_w[4], t_w[3];        // laserOdometry.cpp:126-128
  int n_corner_last, n_surf_last;
  int corner_ring_first[LVO_MAX_RINGS + 2], surf_ring_first[LVO_MAX_RINGS + 2];
  int odo_status;
  // ---- mapping
  double map_x[7];              // parameters[7], laserMapping.cpp:110
  double q_wmap_wodom[4], t_wmap_wodom[3];
  double q_wodom[4], t_wodom[3];
  int cen[3];                   // laserCloudCen{Width,Height,Depth}
  int center[3];                // centerCubeI/J/K
  int shift[3];                 // pending cube shift of the stored map relative to `cen` (applied at rebuild)
  int n_valid, valid_cube[LVO_MAX_VALID];
  int from_off[2][LVO_MAX_VALID + 1];  // offsets of each valid cube inside corner/surf FromMap
  int n_stack[2];               // corner / surf stack sizes
  int n_map[2];                 // points stored in all cubes
  int map_status;
  int map_too_small;
  // ---- solver bookkeeping
  int n_factors;
  // LVO_OPT_FIXPOINT_SKIP: set by k_lm_solve when an outer iteration left the pose bit-for-bit unchanged; the association / fit /
  // solve kernels of the remaining outer iterations of this frame return at once for the lane (reset by k_odo_begin / k_map_begin)
  int odo_done, map_done;
  lvo_stats stats;
  int status;
};

// The sensor settings of one lane (lvo_lane_configure; lvo_create gives every lane the context's), one record per lane in device
// memory.  Not part of LaneState: a lane snapshot saves that struct verbatim, and its bytes must not change.
struct LaneConfig {
  int n_scans;   // 16 | 32 | 64, <= lvo_config::n_scans
  float thres;   // (float)minimum_range
  float leaf[2]; // (float)line_res, (float)plane_res (setLeafSize takes floats)
};

// Per-lane flags of a batched step, [lanes] ints uploaded right after the sweep counts (set_inputs in lvo_api.cu).  A lane without
// LVO_LANE_ACTIVE is idle (lvo_set_lane_active): every per-lane kernel leaves its state alone.  LVO_LANE_MAPS: the lane runs the
// mapping stage in this step (active and on its own skip_frame phase); the other lanes keep their map, poses and map correction.
// LVO_LANE_MAP_FIXED (set together with LVO_LANE_MAPS, lvo_set_lane_map_update): the lane registers against its map but inserts
// nothing and re-filters no cube; only the cube-window shift of this step changes its map.
#define LVO_LANE_ACTIVE 1
#define LVO_LANE_MAPS 2
#define LVO_LANE_MAP_FIXED 4

// Launch accounting (bench.py's gpu_launches) and error capture.
struct LvoLaunchCounter { long long launches; };

// Sub-stage timing under the reference's TicToc names (SURVEY §5 "tracing"): the launch functions mark stage boundaries with CUDA
// events on the launching stream (plain launches only; a null timer or a graph capture records nothing).  An interval runs from
// one mark to the next; after the stream has been synchronised collect() sums the intervals per stage.
enum LvoStage {
  LVO_ST_REG_PREPARE = 0,  // "prepare time"                   scanRegistration.cpp:254
  LVO_ST_REG_SORT,         // "sort q time"                    :409
  LVO_ST_REG_SEPARATE,     // "seperate points time"           :410
  LVO_ST_ODO_ASSOC,        // "data association time"          laserOdometry.cpp:564
  LVO_ST_ODO_SOLVER,       // "solver time"                    :577
  LVO_ST_ODO_REST,         // pose integration, cloud swap, kd-tree (grid) rebuild  :581-641
  LVO_ST_MAP_PREPARE,      // "map prepare time"               laserMapping.cpp:552
  LVO_ST_MAP_TREE,         // "build tree time"                :560
  LVO_ST_MAP_KNN,          // 5-NN part of "mapping data assosiation time" :710 (the graded kernel)
  LVO_ST_MAP_FIT,          // line / plane fits, the rest of :710
  LVO_ST_MAP_SOLVER,       // "mapping solver time"            :721
  LVO_ST_MAP_ADD,          // "add points time"                :784
  LVO_ST_MAP_FILTER,       // "filter time"                    :802
  LVO_ST_MAP_PUB,          // registered cloud ("mapping pub time" :850)
  LVO_ST_COUNT
};
struct LvoStageTimer {
  std::vector<cudaEvent_t> pool;
  std::vector<int> stage_of;   // stage that starts at event i (-1 = end marker)
  int used = 0;
  bool on = false;
  void reset() { used = 0; stage_of.clear(); }
  void mark(int stage, cudaStream_t st) {
    if (!on) return;
    if (used == (int)pool.size()) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) return; pool.push_back(e); }
    cudaEventRecord(pool[used++], st);
    stage_of.push_back(stage);
  }
  void stop(cudaStream_t st) { mark(-1, st); }
  // ms[LVO_ST_COUNT], count[LVO_ST_COUNT]; the stream must be idle
  void collect(float* ms, int* count) const {
    for (int i = 0; i < LVO_ST_COUNT; ++i) { ms[i] = 0.f; count[i] = 0; }
    for (int i = 0; i + 1 < used; ++i) {
      const int s = stage_of[i];
      if (s < 0) continue;
      float t = 0.f;
      if (cudaEventElapsedTime(&t, pool[i], pool[i + 1]) == cudaSuccess) { ms[s] += t; count[s]++; }
    }
  }
  void destroy() { for (cudaEvent_t e : pool) cudaEventDestroy(e); pool.clear(); used = 0; }
};
#define LVO_MARK(tm, stage, st) do { if (tm) (tm)->mark((stage), (st)); } while (0)

#define LVO_CUDA_OK(ctx, expr)                                                                          \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess) {                                                                            \
      lvo_set_error((ctx), std::string(#expr) + ": " + cudaGetErrorString(_e));                         \
      return LVO_E_CUDA;                                                                                \
    }                                                                                                   \
  } while (0)

struct lvo_ctx;
void lvo_set_error(lvo_ctx* ctx, const std::string& msg);

static inline int lvo_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------------------------
// Device helpers shared by all kernels
// ------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// the lane predicates of a batched step (flags: ExtractArgs / OdoArgs / MapArgs::lane_flags)
__device__ __forceinline__ bool lane_active(const int* flags, int lane) { return (__ldg(flags + lane) & LVO_LANE_ACTIVE) != 0; }
__device__ __forceinline__ bool lane_maps(const int* flags, int lane) { return (__ldg(flags + lane) & LVO_LANE_MAPS) != 0; }
// maps in this step and inserts into its map (lvo_set_lane_map_update on): the lanes that take part in the insertion + re-filter
__device__ __forceinline__ bool lane_updates_map(const int* flags, int lane) {
  return (__ldg(flags + lane) & (LVO_LANE_MAPS | LVO_LANE_MAP_FIXED)) == LVO_LANE_MAPS;
}

struct d3 { double x, y, z; };
__device__ __forceinline__ d3 d3cross(const d3& a, const d3& b) { return d3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
// Eigen 3.3.7 QuaternionBase::_transformVector: uv = vec x v; uv += uv; v + w*uv + vec x uv.  q = (x,y,z,w).
__device__ __forceinline__ d3 quat_rotate(const double* q, const d3& v) {
  d3 qv{q[0], q[1], q[2]};
  d3 uv = d3cross(qv, v);
  uv.x += uv.x; uv.y += uv.y; uv.z += uv.z;
  d3 c2 = d3cross(qv, uv);
  return d3{(v.x + q[3] * uv.x) + c2.x, (v.y + q[3] * uv.y) + c2.y, (v.z + q[3] * uv.z) + c2.z};
}
// Eigen generic quaternion product
__device__ __forceinline__ void quat_mul(const double* a, const double* b, double* r) {
  double w = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
  double x = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
  double y = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
  double z = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z; r[3] = w;
}
// pointAssociateToMap (laserMapping.cpp:154-163) / TransformToStart with s = 1 (laserOdometry.cpp:154-172):
// rotate + translate in double, round to float once.
__device__ __forceinline__ float4 transform_point(const double* q, const double* t, float4 p) {
  d3 r = quat_rotate(q, d3{(double)p.x, (double)p.y, (double)p.z});
  return make_float4((float)(r.x + t[0]), (float)(r.y + t[1]), (float)(r.z + t[2]), p.w);
}
// Eigen 3.3.7 QuaternionBase::slerp (Quaternion.h:716-746) of Identity towards q at parameter s: the blend weights of
// q_s = scale0 * Identity + scale1 * q, and their derivatives with respect to q.w (d = Identity.dot(q) = q.w), as forward-mode
// autodiff of the reference functors propagates them (lidarFactor.hpp:27-30,79-82).
struct SlerpW { double scale0, scale1, ds0_dw, ds1_dw; };
__device__ __forceinline__ SlerpW slerp_identity_weights(double w, double s, bool want_derivs) {
  SlerpW o{0.0, 0.0, 0.0, 0.0};
  const double one = 1.0 - 2.220446049250313e-16;
  const double absD = fabs(w);
  if (absD >= one) { o.scale0 = 1.0 - s; o.scale1 = s; }
  else {
    const double theta = acos(absD), sinTheta = sin(theta);
    const double a0 = (1.0 - s) * theta, a1 = s * theta;
    const double s0 = sin(a0), s1 = sin(a1);
    o.scale0 = s0 / sinTheta;
    o.scale1 = s1 / sinTheta;
    if (want_derivs) {
      const double cosTheta = cos(theta);
      const double dtheta_dw = (w < 0 ? 1.0 : -1.0) / sqrt(1.0 - absD * absD);
      o.ds0_dw = ((1.0 - s) * cos(a0) * sinTheta - s0 * cosTheta) / (sinTheta * sinTheta) * dtheta_dw;
      o.ds1_dw = (s * cos(a1) * sinTheta - s1 * cosTheta) / (sinTheta * sinTheta) * dtheta_dw;
    }
  }
  if (w < 0) { o.scale1 = -o.scale1; o.ds1_dw = -o.ds1_dw; }
  return o;
}
// interpolation ratio of a point, laserOdometry.cpp:157-161 / :455-459: float subtraction, double division by SCAN_PERIOD
__device__ __forceinline__ double distortion_ratio(float intensity, int distortion) {
  return distortion ? (double)(intensity - (float)int(intensity)) / 0.1 : 1.0;
}
// TransformToStart, laserOdometry.cpp:154-172.  distortion == 0: s = 1 and Identity.slerp(1, q) is exactly q.
__device__ __forceinline__ float4 transform_to_start(const double* q, const double* t, float4 p, int distortion) {
  if (!distortion) return transform_point(q, t, p);
  const double s = distortion_ratio(p.w, distortion);
  const SlerpW k = slerp_identity_weights(q[3], s, false);
  const double qs[4] = {k.scale0 * 0.0 + k.scale1 * q[0], k.scale0 * 0.0 + k.scale1 * q[1], k.scale0 * 0.0 + k.scale1 * q[2], k.scale0 * 1.0 + k.scale1 * q[3]};
  const d3 r = quat_rotate(qs, d3{(double)p.x, (double)p.y, (double)p.z});
  return make_float4((float)(r.x + s * t[0]), (float)(r.y + s * t[1]), (float)(r.z + s * t[2]), p.w);
}
// TransformToEnd, laserOdometry.cpp:176-191 (its call site :610-625 is disabled by `if (0)` in the reference; distortion mode 2 enables it)
__device__ __forceinline__ float4 transform_to_end(const double* q, const double* t, float4 p) {
  const float4 u = transform_to_start(q, t, p, 1);
  const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];   // Eigen inverse(): conjugate / squaredNorm
  const double qi[4] = {-q[0] / n2, -q[1] / n2, -q[2] / n2, q[3] / n2};
  const d3 e = quat_rotate(qi, d3{(double)u.x - t[0], (double)u.y - t[1], (double)u.z - t[2]});
  return make_float4((float)e.x, (float)e.y, (float)e.z, (float)int(p.w));
}
// FLANN L2_Simple accumulation order, no FMA (TU compiled with -fmad=false)
__device__ __forceinline__ float sqdist3(float4 a, float qx, float qy, float qz) {
  float dx = a.x - qx, dy = a.y - qy, dz = a.z - qz;
  return dx * dx + dy * dy + dz * dz;
}
// cube index of laserMapping.cpp:741-750: int((v + 25.0) / 50.0) + cen, minus one on the negative side
__device__ __forceinline__ int cube_coord(double v, int cen) {
  int c = int((v + 25.0) / 50.0) + cen;
  if (v + 25.0 < 0) c--;
  return c;
}
#endif  // __CUDACC__
