// lvo_depth.cuh — camera-lidar depth association (BASELINE config 5, SURVEY §8a rows A28-A29).
// One call solves one problem ("slot") per lane, all slots in one launch sequence whose length does not depend on the number of slots:
//   k_depth_flag / k_depth_write : the sweep through the slot's 3x4 lidar->camera extrinsic (pcl::transformPointCloud, reference
//                                  src/vloam/CamLidarProcess.cpp:249-253) and the depth cloud of src/vloam/Frame.cpp:328-336:
//                                  every point with z > 0 becomes (10 x / z, 10 y / z, 10, I = z), order preserved
//                                  (flag -> ONE exclusive scan over the packed sweeps of all slots -> scatter); the depth clouds of
//                                  the slots lie back to back, in slot order
//   k_depth_setup                : per slot, the offset and size of its depth cloud (from the scan) and its grid problem
//   lvo_grid_build               : one 2-D uniform grid per slot over the clamped image plane (replaces kdTree_->setInputCloud,
//                                  Frontend.cpp:466)
//   k_depth_assoc                : one warp per keypoint over the keypoints of all slots: exact 3-NN of (10 u, 10 v, 10) in its slot's
//                                  depth cloud (Frontend.cpp:233-241), gate d0^2 < 0.5 (:245), planar interpolation through the three
//                                  points in double (:247-270) and the clamps of :274-293
#pragma once
#include "lvo_internal.h"
#include "lvo_knn.cuh"

// image-plane grid of a slot: 0.125-unit cells over |x|, |y| <= 16 (the cloud is in 10 x normalised coordinates); 257 x 257 cells
// hold the whole clamp box, so the cell edge never has to grow
#define LVO_DEPTH_CELL 0.125f
#define LVO_DEPTH_CLAMP 16.0f
#define LVO_DEPTH_CELLS (257 * 257)

// One lane's problem, device-resident.
struct DepthSlot {
  const unsigned char* pts;          // sweep records (DepthArgs::stride / off_xyz)
  const float* uv;                   // keypoints, normalised coordinates [nkp][2]
  float* depth; int* valid; int* nn; // outputs [nkp], [nkp], [nkp][3] (nn may be null)
  float extr[12];                    // 3x4 row-major lidar -> camera
  unsigned pt_off; int n;            // the sweep's offset in the packed flag array, its point count
  unsigned kp_off; int nkp;          // the keypoints' offset in the packed keypoint sequence, their count
};

struct DepthArgs {
  const DepthSlot* slot; int nslot;  // [nslot] (device)
  int stride, off_xyz;               // record layout shared by all slots (x, y, z floats at off_xyz)
  int n_total, kp_total;             // sum of the slots' n / nkp
  unsigned* flag;                    // [n_total] -> exclusive scan: position in dc
  int* d_n;                          // device copy of n_total (scan length)
  unsigned* d_total;                 // depth-cloud points of all slots (scan total)
  unsigned* dc_off; int* ndc;        // [nslot] offset of a slot's depth cloud in dc, its size
  float4* dc;                        // depth clouds out
  GridSet grid;                      // problem s = slot s's depth cloud
};

__device__ __forceinline__ float3 cam_point(const float* e, const unsigned char* rec) {
  const float* p = reinterpret_cast<const float*>(rec);
  const float x = p[0], y = p[1], z = p[2];
  return make_float3(((e[0] * x + e[1] * y) + e[2] * z) + e[3], ((e[4] * x + e[5] * y) + e[6] * z) + e[7], ((e[8] * x + e[9] * y) + e[10] * z) + e[11]);
}
// grid (gx, nslot): blockIdx.y = slot
__global__ void k_depth_flag(DepthArgs a) {
  const DepthSlot& s = a.slot[blockIdx.y];
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *a.d_n = a.n_total;
  float e[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) e[k] = s.extr[k];
  const unsigned char* base = s.pts + a.off_xyz;
  unsigned* flag = a.flag + s.pt_off;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < s.n; i += gridDim.x * blockDim.x) flag[i] = cam_point(e, base + (size_t)i * a.stride).z > 0.0 ? 1u : 0u;
}
__global__ void k_depth_write(DepthArgs a) {
  const DepthSlot& s = a.slot[blockIdx.y];
  float e[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) e[k] = s.extr[k];
  const unsigned char* base = s.pts + a.off_xyz;
  const unsigned* flag = a.flag + s.pt_off;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < s.n; i += gridDim.x * blockDim.x) {
    const float3 c = cam_point(e, base + (size_t)i * a.stride);
    if (c.z > 0.0) a.dc[flag[i]] = make_float4(c.x * 10.f / c.z, c.y * 10.f / c.z, 10.f, c.z);   // Frame.cpp:330-336
  }
}
// one thread per slot: the slot's depth cloud starts at the scanned flag of its first point (slots without points: at the next slot's)
__global__ void k_depth_setup(DepthArgs a) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.nslot) return;
  const unsigned tot = *a.d_total;
  const unsigned o0 = a.slot[s].pt_off, o1 = s + 1 < a.nslot ? a.slot[s + 1].pt_off : (unsigned)a.n_total;
  const unsigned b0 = o0 < (unsigned)a.n_total ? a.flag[o0] : tot, b1 = o1 < (unsigned)a.n_total ? a.flag[o1] : tot;
  a.dc_off[s] = b0; a.ndc[s] = (int)(b1 - b0);
  GridProblem& q = a.grid.prob[s];
  q.pts = a.dc + b0; q.d_n = a.ndc + s; q.want_cell = LVO_DEPTH_CELL; q.want_cell_z = 0.f; q.mode = 0; q.cells_cap = 0; q.clamp_xy = LVO_DEPTH_CLAMP; q.bbox_from = -1;
}

__global__ void __launch_bounds__(256) k_depth_assoc(DepthArgs a) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  const unsigned ln = threadIdx.x & 31;
  for (int k = wid; k < a.kp_total; k += nw) {
    // the keypoint's slot: the last one whose keypoints start at or before k (a slot without keypoints shares its offset with the next)
    int sl = 0, hi = a.nslot - 1;
    while (sl < hi) { const int mid = (sl + hi + 1) >> 1; if (a.slot[mid].kp_off <= (unsigned)k) sl = mid; else hi = mid - 1; }
    const DepthSlot& S = a.slot[sl];
    const int j = k - (int)S.kp_off;
    const GridView g = grid_view(a.grid, sl);
    const int ndc = a.ndc[sl];
    const float4* dc = a.dc + a.dc_off[sl];
    const float u = S.uv[2 * j], v = S.uv[2 * j + 1];
    const float qx = 10 * u, qy = 10 * v, qz = 10.f;
    TopK<3> tk;
    tk.init();
    bool found = false;
    if (g.dim[0] > 0 && ndc >= 3) {
      // the query's cell is clamped into the table like the points': a query outside the clamp box starts in the border
      // cell that holds the outside points, and all ring bounds stay valid (true distances only grow)
      const int cx = min(max(cell_coord(qx, g.inv_cell) - g.org[0], 0), g.dim[0] - 1), cy = min(max(cell_coord(qy, g.inv_cell) - g.org[1], 0), g.dim[1] - 1);
      for (int dy = -1; dy <= 1; ++dy) scan_row<3>(g, 0, cy + dy, cx - 1, cx + 1, qx, qy, qz, tk, ln);
      warp_merge<3>(tk);
      // grow the search square ring by ring (all depth points share z = 10: the grid has one layer)
      const int rmax = max(g.dim[0], g.dim[1]) + 1;
      for (int r = 2; r <= rmax; ++r) {
        const float bound = (float)(r - 1) * g.cell, b2 = bound * bound;
        if (tk.id[2] != INT_MAX && tk.d[2] < b2) break;   // the three nearest are final
        if (!(tk.d[0] < 0.5f) && b2 >= 0.5f) break;        // the gate on the nearest point can no longer pass
        scan_row<3>(g, 0, cy - r, cx - r, cx + r, qx, qy, qz, tk, ln);
        scan_row<3>(g, 0, cy + r, cx - r, cx + r, qx, qy, qz, tk, ln);
        for (int dy = -r + 1; dy <= r - 1; ++dy) {
          scan_row<3>(g, 0, cy + dy, cx - r, cx - r, qx, qy, qz, tk, ln);
          scan_row<3>(g, 0, cy + dy, cx + r, cx + r, qx, qy, qz, tk, ln);
        }
        warp_merge<3>(tk);
      }
      found = tk.id[2] != INT_MAX && tk.d[0] < 0.5f;      // Frontend.cpp:245
    }
    if (ln == 0) {
      float s = 0.f; int ok = 0;
      int nn[3] = {-1, -1, -1};
      if (found) {
        nn[0] = tk.id[0]; nn[1] = tk.id[1]; nn[2] = tk.id[2];
        float4 dp = dc[tk.id[0]];
        const double x1 = dp.x * dp.w / 10, y1 = dp.y * dp.w / 10, z1 = dp.w;
        double minDepth = z1, maxDepth = z1;
        dp = dc[tk.id[1]];
        const double x2 = dp.x * dp.w / 10, y2 = dp.y * dp.w / 10, z2 = dp.w;
        minDepth = (z2 < minDepth) ? z2 : minDepth; maxDepth = (z2 > maxDepth) ? z2 : maxDepth;
        dp = dc[tk.id[2]];
        const double x3 = dp.x * dp.w / 10, y3 = dp.y * dp.w / 10, z3 = dp.w;
        minDepth = (z3 < minDepth) ? z3 : minDepth; maxDepth = (z3 > maxDepth) ? z3 : maxDepth;
        const double uu = u, vv = v;
        s = (float)((x1 * y2 * z3 - x1 * y3 * z2 - x2 * y1 * z3 + x2 * y3 * z1 + x3 * y1 * z2 - x3 * y2 * z1) /
                    (x1 * y2 - x2 * y1 - x1 * y3 + x3 * y1 + x2 * y3 - x3 * y2 + uu * y1 * z2 - uu * y2 * z1 - vv * x1 * z2 + vv * x2 * z1 - uu * y1 * z3 +
                     uu * y3 * z1 + vv * x1 * z3 - vv * x3 * z1 + uu * y2 * z3 - uu * y3 * z2 - vv * x2 * z3 + vv * x3 * z2));   // :270
        ok = 1;
        if (!isfinite(s)) { s = (float)z1; ok = 1; }
        if (maxDepth - minDepth > 2) { s = 0; ok = 0; }
        else if (s - maxDepth > 0.2) s = (float)maxDepth;
        else if (s - minDepth < -0.2) s = (float)minDepth;
      }
      S.depth[j] = s; S.valid[j] = ok;
      if (S.nn) { S.nn[3 * j] = nn[0]; S.nn[3 * j + 1] = nn[1]; S.nn[3 * j + 2] = nn[2]; }
    }
  }
}

// The launch sequence of one call (16 launches, whatever the number of slots and keypoints).  max_n: the largest n of a slot.
static inline void lvo_launch_depth(cudaStream_t st, const DepthArgs& a, int max_n, const LvoScanScratch& scan, long long* launches) {
  const dim3 gp(max(1, min(lvo_div_up(max_n, 256), max(24, 2368 / a.nslot))), a.nslot);
  k_depth_flag<<<gp, 256, 0, st>>>(a);
  lvo_scan_exclusive(st, a.flag, a.d_n, max(a.n_total, 1), a.d_total, scan, launches);
  k_depth_write<<<gp, 256, 0, st>>>(a);
  k_depth_setup<<<lvo_div_up(a.nslot, 64), 64, 0, st>>>(a);
  lvo_grid_build(st, a.grid, launches);
  k_depth_assoc<<<max(1, min(lvo_div_up((long long)a.kp_total, 8), 1184)), 256, 0, st>>>(a);
  if (launches) *launches += 4;
}
