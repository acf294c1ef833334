// lvo_mapping.cuh — lvo_scan_to_map: the body of process(), reference src/laserMapping.cpp:307-848.
//
// Map layout in HBM: per lane and per type (corner / surf) ONE array of float4 sorted by the reference's cube array
// index i + 21 j + 441 k (:522) plus a 4852-entry exclusive offset table; two generations (ping-pong) so that the
// per-frame rebuild is a pure gather.  The pointer rotations of :323-507 never move data: a shift only changes
// laserCloudCen* and a pending offset that the rebuild applies (cubes that leave the 21x21x11 window are dropped,
// which is what `->clear()` on the recycled cube does).
//
//   k_map_begin        transformAssociateToMap :142-146, centre cube + shift loops :312-507, valid list :512-529
//   k_map_gather       concatenation of the 75 valid cubes in i,j,k loop order :531-537 (defines the kNN point ids)
//   stack downsample   lvo_voxel_run over 2 segments per lane (corner lineRes / surf planeRes) :542-550
//   lvo_grid_build     replaces the two kd-tree builds :558-559
//   k_map_knn          per outer iteration (:562): pointAssociateToMap :154-163, 5-NN + d5^2 < 1 gate :582-584 /
//                      :648-652, one thread per query on the uniform grid
//   k_map_fit          line fit by 3x3 symmetric eigen-solve :586-621, plane fit by 5x3 least squares :650-686,
//                      factor records for LidarEdgeFactor / LidarPlaneNormFactor
//   k_lm_solve         ceres::Solve :712-720
//   k_map_finish       transformUpdate :148-152
//   refilter           insert the transformed stack points into their cubes :737-783 and VoxelGrid every valid cube
//                      :788-801: one lvo_voxel_run over 77 segments per lane and type (none for a lane with a fixed map)
//   k_rebuild_*        new cube offset table + gather into the other map generation
//   k_register         registered full-resolution cloud :838-842
#pragma once
#include "lvo_internal.h"
#include "lvo_knn.cuh"
#include "lvo_solver.cuh"
#include "lvo_voxel.cuh"

#define LVO_SEG_NONVALID 75
#define LVO_SEG_TRASH 76
#define LVO_MSEGS 77

struct MapArgs {
  LaneState* ls;
  int lanes, outer, from_odo;
  const int* lane_flags;             // [lanes] LVO_LANE_* of the step: a lane without LVO_LANE_MAPS keeps its map, poses and counters;
                                     // one with LVO_LANE_MAP_FIXED maps but skips the insertion + re-filter
  const LaneConfig* lcfg;            // [lanes] leaf[0], leaf[1]: each lane's lineRes, planeRes as float (setLeafSize takes floats)
  // inputs: corner_last / surf_last / full-res of this frame
  const float4* in_pts[2]; int in_cap[2];   // less_sharp [cap_lsharp], less_flat [P]; counts n_less_sharp / n_less_flat
  const float4* full; int P;
  // map generations
  float4* map_pts[2][2];             // [gen][type] -> [lanes][map_cap[type]]
  unsigned* cube_start[2][2];        // [gen][type] -> [lanes][LVO_NCUBES + 1]
  int map_cap[2];
  int gen;                           // generation holding the current map
  float4* from_map[2];               // [type] -> [lanes][map_cap[type]]
  float4* stack[2];                  // [type] -> [lanes][in_cap[type]]
  GridSet grid;                      // problems 2*lane+type over from_map
  VoxelEngine vx;
  unsigned* item_off;                // [2*lanes + 1] offsets of each (lane,type) block inside the engine input
  LvoFactor* factors; int factor_cap;
  unsigned* app_cnt;                 // [2*lanes][LVO_NCUBES] appended (non-valid cube) counts
  unsigned* app_first;               // [2*lanes][LVO_NCUBES] first engine output position of those
  unsigned* new_cnt;                 // [2*lanes][LVO_NCUBES + 1]
  // probes
  int* knn_ind[2];                   // [type] -> [lanes][slots][in_cap[type]][5]
  int* fac_valid[2];                 // [type] -> [lanes][slots][in_cap[type]]
  int slots;                         // outer-iteration slots kept (LVO_MAX_OUTER with lvo_config::debug_probes, else 2)
  // LVO_OPT_KNN_REUSE: certified reuse of a query's neighbour set across the outer iterations of a frame (k_map_knn_reuse)
  int knn_reuse;
  float4* knn_ref[2];                // [type] -> [lanes][in_cap[type]] query position of the last full search (x, y, z) and its guard radius (w)
  int* knn_sel[2];                   // [type] -> [lanes][in_cap[type]][5] the up-to-5 nearest points of the last search, ranked at the latest pose (INT_MAX = none)
  int* knn_flag[2];                  // [type] -> [lanes][in_cap[type]] LVO_KF_* bits
  int* fit_list;                     // [lanes][in_cap[0] + in_cap[1]] factor slots whose row changed in this outer iteration (k_map_fit_reuse refits them)
  int* fit_cnt;                      // [lanes][LVO_MAX_OUTER] their number per outer iteration (zeroed by k_map_begin)
  float4* registered;                // [lanes][P] or null
  LvoUncRaw* unc;                    // [lanes][2] pose-uncertainty records (lvo_solver.cuh); k_map_begin clears `solved` of stage 1
};

__device__ __forceinline__ int cube_index(int i, int j, int k) { return i + LVO_CUBE_W * j + LVO_CUBE_W * LVO_CUBE_H * k; }

__global__ void k_map_begin(MapArgs a) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= a.lanes) return;
  LaneState& s = a.ls[lane];
  // a lane that does not map in this step (idle, or off its skip_frame phase): k-NN, fit and solve return for it by its lane flags, the
  // gather / stack / refilter / finish / register kernels see no items, and the rebuild carries its map into the other generation
  // unchanged.  Nothing of its state is written, so that its snapshot does not depend on what the other lanes of the context do.
  if (!lane_maps(a.lane_flags, lane)) return;
  a.unc[2 * lane + 1].solved = 0;   // set again by k_lm_solve unless the map is too small
  if (a.from_odo) { for (int k = 0; k < 4; ++k) s.q_wodom[k] = s.q_w[k]; for (int k = 0; k < 3; ++k) s.t_wodom[k] = s.t_w[k]; }
  // transformAssociateToMap
  quat_mul(s.q_wmap_wodom, s.q_wodom, s.map_x);
  const d3 r = quat_rotate(s.q_wmap_wodom, d3{s.t_wodom[0], s.t_wodom[1], s.t_wodom[2]});
  s.map_x[4] = r.x + s.t_wmap_wodom[0]; s.map_x[5] = r.y + s.t_wmap_wodom[1]; s.map_x[6] = r.z + s.t_wmap_wodom[2];
  const int dims[3] = {LVO_CUBE_W, LVO_CUBE_H, LVO_CUBE_D};
  for (int c = 0; c < 3; ++c) {
    int center = cube_coord(s.map_x[4 + c], s.cen[c]);  // :312-321
    int sh = 0;
    while (center < 3) { center++; sh++; }                 // :323-352 etc: contents move to higher indices
    while (center >= dims[c] - 3) { center--; sh--; }      // :354-383 etc
    s.center[c] = center; s.cen[c] += sh; s.shift[c] = sh;
  }
  int nv = 0;
  for (int i = s.center[0] - 2; i <= s.center[0] + 2; i++)
    for (int j = s.center[1] - 2; j <= s.center[1] + 2; j++)
      for (int k = s.center[2] - 1; k <= s.center[2] + 1; k++)
        if (i >= 0 && i < LVO_CUBE_W && j >= 0 && j < LVO_CUBE_H && k >= 0 && k < LVO_CUBE_D) s.valid_cube[nv++] = cube_index(i, j, k);
  s.n_valid = nv;
  // sizes of the valid cubes in the stored (pre-shift) indexing
  for (int t = 0; t < 2; ++t) {
    const unsigned* cs = a.cube_start[a.gen][t] + (size_t)lane * (LVO_NCUBES + 1);
    int acc = 0;
    for (int v = 0; v < nv; ++v) {
      const int c = s.valid_cube[v];
      const int i = c % LVO_CUBE_W - s.shift[0], j = (c / LVO_CUBE_W) % LVO_CUBE_H - s.shift[1], k = c / (LVO_CUBE_W * LVO_CUBE_H) - s.shift[2];
      int cnt = 0;
      if (i >= 0 && i < LVO_CUBE_W && j >= 0 && j < LVO_CUBE_H && k >= 0 && k < LVO_CUBE_D) { const int oc = cube_index(i, j, k); cnt = (int)(cs[oc + 1] - cs[oc]); }
      s.from_off[t][v] = acc;
      acc += cnt;
    }
    for (int v = nv; v <= LVO_MAX_VALID; ++v) s.from_off[t][v] = acc;
  }
  s.stats.map_corner_from_map = s.from_off[0][LVO_MAX_VALID];
  s.stats.map_surf_from_map = s.from_off[1][LVO_MAX_VALID];
  s.map_too_small = !(s.from_off[0][LVO_MAX_VALID] > 10 && s.from_off[1][LVO_MAX_VALID] > 50);  // :554
  s.map_status = s.map_too_small ? LVO_W_MAP_TOO_SMALL : LVO_OK;
  s.map_done = 0; s.stats.map_outer_executed = 0;
  for (int o = 0; o < LVO_MAX_OUTER; ++o) { s.stats.map_corner_corr[o] = 0; s.stats.map_surf_corr[o] = 0; s.stats.map_lm_iters[o] = 0; s.stats.map_final_cost[o] = 0; s.stats.map_knn_full[o] = 0; if (a.fit_cnt) a.fit_cnt[lane * LVO_MAX_OUTER + o] = 0; }
  for (int c = 0; c < 3; ++c) { s.stats.center_cube[c] = s.center[c]; s.stats.cen[c] = s.cen[c]; }
}

// grid (LVO_MAX_VALID, 2 * lanes): copy one valid cube into FromMap
__global__ void k_map_gather(MapArgs a) {
  const int v = blockIdx.x, lt = blockIdx.y, lane = lt >> 1, t = lt & 1;
  const LaneState& s = a.ls[lane];
  const bool maps = lane_maps(a.lane_flags, lane);
  if (v >= s.n_valid || !maps) return;
  const int c = s.valid_cube[v];
  const int i = c % LVO_CUBE_W - s.shift[0], j = (c / LVO_CUBE_W) % LVO_CUBE_H - s.shift[1], k = c / (LVO_CUBE_W * LVO_CUBE_H) - s.shift[2];
  if (!(i >= 0 && i < LVO_CUBE_W && j >= 0 && j < LVO_CUBE_H && k >= 0 && k < LVO_CUBE_D)) return;
  const int oc = cube_index(i, j, k);
  const unsigned* cs = a.cube_start[a.gen][t] + (size_t)lane * (LVO_NCUBES + 1);
  const unsigned b = cs[oc], e = cs[oc + 1];
  const float4* src = a.map_pts[a.gen][t] + (size_t)lane * a.map_cap[t];
  float4* dst = a.from_map[t] + (size_t)lane * a.map_cap[t] + s.from_off[t][v];
  for (unsigned x = b + threadIdx.x; x < e; x += blockDim.x) dst[x - b] = src[x];
}

// ---- stack downsample (engine run A) -------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_stack_offsets(MapArgs a) {
  __shared__ unsigned sm[33];
  const int L2 = 2 * a.lanes;
  unsigned acc = 0;
  for (int base = 0; base < L2; base += blockDim.x) {
    const int lt = base + threadIdx.x;
    unsigned v = 0;
    if (lt < L2) {
      const LaneState& s = a.ls[lt >> 1];
      if (lane_maps(a.lane_flags, lt >> 1)) v = (unsigned)((lt & 1) ? s.n_less_flat : s.n_less_sharp);
      a.vx.seg_leaf[lt] = a.lcfg[lt >> 1].leaf[lt & 1];
    }
    unsigned tot;
    const unsigned ex = block_excl_scan(v, sm, &tot);
    if (lt < L2) a.item_off[lt] = acc + ex;
    acc += tot;
  }
  if (threadIdx.x == 0) { a.item_off[L2] = acc; *a.vx.d_n = (int)acc; *a.vx.d_nsegs = L2; }
}
__global__ void k_stack_gather(MapArgs a) {
  const int lt = blockIdx.y, lane = lt >> 1, t = lt & 1;
  const LaneState& s = a.ls[lane];
  const int n = t ? s.n_less_flat : s.n_less_sharp;
  if (!lane_maps(a.lane_flags, lane)) return;
  const float4* src = a.in_pts[t] + (size_t)lane * a.in_cap[t];
  const unsigned off = a.item_off[lt];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    a.vx.in_pts[off + i] = src[i];
    a.vx.in_seg[off + i] = lt;
    a.vx.in_aux[off + i] = 0;
  }
}
__global__ void k_stack_scatter(MapArgs a) {
  const int lt = blockIdx.y, lane = lt >> 1, t = lt & 1;
  LaneState& s = a.ls[lane];
  const unsigned b = a.vx.seg_out_start[lt], n = a.vx.seg_out_cnt[lt];
  if (!lane_maps(a.lane_flags, lane)) return;   // keeps n_stack and the stack (parity probes) of the lane's last mapping step
  float4* dst = a.stack[t] + (size_t)lane * a.in_cap[t];
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = a.vx.out_pts[b + i];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    s.n_stack[t] = (int)n;
    if (t == 0) s.stats.map_corner_stack = (int)n; else s.stats.map_surf_stack = (int)n;
  }
}

// ---- association + fit ------------------------------------------------------------------------------------------------
// Line fit (:586-621) / plane fit (:650-686) of ONE query from its 5 neighbours; executed by one thread.
__device__ __forceinline__ void fit_factor(int t, const float4 ori, const float4* __restrict__ M, const int* id, LvoFactor& fac) {
  float4 nb[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) nb[j] = M[id[j]];
  if (t == 0) {
    d3 center{0, 0, 0};
#pragma unroll
    for (int j = 0; j < 5; ++j) { center.x = center.x + (double)nb[j].x; center.y = center.y + (double)nb[j].y; center.z = center.z + (double)nb[j].z; }
    center.x = center.x / 5.0; center.y = center.y / 5.0; center.z = center.z / 5.0;
    double cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const double z[3] = {(double)nb[j].x - center.x, (double)nb[j].y - center.y, (double)nb[j].z - center.z};
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) cov[r * 3 + c] = cov[r * 3 + c] + z[r] * z[c];
    }
    double w[3], V[9];
    sym_eigen_dev<3>(cov, w, V);
    if (w[2] > 3 * w[1]) {  // :611
      const double ux = V[0 * 3 + 2], uy = V[1 * 3 + 2], uz = V[2 * 3 + 2];
      fac.type = 0; fac.d = 1.0;
      fac.c[0] = ori.x; fac.c[1] = ori.y; fac.c[2] = ori.z;
      fac.a[0] = 0.1 * ux + center.x; fac.a[1] = 0.1 * uy + center.y; fac.a[2] = 0.1 * uz + center.z;
      const double lb[3] = {-0.1 * ux + center.x, -0.1 * uy + center.y, -0.1 * uz + center.z};   // point_b :606-608
      lvo_edge_direction(fac.a, lb, fac.b);
    }
  } else {
    double A[15], b[5] = {-1, -1, -1, -1, -1}, n[3];
#pragma unroll
    for (int j = 0; j < 5; ++j) { A[j * 3 + 0] = nb[j].x; A[j * 3 + 1] = nb[j].y; A[j * 3 + 2] = nb[j].z; }
    // a rank-deficient 5x3 (Eigen's colPivHouseholderQr would still return a finite vector) gives no usable normal: no factor
    if (!lsq_qr_5x3(A, b, n)) return;
    const double nn = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    if (!(nn > 0.0) || !isfinite(nn)) return;
    const double negOA = 1 / nn;
    n[0] /= nn; n[1] /= nn; n[2] /= nn;
    bool planeValid = true;
#pragma unroll
    for (int j = 0; j < 5; ++j)
      if (!(fabs(n[0] * nb[j].x + n[1] * nb[j].y + n[2] * nb[j].z + negOA) <= 0.2)) { planeValid = false; }  // :672-678 (a NaN never passes)
    if (planeValid) {
      fac.type = 2;
      fac.c[0] = ori.x; fac.c[1] = ori.y; fac.c[2] = ori.z;
      fac.a[0] = n[0]; fac.a[1] = n[1]; fac.a[2] = n[2];
      fac.b[0] = fac.b[1] = fac.b[2] = 0;
      fac.d = negOA;
    }
  }
}

// 5-NN of every stack point (one thread per query): pointAssociateToMap :154-163, nearestKSearch + gate :582-584 / :648-652.
// Writes the index sets (all -1 when d5^2 >= 1.0).  This is the graded kNN kernel (SURVEY §8d).
__global__ void __launch_bounds__(128) k_map_knn(MapArgs a) {
  const int lane = blockIdx.y;
  const LaneState& s = a.ls[lane];
  if (!lane_maps(a.lane_flags, lane) || s.map_too_small || s.map_done) return;   // :554 / fixed point reached (LVO_OPT_FIXPOINT_SKIP)
  const int n0 = s.n_stack[0], ntot = n0 + s.n_stack[1];
  const GridView g0 = grid_view(a.grid, 2 * lane), g1 = grid_view(a.grid, 2 * lane + 1);
  for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < ntot; f += gridDim.x * blockDim.x) {
    const int t = f >= n0 ? 1 : 0;
    const int i = t ? f - n0 : f;
    const float4 ori = a.stack[t][(size_t)lane * a.in_cap[t] + i];
    const float4 sel = transform_point(s.map_x, s.map_x + 4, ori);
    TopK<5> tk;
    const bool ok = thread_knn<5>(t ? g1 : g0, sel.x, sel.y, sel.z, 1.0f, tk);
    int* ki = a.knn_ind[t] + (((size_t)lane * a.slots + a.outer % a.slots) * a.in_cap[t] + i) * 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) ki[k] = ok ? tk.id[k] : -1;
  }
}
// ---- certified reuse of the neighbour sets across outer iterations (LVO_OPT_KNN_REUSE) -----------------------------------------
// The ten outer iterations of a frame (:562) search the SAME map with a pose that moves less and less, so almost every query keeps
// its five neighbours from one iteration to the next.  A full search at position q_ref leaves, besides the set S of the (up to)
// five nearest points, a GUARD radius: a lower bound on the distance from q_ref to every map point outside S — the smaller of
// the sixth-best candidate distance and the distance from q_ref to the boundary of the 3 x 3 x 3 cell block that was scanned.
// At a later position q_new (moved by delta = |q_new - q_ref|) every point outside S is at least guard - delta away, so
//   (a) |S| = 5 and the largest new distance inside S is below guard - delta: S is exactly the 5-NN set at q_new, and ranking its
//       members by the reference's (distance, index) key with distances computed by the same float expression gives the very row a
//       full search returns (no outside point can even tie);
//   (b) guard - delta > 1: every point outside S fails the d5^2 < 1.0 gate (:584 / :652), so the row is S (if |S| = 5 and its
//       fifth distance passes the gate) or "no correspondence", again exactly what a full search returns;
//   otherwise the query is searched in full again.  All comparisons carry margins (1e-4 relative + 1e-5 m) that dwarf float rounding
//   (~1e-7 relative), and they only decide WHETHER the shortcut is taken, never a result.  A query whose row did not change keeps its
//   factor record (the fit depends only on the query point and on the ordered neighbour points), so k_map_fit_reuse skips it.
#define LVO_KNN_PRUNE_SQ 1.21f   // full searches rank candidates inside 1.1 m only: the gate is 1 m, the rest only feeds the guard radius
#define LVO_KF_ROW 1       // the row of the latest iteration is valid (5 neighbours inside the gate)
#define LVO_KF_FACTOR 2    // the factor record of the latest fit is valid (type >= 0)
#define LVO_KF_CHANGED 4   // the row changed in this iteration: k_map_fit_reuse must refit

// guard radius of a full search at (qx, qy, qz): min(sixth-best distance, distance to the boundary of the scanned 3 x 3 x 3 block),
// shrunk by the safety margin.  The block reaches one whole cell beyond the query's own cell on every side.
__device__ __forceinline__ float knn_guard(const GridView& g, float qx, float qy, float qz, const TopK<6>& tk) {
  const float fx = floorf(qx * g.inv_cell), fy = floorf(qy * g.inv_cell), fz = floorf(qz * g.inv_cell_z);
  if (!(g.dim[0] > 0 && fabsf(fx) < 8.0e6f && fabsf(fy) < 8.0e6f && fabsf(fz) < 8.0e6f)) return 0.f;   // cell coordinates exact in float (and not clamped by cell_coord)
  const float cz_size = 1.0f / g.inv_cell_z;
  const float lx = qx - fx * g.cell, ly = qy - fy * g.cell, lz = qz - fz * cz_size;   // offsets inside the cell, in [0, cell]
  const float bx = fminf(lx, g.cell - lx) + g.cell, by = fminf(ly, g.cell - ly) + g.cell, bz = fminf(lz, cz_size - lz) + cz_size;
  float gd = fminf(fminf(bx, by), bz);
  // candidates are only ranked inside LVO_KNN_PRUNE_SQ (TopK::init(bound)): an empty sixth slot means "nothing else inside that radius"
  gd = fminf(gd, sqrtf(tk.d[5]));
  return fmaxf(gd * 0.9999f - 1e-5f, 0.f);
}

// Full search of one query by ONE thread (the form of thread_knn, six best): used in outer iteration 0, where every query of the lane is
// searched and the thread-per-query form keeps the most searches in flight (measured: 135 us against 220 us for the tile form at 128 lanes).
__device__ __forceinline__ void thread_knn6_block(const GridView& g, float qx, float qy, float qz, TopK<6>& tk) {
  tk.init(LVO_KNN_PRUNE_SQ);
  if (g.dim[0] <= 0) return;
  const int cx = cell_coord(qx, g.inv_cell) - g.org[0], cy = cell_coord(qy, g.inv_cell) - g.org[1], cz = cell_coord(qz, g.inv_cell_z) - g.org[2];
  unsigned rb[9], re[9];
  const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dim[0] - 1);
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int z = cz + k / 3 - 1, y = cy + k % 3 - 1;
    rb[k] = re[k] = 0;
    if (z >= 0 && z < g.dim[2] && y >= 0 && y < g.dim[1] && x0 <= x1) {
      const int rowbase = (z * g.dim[1] + y) * g.dim[0];
      rb[k] = __ldg(g.cell_start + rowbase + x0); re[k] = __ldg(g.cell_start + rowbase + x1 + 1);
    }
  }
#pragma unroll 1
  for (int k = 0; k < 9; ++k) {
    unsigned t = rb[k];
    const unsigned e = re[k];
    for (; t + 4 <= e; t += 4) {
      const float4 p0 = __ldg(g.pts + t), p1 = __ldg(g.pts + t + 1), p2 = __ldg(g.pts + t + 2), p3 = __ldg(g.pts + t + 3);
      tk.insert(sqdist3(p0, qx, qy, qz), __float_as_int(p0.w));
      tk.insert(sqdist3(p1, qx, qy, qz), __float_as_int(p1.w));
      tk.insert(sqdist3(p2, qx, qy, qz), __float_as_int(p2.w));
      tk.insert(sqdist3(p3, qx, qy, qz), __float_as_int(p3.w));
    }
    if (t < e) {
      const float4 p0 = __ldg(g.pts + t);
      const float4 p1 = t + 1 < e ? __ldg(g.pts + t + 1) : p0;
      const float4 p2 = t + 2 < e ? __ldg(g.pts + t + 2) : p0;
      tk.insert(sqdist3(p0, qx, qy, qz), __float_as_int(p0.w));
      if (t + 1 < e) tk.insert(sqdist3(p1, qx, qy, qz), __float_as_int(p1.w));
      if (t + 2 < e) tk.insert(sqdist3(p2, qx, qy, qz), __float_as_int(p2.w));
    }
  }
}

// (distance, index)-ranked merge of the per-lane lists of a TW-lane tile; afterwards every lane of the tile holds the tile-wide best K
template <int K, int TW>
__device__ __forceinline__ void tile_merge(TopK<K>& tk) {
  float rd[K]; int ri[K];
  int ptr = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float cd = FLT_MAX; int ci = INT_MAX;
#pragma unroll
    for (int j = 0; j < K; ++j) if (j == ptr) { cd = tk.d[j]; ci = tk.id[j]; }
    float bd = cd; int bi = ci;
#pragma unroll
    for (int o = TW / 2; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, bd, o, TW);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o, TW);
      if (TopK<K>::less(od, oi, bd, bi)) { bd = od; bi = oi; }
    }
    rd[k] = bd; ri[k] = bi;
    if (bi == ci && bd == cd && ci != INT_MAX) ptr++;  // ids are unique, so exactly one lane advances
  }
#pragma unroll
  for (int k = 0; k < K; ++k) { tk.d[k] = rd[k]; tk.id[k] = ri[k]; }
}

// Full search of one query by an 8-lane tile (four queries per warp; every call is made by all 32 lanes): the 9 rows of the
// 3 x 3 x 3 cell block around the query (cell >= 1 m covers the 1 m gate), lanes strided over the concatenated candidate ranges
// (two loads in flight per lane), six best candidates by (distance, index), and the guard radius of the certificate above.
// One thread walking the block on its own has a dependent chain of ~8-30 load round trips (corner queries see 50-170 candidates)
// and a warp waits for its slowest lane (ncu: 10 of 32 threads active); the tile shares a query's candidates between 8 lanes.
__device__ __forceinline__ void tile8_knn6_block(const GridView& g, bool active, float qx, float qy, float qz, TopK<6>& tk, float& guard) {
  const int tl = (int)tile_lane<8>();
  tk.init(LVO_KNN_PRUNE_SQ);
  guard = 0.f;
  const int cx = cell_coord(qx, g.inv_cell) - g.org[0], cy = cell_coord(qy, g.inv_cell) - g.org[1], cz = cell_coord(qz, g.inv_cell_z) - g.org[2];
  auto consider = [&](float4 p, int) { tk.insert(sqdist3(p, qx, qy, qz), __float_as_int(p.w)); };
#pragma unroll 1
  for (int base = 0; base < 9; base += 8) {   // rows 0..7, then row 8
    const int row = base + tl;
    unsigned b = 0, e = 0;
    if (active && g.dim[0] > 0 && row < 9) row_bounds(g, cz + row / 3 - 1, cy + row % 3 - 1, cx - 1, cx + 1, b, e);
    tile_scan_ranges<8, 8>(g.pts, b, e, consider);
  }
  tile_merge<6, 8>(tk);
  guard = knn_guard(g, qx, qy, qz, tk);
}

__global__ void __launch_bounds__(128) k_map_knn_reuse(MapArgs a) {
  __shared__ float4 s_sel[128];
  __shared__ int s_list[128], s_fit[128];
  __shared__ int s_n, s_nfit, s_off;
  const int lane = blockIdx.y;
  const LaneState& s = a.ls[lane];
  if (!lane_maps(a.lane_flags, lane) || s.map_too_small || s.map_done) return;   // :554 / fixed point reached (LVO_OPT_FIXPOINT_SKIP)
  const int n0 = s.n_stack[0], ntot = n0 + s.n_stack[1];
  int nc = 0, nsf = 0;   // factors kept from the previous iteration (unchanged rows)
  __shared__ GridView gv[2];   // shared, not registers: the certificate phase wants occupancy
  if (threadIdx.x < 2) gv[threadIdx.x] = grid_view(a.grid, 2 * lane + threadIdx.x);
  const float4* M0 = a.from_map[0] + (size_t)lane * a.map_cap[0];
  const float4* M1 = a.from_map[1] + (size_t)lane * a.map_cap[1];
  const int slot = a.outer % a.slots;
  for (int base = blockIdx.x * blockDim.x; base < ntot; base += gridDim.x * blockDim.x) {
    if (threadIdx.x == 0) { s_n = 0; s_nfit = 0; }
    __syncthreads();
    // ---- phase A, one thread per query: the query in the map frame; from the second outer iteration on, the certificate
    const int f = base + threadIdx.x;
    bool need_full = false, refit = false;
    if (f < ntot) {
      need_full = true;
      const int t = f >= n0 ? 1 : 0;
      const int i = t ? f - n0 : f;
      const size_t qi = (size_t)lane * a.in_cap[t] + i;
      const float4 ori = a.stack[t][qi];
      const float4 sel = transform_point(s.map_x, s.map_x + 4, ori);   // pointAssociateToMap :154-163
      s_sel[threadIdx.x] = sel;
      if (a.outer > 0) {
        const float4 ref = a.knn_ref[t][qi];
        const int flag = a.knn_flag[t][qi];
        int id[5], old[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) old[k] = id[k] = a.knn_sel[t][qi * 5 + k];
        const float4* M = t ? M1 : M0;
        float d[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) d[k] = id[k] != INT_MAX ? sqdist3(M[id[k]], sel.x, sel.y, sel.z) : FLT_MAX;
        // rank by (distance, index): insertion sort of five (INT_MAX entries carry FLT_MAX and stay last)
#pragma unroll
        for (int k = 1; k < 5; ++k)
#pragma unroll
          for (int j = k; j > 0; --j)
            if (TopK<5>::less(d[j], id[j], d[j - 1], id[j - 1])) {
              const float td = d[j]; d[j] = d[j - 1]; d[j - 1] = td;
              const int ti = id[j]; id[j] = id[j - 1]; id[j - 1] = ti;
            }
        const float dx = sel.x - ref.x, dy = sel.y - ref.y, dz = sel.z - ref.z;
        const float delta = sqrtf(dx * dx + dy * dy + dz * dz) * 1.0001f + 1e-5f;
        const float B = ref.w - delta;           // every point outside the set is farther than this from the new position
        const bool full_set = id[4] != INT_MAX;
        bool decided = false, row_ok = false;
        if (full_set && sqrtf(d[4]) * 1.0001f + 1e-5f < B) { decided = true; row_ok = (double)d[4] < 1.0; }
        else if (B > 1.0002f) { decided = true; row_ok = full_set && (double)d[4] < 1.0; }
        if (decided) {
          need_full = false;
          bool reordered = false;
#pragma unroll
          for (int k = 0; k < 5; ++k) if (old[k] != id[k]) { reordered = true; a.knn_sel[t][qi * 5 + k] = id[k]; }
          if (a.slots > 2) {   // per-iteration probe rows (lvo_config::debug_probes); the path itself reads knn_sel / knn_flag
            int* ki = a.knn_ind[t] + (((size_t)lane * a.slots + slot) * a.in_cap[t] + i) * 5;
#pragma unroll
            for (int k = 0; k < 5; ++k) ki[k] = row_ok ? id[k] : -1;
          }
          const bool changed = row_ok != ((flag & LVO_KF_ROW) != 0) || (row_ok && reordered);
          a.knn_flag[t][qi] = (flag & LVO_KF_FACTOR) | (row_ok ? LVO_KF_ROW : 0) | (changed ? LVO_KF_CHANGED : 0);
          refit = changed;
          if (!changed) {   // the factor record of the previous iteration stands
            const int v = (flag & LVO_KF_FACTOR) ? 1 : 0;
            if (a.slots > 2) a.fac_valid[t][((size_t)lane * a.slots + slot) * a.in_cap[t] + i] = v;   // probe (lvo_config::debug_probes)
            if (v) { if (t == 0) nc++; else nsf++; }
          }
        }
      }
    }
    // ---- the queries that need a full search, compacted so that the 8-lane tiles below are all busy
    {
      const unsigned m = __ballot_sync(0xffffffffu, need_full);
      int off = 0;
      if ((threadIdx.x & 31) == 0 && m) off = atomicAdd(&s_n, __popc(m));
      off = __shfl_sync(0xffffffffu, off, 0);
      if (need_full) s_list[off + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = (int)threadIdx.x;
      const unsigned m2 = __ballot_sync(0xffffffffu, refit);
      int off2 = 0;
      if ((threadIdx.x & 31) == 0 && m2) off2 = atomicAdd(&s_nfit, __popc(m2));
      off2 = __shfl_sync(0xffffffffu, off2, 0);
      if (refit) s_fit[off2 + __popc(m2 & ((1u << (threadIdx.x & 31)) - 1u))] = (int)threadIdx.x;
    }
    __syncthreads();
    const int nfull = s_n;
    // the factor slots k_map_fit_reuse has to refit: the rows that changed under the certificate and every query searched in full
    // (iteration 0 refits everything and needs no list)
    const int nfit = s_nfit + nfull;
    if (a.outer > 0 && nfit > 0) {
      if (threadIdx.x == 0) s_off = atomicAdd(&a.fit_cnt[lane * LVO_MAX_OUTER + a.outer], nfit);
      __syncthreads();
      int* fl = a.fit_list + (size_t)lane * (a.in_cap[0] + a.in_cap[1]) + s_off;
      if ((int)threadIdx.x < nfit) fl[threadIdx.x] = base + ((int)threadIdx.x < s_nfit ? s_fit[threadIdx.x] : s_list[threadIdx.x - s_nfit]);
    }
    if (threadIdx.x == 0 && nfull) atomicAdd(&a.ls[lane].stats.map_knn_full[a.outer], nfull);
    // ---- phase B.  Outer iteration 0: every query is searched, one thread each.
    if (a.outer == 0) {
      if (f < ntot) {
        const int t = f >= n0 ? 1 : 0;
        const int i = t ? f - n0 : f;
        const size_t qi = (size_t)lane * a.in_cap[t] + i;
        const float4 sel = s_sel[threadIdx.x];
        TopK<6> tk;
        thread_knn6_block(gv[t], sel.x, sel.y, sel.z, tk);
        const float guard = knn_guard(gv[t], sel.x, sel.y, sel.z, tk);
        const bool row_ok = tk.id[4] != INT_MAX && (double)tk.d[4] < 1.0;
#pragma unroll
        for (int k = 0; k < 5; ++k) a.knn_sel[t][qi * 5 + k] = tk.id[k];
        if (a.slots > 2) {
          int* ki = a.knn_ind[t] + (((size_t)lane * a.slots + slot) * a.in_cap[t] + i) * 5;
#pragma unroll
          for (int k = 0; k < 5; ++k) ki[k] = row_ok ? tk.id[k] : -1;
        }
        a.knn_ref[t][qi] = make_float4(sel.x, sel.y, sel.z, guard);
        a.knn_flag[t][qi] = (row_ok ? LVO_KF_ROW : 0) | LVO_KF_CHANGED;
      }
      __syncthreads();
      continue;
    }
    // Later iterations: the few queries without a certificate, 16 tiles of 8 lanes per block; a warp's four tiles take entries
    // 4 w .. 4 w + 3 of every group of 16
    const int w = threadIdx.x >> 5, tile = (threadIdx.x & 31) >> 3;
    for (int e0 = 4 * w; e0 < nfull; e0 += 16) {   // uniform per warp
      const int e = e0 + tile;
      const bool active = e < nfull;
      const int src = active ? s_list[e] : 0;
      const int f2 = base + src;
      const int t = (active && f2 >= n0) ? 1 : 0;
      const float4 sel = s_sel[src];
      TopK<6> tk;
      float guard;
      // both types in one warp: the grid is selected per tile (all members are per-tile values)
      tile8_knn6_block(gv[t], active, sel.x, sel.y, sel.z, tk, guard);
      if (active && tile_lane<8>() == 0) {
        const int i = t ? f2 - n0 : f2;
        const size_t qi = (size_t)lane * a.in_cap[t] + i;
        const bool row_ok = tk.id[4] != INT_MAX && (double)tk.d[4] < 1.0;
#pragma unroll
        for (int k = 0; k < 5; ++k) a.knn_sel[t][qi * 5 + k] = tk.id[k];
        if (a.slots > 2) {
          int* ki = a.knn_ind[t] + (((size_t)lane * a.slots + slot) * a.in_cap[t] + i) * 5;
#pragma unroll
          for (int k = 0; k < 5; ++k) ki[k] = row_ok ? tk.id[k] : -1;
        }
        a.knn_ref[t][qi] = make_float4(sel.x, sel.y, sel.z, guard);
        // a full search always asks for a refit (it is the rare path after the first iteration)
        const int oldf = a.knn_flag[t][qi];
        a.knn_flag[t][qi] = (oldf & LVO_KF_FACTOR) | (row_ok ? LVO_KF_ROW : 0) | LVO_KF_CHANGED;
      }
    }
    __syncthreads();
  }
  nc = __reduce_add_sync(0xffffffffu, nc);
  nsf = __reduce_add_sync(0xffffffffu, nsf);
  if ((threadIdx.x & 31) == 0) {
    if (nc) atomicAdd(&a.ls[lane].stats.map_corner_corr[a.outer], nc);
    if (nsf) atomicAdd(&a.ls[lane].stats.map_surf_corr[a.outer], nsf);
  }
}

// fits for the rows that changed (the list k_map_knn_reuse wrote; iteration 0: every query); the others keep their factor record
__global__ void __launch_bounds__(128) k_map_fit_reuse(MapArgs a) {
  const int lane = blockIdx.y;
  LaneState& s = a.ls[lane];
  if (!lane_maps(a.lane_flags, lane) || s.map_too_small || s.map_done) return;
  const int n0 = s.n_stack[0], ntot = n0 + s.n_stack[1];
  const int n = a.outer > 0 ? a.fit_cnt[lane * LVO_MAX_OUTER + a.outer] : ntot;
  const int* fl = a.fit_list + (size_t)lane * (a.in_cap[0] + a.in_cap[1]);
  const float4* M0 = a.from_map[0] + (size_t)lane * a.map_cap[0];
  const float4* M1 = a.from_map[1] + (size_t)lane * a.map_cap[1];
  const int slot = a.outer % a.slots;
  int nc = 0, nsf = 0;
  for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const int e = base + threadIdx.x;
    if (e < n) {
      const int f2 = a.outer > 0 ? fl[e] : e;
      const int t = f2 >= n0 ? 1 : 0;
      const int i = t ? f2 - n0 : f2;
      const size_t qi = (size_t)lane * a.in_cap[t] + i;
      const int flag = a.knn_flag[t][qi];
      LvoFactor fac;
      fac.type = -1; fac.pad = 0; fac.d = 0;
      if (flag & LVO_KF_ROW) {
        int id[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) id[k] = a.knn_sel[t][qi * 5 + k];
        fit_factor(t, a.stack[t][qi], t ? M1 : M0, id, fac);
      }
      a.factors[(size_t)lane * a.factor_cap + f2] = fac;
      const int v = fac.type >= 0 ? 1 : 0;
      if (a.slots > 2) a.fac_valid[t][((size_t)lane * a.slots + slot) * a.in_cap[t] + i] = v;   // probe
      a.knn_flag[t][qi] = (flag & LVO_KF_ROW) | (v ? LVO_KF_FACTOR : 0);
      if (v) { if (t == 0) nc++; else nsf++; }
    }
  }
  nc = __reduce_add_sync(0xffffffffu, nc);
  nsf = __reduce_add_sync(0xffffffffu, nsf);
  if ((threadIdx.x & 31) == 0) {
    if (nc) atomicAdd(&s.stats.map_corner_corr[a.outer], nc);
    if (nsf) atomicAdd(&s.stats.map_surf_corr[a.outer], nsf);
  }
}

// line / plane fit of every accepted query (one thread per query) -> factor records
__global__ void __launch_bounds__(128) k_map_fit(MapArgs a) {
  const int lane = blockIdx.y;
  LaneState& s = a.ls[lane];
  if (!lane_maps(a.lane_flags, lane) || s.map_too_small || s.map_done) return;   // :554 / fixed point reached (LVO_OPT_FIXPOINT_SKIP)
  const int n0 = s.n_stack[0], ntot = n0 + s.n_stack[1];
  const float4* M0 = a.from_map[0] + (size_t)lane * a.map_cap[0];
  const float4* M1 = a.from_map[1] + (size_t)lane * a.map_cap[1];
  int nc = 0, nsf = 0;
  for (int base = blockIdx.x * blockDim.x; base < ntot; base += gridDim.x * blockDim.x) {
    const int f = base + threadIdx.x;
    if (f < ntot) {
      const int t = f >= n0 ? 1 : 0;
      const int i = t ? f - n0 : f;
      const int* ki = a.knn_ind[t] + (((size_t)lane * a.slots + a.outer % a.slots) * a.in_cap[t] + i) * 5;
      int id[5];
#pragma unroll
      for (int k = 0; k < 5; ++k) id[k] = ki[k];
      LvoFactor fac;
      fac.type = -1; fac.pad = 0; fac.d = 0;
      if (id[0] >= 0) fit_factor(t, a.stack[t][(size_t)lane * a.in_cap[t] + i], t ? M1 : M0, id, fac);
      a.factors[(size_t)lane * a.factor_cap + f] = fac;
      a.fac_valid[t][((size_t)lane * a.slots + a.outer % a.slots) * a.in_cap[t] + i] = fac.type >= 0 ? 1 : 0;
      if (fac.type >= 0) { if (t == 0) nc++; else nsf++; }
    }
  }
  nc = __reduce_add_sync(0xffffffffu, nc);
  nsf = __reduce_add_sync(0xffffffffu, nsf);
  if ((threadIdx.x & 31) == 0) {
    if (nc) atomicAdd(&s.stats.map_corner_corr[a.outer], nc);
    if (nsf) atomicAdd(&s.stats.map_surf_corr[a.outer], nsf);
  }
}

__global__ void k_map_finish(MapArgs a) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= a.lanes || !lane_maps(a.lane_flags, lane)) return;
  LaneState& s = a.ls[lane];
  // transformUpdate :148-152: q_wmap_wodom = q_w_curr * q_wodom_curr.inverse(); t_wmap_wodom = t_w_curr - q_wmap_wodom * t_wodom_curr
  const double* q = s.q_wodom;
  const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const double qi[4] = {-q[0] / n2, -q[1] / n2, -q[2] / n2, q[3] / n2};
  quat_mul(s.map_x, qi, s.q_wmap_wodom);
  const d3 r = quat_rotate(s.q_wmap_wodom, d3{s.t_wodom[0], s.t_wodom[1], s.t_wodom[2]});
  s.t_wmap_wodom[0] = s.map_x[4] - r.x; s.t_wmap_wodom[1] = s.map_x[5] - r.y; s.t_wmap_wodom[2] = s.map_x[6] - r.z;
}

// ---- insertion + per-cube re-filter (engine run B) ------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_refilter_offsets(MapArgs a) {
  __shared__ unsigned sm[33];
  const int L2 = 2 * a.lanes;
  // one (lane, type) row of segments per warp: the lane's leaf for its valid cubes, 0 (pseudo segment) for the rest.  Each lane of the
  // warp loads the leaf of one of the warp's next 32 rows, so that the rows wait for one load, not for one each.
  const int nw = blockDim.x >> 5, ln = threadIdx.x & 31;
  for (int r0 = threadIdx.x >> 5; r0 < L2; r0 += 32 * nw) {
    const int mine = r0 + ln * nw;
    const float my_leaf = mine < L2 ? a.lcfg[mine >> 1].leaf[mine & 1] : 0.f;
    for (int j = 0; j < 32; ++j) {
      const float leaf = __shfl_sync(0xffffffffu, my_leaf, j);
      const int lt = r0 + j * nw;
      if (lt >= L2) break;   // the same for the whole warp
      for (int k = ln; k < LVO_MSEGS; k += 32) a.vx.seg_leaf[lt * LVO_MSEGS + k] = k < LVO_MAX_VALID ? leaf : 0.f;
    }
  }
  unsigned acc = 0;
  for (int base = 0; base < L2; base += blockDim.x) {
    const int lt = base + threadIdx.x;
    unsigned v = 0;
    if (lt < L2 && lane_updates_map(a.lane_flags, lt >> 1)) { const LaneState& s = a.ls[lt >> 1]; v = (unsigned)(s.from_off[lt & 1][LVO_MAX_VALID] + s.n_stack[lt & 1]); }
    unsigned tot;
    const unsigned ex = block_excl_scan(v, sm, &tot);
    if (lt < L2) a.item_off[lt] = acc + ex;
    acc += tot;
  }
  if (threadIdx.x == 0) { a.item_off[L2] = acc; *a.vx.d_n = (int)acc; *a.vx.d_nsegs = L2 * LVO_MSEGS; }
}
__global__ void k_refilter_gather(MapArgs a) {
  const int lt = blockIdx.y, lane = lt >> 1, t = lt & 1;
  const LaneState& s = a.ls[lane];
  const int nfrom = s.from_off[t][LVO_MAX_VALID], nst = s.n_stack[t];
  if (!lane_updates_map(a.lane_flags, lane)) return;
  const unsigned off = a.item_off[lt];
  const float4* FM = a.from_map[t] + (size_t)lane * a.map_cap[t];
  const float4* ST = a.stack[t] + (size_t)lane * a.in_cap[t];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nfrom + nst; i += gridDim.x * blockDim.x) {
    float4 p; int seg; unsigned aux = 0;
    if (i < nfrom) {
      p = FM[i];
      // valid-cube rank by binary search in from_off
      int lo = 0, hi = s.n_valid - 1;
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s.from_off[t][mid] <= i) lo = mid; else hi = mid - 1; }
      seg = lo;
    } else {
      p = transform_point(s.map_x, s.map_x + 4, ST[i - nfrom]);  // :739 / :763 with the final pose
      const int ci = cube_coord((double)p.x, s.cen[0]), cj = cube_coord((double)p.y, s.cen[1]), ck = cube_coord((double)p.z, s.cen[2]);
      if (ci >= 0 && ci < LVO_CUBE_W && cj >= 0 && cj < LVO_CUBE_H && ck >= 0 && ck < LVO_CUBE_D) {
        const int di = ci - (s.center[0] - 2), dj = cj - (s.center[1] - 2), dk = ck - (s.center[2] - 1);
        aux = (unsigned)cube_index(ci, cj, ck);
        if (di >= 0 && di < 5 && dj >= 0 && dj < 5 && dk >= 0 && dk < 3) seg = (di * 5 + dj) * 3 + dk;  // centre is >= 3 cubes from every face: the list is never clipped
        else seg = LVO_SEG_NONVALID;
      } else seg = LVO_SEG_TRASH;
    }
    a.vx.in_pts[off + i] = p;
    a.vx.in_seg[off + i] = lt * LVO_MSEGS + seg;
    a.vx.in_aux[off + i] = aux;
  }
}
__global__ void k_rebuild_reset(MapArgs a) {
  const int n = 2 * a.lanes * LVO_NCUBES;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { a.app_cnt[i] = 0; a.app_first[i] = 0xffffffffu; }
}
// appended points (non-valid cubes): count per cube and first engine-output position
__global__ void k_rebuild_appended(MapArgs a) {
  const int lt = blockIdx.y;
  const int seg = lt * LVO_MSEGS + LVO_SEG_NONVALID;
  const unsigned b = a.vx.seg_out_start[seg], n = a.vx.seg_out_cnt[seg];
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned cube = a.vx.out_aux[b + i];
    atomicAdd(&a.app_cnt[(size_t)lt * LVO_NCUBES + cube], 1u);
    atomicMin(&a.app_first[(size_t)lt * LVO_NCUBES + cube], b + i);
  }
}
// one block per (lane, type): new per-cube counts and their exclusive scan.  A lane that does not map in this step counts as having
// no valid cube (its n_valid / valid_cube stay for lvo_map_cloud) and no shift (k_map_end left it 0): its map passes through unchanged.
// A lane with a fixed map (LVO_LANE_MAP_FIXED) also counts as having no valid cube, but with the shift k_map_begin computed in this
// step: its map passes through shifted, cubes that left the window dropped, and its n_map / totals are written.
__global__ void __launch_bounds__(256) k_rebuild_offsets(MapArgs a) {
  __shared__ unsigned sm[33];
  __shared__ signed char vrank[LVO_NCUBES];
  const int lt = blockIdx.x, lane = lt >> 1, t = lt & 1;
  LaneState& s = a.ls[lane];
  const bool maps = lane_maps(a.lane_flags, lane), updates = lane_updates_map(a.lane_flags, lane);
  for (int c = threadIdx.x; c < LVO_NCUBES; c += blockDim.x) vrank[c] = -1;
  __syncthreads();
  if (updates && threadIdx.x < s.n_valid) vrank[s.valid_cube[threadIdx.x]] = (signed char)threadIdx.x;
  __syncthreads();
  const unsigned* cs = a.cube_start[a.gen][t] + (size_t)lane * (LVO_NCUBES + 1);
  unsigned* ncs = a.cube_start[a.gen ^ 1][t] + (size_t)lane * (LVO_NCUBES + 1);
  unsigned carry = 0;
  for (int base = 0; base < LVO_NCUBES; base += blockDim.x) {
    const int c = base + threadIdx.x;
    unsigned cnt = 0;
    if (c < LVO_NCUBES) {
      const int v = vrank[c];
      if (v >= 0) cnt = a.vx.seg_out_cnt[lt * LVO_MSEGS + v];
      else {
        const int i = c % LVO_CUBE_W - s.shift[0], j = (c / LVO_CUBE_W) % LVO_CUBE_H - s.shift[1], k = c / (LVO_CUBE_W * LVO_CUBE_H) - s.shift[2];
        if (i >= 0 && i < LVO_CUBE_W && j >= 0 && j < LVO_CUBE_H && k >= 0 && k < LVO_CUBE_D) { const int oc = cube_index(i, j, k); cnt = cs[oc + 1] - cs[oc]; }
        cnt += a.app_cnt[(size_t)lt * LVO_NCUBES + c];
      }
    }
    unsigned tot;
    const unsigned ex = block_excl_scan(cnt, sm, &tot);
    // capacity overflow: the offsets are clamped to map_cap, so the cubes past the capacity lose their tail CONSISTENTLY (table,
    // n_map and the copy below agree) and the lane stays safe for the following frames; the frame reports LVO_E_CAPACITY
    if (c < LVO_NCUBES) ncs[c] = min(carry + ex, (unsigned)a.map_cap[t]);
    carry += tot;
  }
  if (threadIdx.x == 0) {
    const unsigned kept = min(carry, (unsigned)a.map_cap[t]);
    ncs[LVO_NCUBES] = kept;
    if (!maps) return;
    s.n_map[t] = (int)kept;
    if (t == 0) s.stats.map_corner_total = (int)kept; else s.stats.map_surf_total = (int)kept;
    if (carry > (unsigned)a.map_cap[t]) s.map_status = LVO_E_CAPACITY;
  }
}
// destination-parallel gather into the other generation
__global__ void __launch_bounds__(256) k_rebuild_copy(MapArgs a) {
  __shared__ signed char vrank[LVO_NCUBES];
  const int lt = blockIdx.y, lane = lt >> 1, t = lt & 1;
  const LaneState& s = a.ls[lane];
  const bool updates = lane_updates_map(a.lane_flags, lane);   // see k_rebuild_offsets
  for (int c = threadIdx.x; c < LVO_NCUBES; c += blockDim.x) vrank[c] = -1;
  __syncthreads();
  if (updates && threadIdx.x < s.n_valid) vrank[s.valid_cube[threadIdx.x]] = (signed char)threadIdx.x;
  __syncthreads();
  const unsigned* cs = a.cube_start[a.gen][t] + (size_t)lane * (LVO_NCUBES + 1);
  const unsigned* ncs = a.cube_start[a.gen ^ 1][t] + (size_t)lane * (LVO_NCUBES + 1);
  const float4* src = a.map_pts[a.gen][t] + (size_t)lane * a.map_cap[t];
  float4* dst = a.map_pts[a.gen ^ 1][t] + (size_t)lane * a.map_cap[t];
  const unsigned n = min(ncs[LVO_NCUBES], (unsigned)a.map_cap[t]);
  for (unsigned d = blockIdx.x * blockDim.x + threadIdx.x; d < n; d += gridDim.x * blockDim.x) {
    int lo = 0, hi = LVO_NCUBES - 1;  // last cube with ncs[c] <= d
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (ncs[mid] <= d) lo = mid; else hi = mid - 1; }
    const int c = lo;
    const unsigned r = d - ncs[c];
    const int v = vrank[c];
    float4 p;
    if (v >= 0) p = a.vx.out_pts[a.vx.seg_out_start[lt * LVO_MSEGS + v] + r];
    else {
      const int i = c % LVO_CUBE_W - s.shift[0], j = (c / LVO_CUBE_W) % LVO_CUBE_H - s.shift[1], k = c / (LVO_CUBE_W * LVO_CUBE_H) - s.shift[2];
      unsigned ocnt = 0, ob = 0;
      if (i >= 0 && i < LVO_CUBE_W && j >= 0 && j < LVO_CUBE_H && k >= 0 && k < LVO_CUBE_D) { const int oc = cube_index(i, j, k); ob = cs[oc]; ocnt = cs[oc + 1] - ob; }
      if (r < ocnt) p = src[ob + r];
      else p = a.vx.out_pts[a.app_first[(size_t)lt * LVO_NCUBES + c] + (r - ocnt)];
    }
    dst[d] = p;
  }
}
__global__ void k_map_end(MapArgs a) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= a.lanes) return;
  LaneState& s = a.ls[lane];
  s.shift[0] = s.shift[1] = s.shift[2] = 0;
}
__global__ void k_register(MapArgs a) {
  const int lane = blockIdx.y;
  const LaneState& s = a.ls[lane];
  const int n = s.n_kept;
  if (!lane_maps(a.lane_flags, lane)) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    a.registered[(size_t)lane * a.P + i] = transform_point(s.map_x, s.map_x + 4, a.full[(size_t)lane * a.P + i]);
}

static inline void lvo_launch_mapping(cudaStream_t st, MapArgs a, const SolveArgs& solve_proto, int outer_iters, int lanes, bool want_registered,
                                      long long* launches, LvoStageTimer* tm = nullptr) {
  const int L2 = 2 * lanes;
  LVO_MARK(tm, LVO_ST_MAP_PREPARE, st);
  k_map_begin<<<lvo_div_up(lanes, 64), 64, 0, st>>>(a);
  k_map_gather<<<dim3(LVO_MAX_VALID, L2), 128, 0, st>>>(a);
  k_stack_offsets<<<1, 256, 0, st>>>(a);
  k_stack_gather<<<dim3(16, L2), 256, 0, st>>>(a);
  if (launches) *launches += 4;
  int seg_bits = 1; while ((1 << seg_bits) < L2) seg_bits++;
  lvo_voxel_run(st, a.vx, lanes * (a.in_cap[0] + a.in_cap[1]), L2, seg_bits, launches);
  k_stack_scatter<<<dim3(8, L2), 256, 0, st>>>(a);
  if (launches) *launches += 1;
  LVO_MARK(tm, LVO_ST_MAP_TREE, st);
  lvo_grid_build(st, a.grid, launches);
  const int nstack_cap = a.in_cap[0] + a.in_cap[1];
  dim3 ga(max(1, min(lvo_div_up(nstack_cap, 128), 128)), lanes);
  // The reuse kernels loop over a lane's queries with few blocks: a stack holds ~4 k points (capacity 139 k), and every block of a
  // capacity-sized grid pays the dependent loads of the lane state before it can exit (16 384 blocks cost ~50 us when all of them are idle).
  dim3 gr(max(1, min(lvo_div_up(nstack_cap, 128), 32)), lanes), gf(max(1, min(lvo_div_up(nstack_cap, 128), 8)), lanes), gf2(max(1, min(lvo_div_up(nstack_cap, 128), 16)), lanes);
  for (int o = 0; o < outer_iters; ++o) {
    a.outer = o;
    LVO_MARK(tm, LVO_ST_MAP_KNN, st);
    if (a.knn_reuse) k_map_knn_reuse<<<gr, 128, 0, st>>>(a);
    else k_map_knn<<<ga, 128, 0, st>>>(a);
    LVO_MARK(tm, LVO_ST_MAP_FIT, st);
    if (a.knn_reuse) k_map_fit_reuse<<<o == 0 ? gr : (o <= 2 ? gf2 : gf), 128, 0, st>>>(a);   // ~25 % / 8 % / < 3 % of the rows change in iterations 1 / 2 / later
    else k_map_fit<<<ga, 128, 0, st>>>(a);
    if (launches) *launches += 1;
    SolveArgs sa = solve_proto;
    sa.lane_flags = a.lane_flags;
    sa.which = 1; sa.outer = o; sa.n_outer = outer_iters; sa.factors = a.factors; sa.factor_cap = a.factor_cap; sa.distort = 0; sa.reset_cnt = nullptr;  // LidarEdgeFactor(..., 1.0), :610
    LVO_MARK(tm, LVO_ST_MAP_SOLVER, st);
    lvo_launch_lm(st, sa, lanes, 16384);
    if (launches) *launches += 2;
  }
  LVO_MARK(tm, LVO_ST_MAP_ADD, st);
  k_map_finish<<<lvo_div_up(lanes, 64), 64, 0, st>>>(a);
  k_refilter_offsets<<<1, 256, 0, st>>>(a);
  k_refilter_gather<<<dim3(64, L2), 256, 0, st>>>(a);
  if (launches) *launches += 3;
  LVO_MARK(tm, LVO_ST_MAP_FILTER, st);
  int seg_bits2 = 1; while ((1 << seg_bits2) < L2 * LVO_MSEGS) seg_bits2++;
  lvo_voxel_run(st, a.vx, a.vx.cap_items, L2 * LVO_MSEGS, seg_bits2, launches);
  k_rebuild_reset<<<148, 256, 0, st>>>(a);
  k_rebuild_appended<<<dim3(4, L2), 256, 0, st>>>(a);
  k_rebuild_offsets<<<L2, 256, 0, st>>>(a);
  k_rebuild_copy<<<dim3(64, L2), 256, 0, st>>>(a);
  k_map_end<<<lvo_div_up(lanes, 64), 64, 0, st>>>(a);
  if (launches) *launches += 5;
  LVO_MARK(tm, LVO_ST_MAP_PUB, st);
  if (want_registered && a.registered) { k_register<<<dim3(64, lanes), 256, 0, st>>>(a); if (launches) *launches += 1; }
}
