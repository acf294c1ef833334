// lvo_odometry.cuh — lvo_scan_to_scan: the odometry frame body, reference src/laserOdometry.cpp:353-641.
// OdoArgs::distortion selects the compile-time switch of :67: 0 = DISTORTION 0 (the shipped value), 1 = DISTORTION 1 as the
// file is written (per-point interpolation ratio in TransformToStart :157-163 and in the factors :455-459 / :549-553; the
// TransformToEnd block :610-625 stays disabled by its `if (0)`), 2 = DISTORTION 1 with that block enabled (k_odo_to_end).
//
//   k_odo_begin      first-frame handling (:355-358), per-outer-iteration counter reset
//   k_odo_assoc      one 8-lane tile per feature (4 features per warp): TransformToStart (:154-172, s = 1), 1-NN in the previous sweep's
//                    less-sharp / less-flat cloud on the uniform grid with the d^2 < 25 gate (:386-389, :470-473),
//                    then the adjacent-ring searches of :395-440 / :481-532 as ring-filtered nearest-neighbour searches
//                    on the same grid (the clouds are ring-ordered by construction), with the reference's walk order
//                    as tie-break;
//                    emits LidarEdgeFactor / LidarPlaneFactor parameter records (:444-462, :536-557)
//   k_lm_solve       (lvo_solver.cuh) ceres::Solve, :571-576
//   k_odo_finish     pose integration :581-582, swap of the "last" clouds :627-636, ring-offset tables
//   lvo_grid_build   (lvo_knn.cuh) replaces kdtree->setInputCloud :640-641
#pragma once
#include "lvo_internal.h"
#include "lvo_knn.cuh"
#include "lvo_solver.cuh"

#define LVO_ODO_GRIDS 6         // search structures per lane over the previous sweep's two clouds
#define LVO_ODO_FAST_AZ_HALF 16 // widest azimuth half-window (buckets) the thread-per-feature kernel scans itself

struct OdoArgs {
  LaneState* ls;
  int lanes, outer;
  int distortion;    // 0 | 1 | 2, see the header comment
  const int* lane_flags;   // [lanes] LVO_LANE_* of the step: an idle lane's pose, "last" clouds, status and stats are left alone
  // current features (stride caps)
  const float4* sharp; float4* less_sharp; const float4* flat; float4* less_flat;
  float4* full;      // [lanes][P] ring-ordered full-resolution cloud (only touched by k_odo_to_end)
  int cap_sharp, cap_lsharp, cap_flat, P;
  // previous sweep
  float4* corner_last; float4* surf_last;  // [lanes][cap_lsharp], [lanes][P]
  GridSet grid;                            // problems LVO_ODO_GRIDS*lane + {0/1 corner/surf fine xyz, 2/3 corner/surf (ring,azimuth), 4/5 corner/surf middle xyz}
  LvoFactor* factors; int factor_cap;
  int* slow_list;    // [lanes][cap_sharp + cap_flat] features the fast kernel hands to the tile kernel
  int* slow_cnt;     // [lanes]
  int* corner_corr;  // [lanes][slots][cap_sharp][2]   probes; the association of outer iteration o reads those of o - 1
  int* plane_corr;   // [lanes][slots][cap_flat][3]
  int slots;         // outer-iteration slots kept: LVO_MAX_OUTER with lvo_config::debug_probes, else 2 (slot = outer % slots)
  // LVO_OPT_ODO_REUSE: certified reuse of a feature's correspondence across the outer iterations of a frame (see odo_certified)
  int reuse;
  float4* ref;       // [lanes][cap_sharp + cap_flat] feature position (TransformToStart) at its last full association
  float4* guard;     // [lanes][cap_sharp + cap_flat] guard radii of that association: x closest point, y same-ring point, z adjacent-ring point; w != 0: record valid
  int4* sel;         // [lanes][cap_sharp + cap_flat] what that association chose: x closest, y same-ring, z adjacent-ring point (-1: none inside the 5 m gate)
  LvoUncRaw* unc;    // [lanes][2] pose-uncertainty records (lvo_solver.cuh); k_odo_begin clears `solved` of stage 0
};

// ---- certified reuse of a correspondence across outer iterations (LVO_OPT_ODO_REUSE) ---------------------------------------------
// The outer iterations of a frame (:364) associate the SAME two clouds from a pose that moves less and less, and a factor record
// depends only on WHICH points were chosen (closest j; l / m in the same / adjacent rings), never on the pose.  A full association
// at position q_ref therefore also records, for each of its (up to) three searches, a GUARD radius: a lower bound on the distance
// from q_ref to every OTHER eligible point of that search — the smaller of the second-best candidate distance and the radius of the
// region that was scanned completely (box half-width, azimuth window, the 5 m gate).  At a later position q_new, moved by delta, every
// other eligible point is at least guard - delta away; if the chosen point's new distance is below that, and inside the 5 m gate
// (:389 / :473), it is still the strict minimum.  The eligibility of l / m depends only on j and on fixed ring ids and indices, so
// with j unchanged the filters are unchanged.  All three certified: the factor record stands and the feature is skipped.  Margins of
// 1e-4 relative + 1e-5 m dwarf float rounding and only decide WHETHER the shortcut is taken.
#define LVO_ODO_FEW 24       // uncertified features per block of 128 below which they are handed to the warp-per-feature kernel
#ifndef LVO_ODO_SLACK
#define LVO_ODO_SLACK 0.05f   // extra radius (m) scanned around a full association so that the next iterations can be certified
#endif
__device__ __forceinline__ float odo_guard_of(float d2_other, float region) {
  const float g = fminf(sqrtf(d2_other), region);
  return fmaxf(g * 0.9999f - 1e-5f, 0.f);
}
// radius around the query (horizontal range rho) inside which every point lies in the azimuth window of half-width h buckets
// (inverse of az_halfwidth: two buckets of the half-width are quantisation / rounding margin)
__device__ __forceinline__ float az_region(int h, float rho) {
  if (2 * h + 1 >= LVO_AZ_BUCKETS) return FLT_MAX;
  const float ang = (float)(h - 2) * (6.28318548f / (float)LVO_AZ_BUCKETS);
  if (ang <= 0.f) return 0.f;
  if (ang >= 1.5f) return rho * 0.99f;   // beyond ~86 degrees: a point outside the window is farther than rho sin(1.5)
  return rho * sinf(ang) * 0.999f;
}
__device__ __forceinline__ int az_halfwidth(float d2, float rho);
__device__ __forceinline__ int az_halfwidth_slack(float d2, float rho) {
  const float d = sqrtf(d2) + LVO_ODO_SLACK;
  return az_halfwidth(d * d, rho);
}
// true iff the choices of this feature's last full association (a.sel) are certified at `sel`: a chosen point is still the strict
// minimum of its search and inside the gate; a search that found nothing inside the gate still finds nothing.  p receives the choices.
__device__ __forceinline__ bool odo_certified(const OdoArgs& a, size_t fi, bool corner, float4 sel, const float4* C, int4& p) {
  const float4 g = a.guard[fi];
  if (g.w == 0.f) return false;
  p = a.sel[fi];
  const float4 r = a.ref[fi];
  const float dx = sel.x - r.x, dy = sel.y - r.y, dz = sel.z - r.z;
  const float delta = sqrtf(dx * dx + dy * dy + dz * dz) * 1.0001f + 1e-5f;
  auto still = [&](int idx, float guard) {
    if (idx < 0) return guard - delta > 5.001f;   // every eligible point stays outside the gate
    const float dd = sqdist3(C[idx], sel.x, sel.y, sel.z);
    return dd < 25.0f && sqrtf(dd) * 1.0001f + 1e-5f + delta < guard;
  };
  if (!still(p.x, g.x)) return false;
  if (p.x < 0) return true;   // no closest point inside the gate: no factor, as before
  return still(p.z, g.z) && (corner || still(p.y, g.y));
}

__global__ void k_odo_begin(OdoArgs a) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= a.lanes) return;
  LaneState& s = a.ls[lane];
  if (!lane_active(a.lane_flags, lane)) return;   // idle: the association and solve kernels return for it by its lane flags
  s.odo_status = s.odo_inited ? LVO_OK : LVO_W_FIRST_FRAME;
  s.odo_done = 0; s.stats.odo_outer_executed = 0;
  for (int o = 0; o < LVO_MAX_OUTER; ++o) { s.stats.odo_corner_corr[o] = 0; s.stats.odo_plane_corr[o] = 0; s.stats.odo_lm_iters[o] = 0; s.stats.odo_final_cost[o] = 0; s.stats.odo_slow[o] = 0; s.stats.odo_certified[o] = 0; }
  for (int k = 0; k < 6; ++k) s.stats.odo_slow_why[k] = 0;
  a.slow_cnt[lane] = 0;
  a.unc[2 * lane].solved = 0;   // set again by k_lm_solve unless this is the first frame
}

struct Best { float d; int pos; int j; };
__device__ __forceinline__ Best best_min(Best a, Best b) { return (b.d < a.d || (b.d == a.d && b.pos < a.pos)) ? b : a; }
// (d, pos) lexicographic minimum over the warp: two REDUX + ballot + shuffle (d >= 0 so its bit pattern orders like its value)
__device__ __forceinline__ Best warp_best(Best v) {
  const unsigned md = __reduce_min_sync(0xffffffffu, __float_as_uint(v.d));
  const bool dmin = __float_as_uint(v.d) == md;
  const unsigned mp = __reduce_min_sync(0xffffffffu, dmin ? (unsigned)v.pos : 0xffffffffu);
  const unsigned who = __ballot_sync(0xffffffffu, dmin && (unsigned)v.pos == mp);
  const int src = __ffs(who) - 1;
  Best r;
  r.d = __uint_as_float(md); r.pos = (int)mp; r.j = __shfl_sync(0xffffffffu, v.j, src);
  return r;
}

// The adjacent-ring searches of :395-440 / :481-532.  The reference walks the ring-ordered cloud upwards from the
// closest point, then downwards, and keeps the first strict minimum among the points of the wanted rings with
// d^2 < 25.  The same point is the ring-filtered nearest neighbour, with the position in the reference's walk as the
// tie-break key (indices above `closest` ascending, then indices below it descending).  It is searched on a
// (ring, azimuth) grid of the previous sweep: a point within distance d of the query lies within asin(d / rho_xy) of
// the query's azimuth, so only a window of azimuth buckets of each wanted ring is scanned: first +-2 buckets, then
// the window implied by the best distance found so far (or by the 5 m gate).  Margins of two buckets absorb every
// rounding in atan2f / asinf; the ranking itself uses the exact reference expression.
//   bestA : nearest point of the SAME ring (other than closest)       -> minPointInd2 of the plane search
//   bestB : nearest point of rings cid-2, cid-1, cid+1, cid+2         -> minPointInd2 (corner) / minPointInd3 (plane)
// candidate range(s) of buckets lo..hi of one ring (lo / hi may lie outside [0, NB): wrap).  part 0 / part 1.
__device__ __forceinline__ void az_bounds(const GridView& g, int ring, int lo, int hi, int part, unsigned& b, unsigned& e) {
  b = e = 0;
  if (hi < lo) return;
  const unsigned* row = g.cell_start + ring * LVO_AZ_BUCKETS;
  if (hi - lo + 1 >= LVO_AZ_BUCKETS) { if (part == 0) { b = __ldg(row); e = __ldg(row + LVO_AZ_BUCKETS); } return; }
  const int l = lo & (LVO_AZ_BUCKETS - 1), h = hi & (LVO_AZ_BUCKETS - 1);
  if (l <= h) { if (part == 0) { b = __ldg(row + l); e = __ldg(row + h + 1); } }
  else if (part == 0) { b = __ldg(row + l); e = __ldg(row + LVO_AZ_BUCKETS); }
  else { b = __ldg(row); e = __ldg(row + h + 1); }
}
// half-width (in buckets) of the azimuth window that contains every point within sqrt(d2) of the query
__device__ __forceinline__ int az_halfwidth(float d2, float rho) {
  const float d = sqrtf(d2) * 1.00001f + 1e-6f;
  if (!(d < rho * 0.999f)) return LVO_AZ_BUCKETS;  // the window is the whole ring
  const float w = asinf(d / rho);
  return (int)ceilf(w * ((float)LVO_AZ_BUCKETS / 6.28318548f)) + 2;
}
// ---- one 8-lane tile per feature (four features per warp); every call below is made by all 32 lanes --------------------
// rows 3k .. 3k+2 (k = part) of the 3x3 row block around (cx, cy, cz): lanes 0..2 of the tile fetch the bounds
template <int TW>
__device__ __forceinline__ void tile_block_nn1(const GridView& g, bool active, float4 sel, float& d, int& id, float& d2) {
  const int tl = (int)tile_lane<TW>();
  const int cx = cell_coord(sel.x, g.inv_cell) - g.org[0], cy = cell_coord(sel.y, g.inv_cell) - g.org[1], cz = cell_coord(sel.z, g.inv_cell_z) - g.org[2];
  auto consider = [&](float4 p, int) {
    const int i = __float_as_int(p.w);
    const float dd = sqdist3(p, sel.x, sel.y, sel.z);
    if (dd < d || (dd == d && i < id)) { if (id != INT_MAX) d2 = fminf(d2, d); d = dd; id = i; }
    else if (i != id) d2 = fminf(d2, dd);   // d2: best distance among the other candidates (guard radius of LVO_OPT_ODO_REUSE)
  };
  for (int base = 0; base < 9; base += TW) {   // 9 rows: two steps for 8-lane tiles, one for full warps
    const int row = base + tl;
    unsigned b = 0, e = 0;
    if (active && g.dim[0] > 0 && row < 9) row_bounds(g, cz + row / 3 - 1, cy + row % 3 - 1, cx - 1, cx + 1, b, e);
    tile_scan_ranges<TW, (TW < 9 ? TW : 9)>(g.pts, b, e, consider);
  }
}
// Box query: every cell that intersects [q - rad, q + rad] (at most 3 x 3 rows when rad < cell).  Used when an upper bound
// on the nearest-neighbour distance is known (the previous outer iteration's closest point): any point that beats or ties
// the bound lies inside the box.
template <int TW>
__device__ __forceinline__ void tile_box_nn1(const GridView& g, bool active, float4 sel, float rad, float& d, int& id, float& d2) {
  const int tl = (int)tile_lane<TW>();
  auto consider = [&](float4 p, int) {
    const int i = __float_as_int(p.w);
    const float dd = sqdist3(p, sel.x, sel.y, sel.z);
    if (dd < d || (dd == d && i < id)) { if (id != INT_MAX) d2 = fminf(d2, d); d = dd; id = i; }
    else if (i != id) d2 = fminf(d2, dd);   // d2: best distance among the other candidates (guard radius of LVO_OPT_ODO_REUSE)
  };
  const int x0 = cell_coord(sel.x - rad, g.inv_cell) - g.org[0], x1 = cell_coord(sel.x + rad, g.inv_cell) - g.org[0];
  const int y0 = cell_coord(sel.y - rad, g.inv_cell) - g.org[1], y1 = cell_coord(sel.y + rad, g.inv_cell) - g.org[1];
  const int z0 = cell_coord(sel.z - rad, g.inv_cell_z) - g.org[2], z1 = cell_coord(sel.z + rad, g.inv_cell_z) - g.org[2];
  const int ny = y1 - y0 + 1, nrows = ny * (z1 - z0 + 1);   // <= 9 by construction (rad < cell)
  for (int base = 0; base < 9; base += TW) {
    if (base > 0 && !__any_sync(0xffffffffu, active && nrows > base)) break;
    const int row = base + tl;
    unsigned b = 0, e = 0;
    if (active && g.dim[0] > 0 && row < nrows) row_bounds(g, z0 + row / ny, y0 + row % ny, x0, x1, b, e);
    tile_scan_ranges<TW, (TW < 9 ? TW : 9)>(g.pts, b, e, consider);
  }
}
// Shell r >= 2 of a grid, TW/2 rows per step.  Rows (and end cells) whose cell box is farther from the query than the
// current bound min(best, gate) are skipped: a point `k` cells away along an axis is more than (k - 1) cells away.
template <int TW>
__device__ __forceinline__ void tile_shell_nn1(const GridView& g, bool active, float4 sel, int r, float gate, float& d, int& id, float& d2) {
  const int tl = (int)tile_lane<TW>();
  constexpr int H = TW / 2;
  const int cx = cell_coord(sel.x, g.inv_cell) - g.org[0], cy = cell_coord(sel.y, g.inv_cell) - g.org[1], cz = cell_coord(sel.z, g.inv_cell_z) - g.org[2];
  auto consider = [&](float4 p, int) {
    const int i = __float_as_int(p.w);
    const float dd = sqdist3(p, sel.x, sel.y, sel.z);
    if (dd < d || (dd == d && i < id)) { if (id != INT_MAX) d2 = fminf(d2, d); d = dd; id = i; }
    else if (i != id) d2 = fminf(d2, dd);   // d2: best distance among the other candidates (guard radius of LVO_OPT_ODO_REUSE)
  };
  const float cz_size = 1.0f / g.inv_cell_z;
  const int side = 2 * r + 1, nrows = side * side;
  for (int base = 0; base < nrows; base += H) {   // lanes 0..H-1 left / full part, lanes H..TW-1 right part
    const int row = base + (tl % H);
    unsigned b = 0, e = 0;
    if (active && row < nrows) {
      const int dz = row / side - r, dy = row % side - r;
      const float gz = (float)max(abs(dz) - 1, 0) * cz_size, gy = (float)max(abs(dy) - 1, 0) * g.cell;
      const float bound = fminf(d, gate);
      if (!(gz * gz + gy * gy > bound)) {
        const bool edge = dz == -r || dz == r || dy == -r || dy == r;
        if (edge) { if (tl < H) row_bounds(g, cz + dz, cy + dy, cx - r, cx + r, b, e); }
        else {
          const float gx = (float)(r - 1) * g.cell;
          if (!(gz * gz + gy * gy + gx * gx > bound)) row_bounds(g, cz + dz, cy + dy, tl < H ? cx - r : cx + r, tl < H ? cx - r : cx + r, b, e);
        }
      }
    }
    tile_scan_ranges<TW, TW>(g.pts, b, e, consider);
  }
}

// factor record + correspondence probes of one feature (laserOdometry.cpp:442-462 / :534-557); returns the factor type
__device__ __forceinline__ int odo_emit(const OdoArgs& a, int lane, int f, int ns, bool corner, bool ok, float4 pt, const float4* C, int closest, float4 pj,
                                        int same, int other, float4 sel = make_float4(0.f, 0.f, 0.f, 0.f), float4 guard = make_float4(0.f, 0.f, 0.f, 0.f)) {
  if (a.reuse) {
    const size_t fi = (size_t)lane * (a.cap_sharp + a.cap_flat) + f;
    a.ref[fi] = sel; a.guard[fi] = guard;
    a.sel[fi] = make_int4(ok ? closest : -1, ok ? same : -1, ok ? other : -1, 0);
  }
  LvoFactor fac;
  fac.type = -1; fac.pad = 0;
  fac.d = distortion_ratio(pt.w, a.distortion);   // s of LidarEdgeFactor / LidarPlaneFactor, :455-459 / :549-553
  int i1 = -1, i2 = -1, i3 = -1;
  if (ok) {
    if (corner) {
      if (other >= 0) {
        i1 = closest; i2 = other;
        const float4 pb = C[other];
        fac.type = 0;
        fac.c[0] = pt.x; fac.c[1] = pt.y; fac.c[2] = pt.z;
        fac.a[0] = pj.x; fac.a[1] = pj.y; fac.a[2] = pj.z;
        const double lb[3] = {pb.x, pb.y, pb.z};
        lvo_edge_direction(fac.a, lb, fac.b);
      }
    } else if (same >= 0 && other >= 0) {
      i1 = closest; i2 = same; i3 = other;
      const float4 pl = C[same], pm = C[other];
      // LidarPlaneFactor constructor, lidarFactor.hpp:64-65
      const d3 jl{(double)pj.x - (double)pl.x, (double)pj.y - (double)pl.y, (double)pj.z - (double)pl.z};
      const d3 jm{(double)pj.x - (double)pm.x, (double)pj.y - (double)pm.y, (double)pj.z - (double)pm.z};
      d3 n = d3cross(jl, jm);
      const double nn = sqrt(n.x * n.x + n.y * n.y + n.z * n.z);
      fac.type = 1;
      fac.c[0] = pt.x; fac.c[1] = pt.y; fac.c[2] = pt.z;
      fac.a[0] = pj.x; fac.a[1] = pj.y; fac.a[2] = pj.z;
      fac.b[0] = n.x / nn; fac.b[1] = n.y / nn; fac.b[2] = n.z / nn;
    }
  }
  a.factors[(size_t)lane * a.factor_cap + f] = fac;
  if (corner) {
    int* c = a.corner_corr + (((size_t)lane * a.slots + a.outer % a.slots) * a.cap_sharp + f) * 2;
    c[0] = i1; c[1] = i2;
  } else {
    int* c = a.plane_corr + (((size_t)lane * a.slots + a.outer % a.slots) * a.cap_flat + (f - ns)) * 3;
    c[0] = i1; c[1] = i2; c[2] = i3;
  }
  return fac.type;
}

// Fast path for outer iterations >= 1: ONE THREAD per feature.  A feature qualifies when the previous outer iteration
// produced a factor for it (so the previous closest / same-ring / adjacent-ring points exist and bound the new searches)
// and the bounds are tight enough for a box query on the fine grid; every search then touches a handful of candidates and
// the per-feature overhead is shared by 32 features per warp instead of 4.  Features that do not qualify are appended to
// `slow_list` and processed by the tile kernel below.  Same results: both paths compute exact minima with the same keys.
// four independent loads in flight per thread
template <class F>
__device__ __forceinline__ void scan_range4(const float4* __restrict__ pts, unsigned b, unsigned e, F&& f) {
  for (unsigned t = b; t < e; t += 4) {
    const unsigned last = e - 1;
    const float4 p0 = __ldg(pts + t), p1 = __ldg(pts + min(t + 1, last)), p2 = __ldg(pts + min(t + 2, last)), p3 = __ldg(pts + min(t + 3, last));
    f(p0);
    if (t + 1 < e) f(p1);
    if (t + 2 < e) f(p2);
    if (t + 3 < e) f(p3);
  }
}

__global__ void __launch_bounds__(128) k_odo_assoc_fast(OdoArgs a) {
  __shared__ GridView gv[4];
  const int lane = blockIdx.y;
  LaneState& s = a.ls[lane];
  if (!lane_active(a.lane_flags, lane) || !s.odo_inited || s.odo_done) return;   // idle / first frame / fixed point reached (LVO_OPT_FIXPOINT_SKIP)
  if (threadIdx.x < 4) gv[threadIdx.x] = grid_view(a.grid, LVO_ODO_GRIDS * lane + threadIdx.x);
  __syncthreads();
  const int ns = s.n_sharp, nf = s.n_flat;
  const int f0 = blockIdx.x * blockDim.x + threadIdx.x;
  int made_c = 0, made_p = 0;
  bool certified = false;
  int f = f0;
  if (a.reuse && a.outer > 0) {
    // ---- phase A (LVO_OPT_ODO_REUSE), one thread per feature: certificate of the previous iteration's correspondence.  The features
    // that fail are compacted, so that the searches below run in full warps instead of one lane per warp.
    __shared__ int s_list[128];
    __shared__ int s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    bool need = false;
    if (f0 < ns + nf) {
      const bool corner = f0 < ns;
      const float4* C = corner ? a.corner_last + (size_t)lane * a.cap_lsharp : a.surf_last + (size_t)lane * a.P;
      const float4 pt = corner ? a.sharp[(size_t)lane * a.cap_sharp + f0] : a.flat[(size_t)lane * a.cap_flat + (f0 - ns)];
      const float4 sel = transform_to_start(s.para_q, s.para_t, pt, a.distortion);
      int4 p;
      certified = odo_certified(a, (size_t)lane * (a.cap_sharp + a.cap_flat) + f0, corner, sel, C, p);
      if (certified) {
        // same choices as in the last full association: the factor record (or its absence) stands; this iteration's row repeats it
        const bool valid = p.x >= 0 && p.z >= 0 && (corner || p.y >= 0);
        if (corner) { int* c = a.corner_corr + (((size_t)lane * a.slots + a.outer % a.slots) * a.cap_sharp + f0) * 2; c[0] = valid ? p.x : -1; c[1] = valid ? p.z : -1; }
        else { int* c = a.plane_corr + (((size_t)lane * a.slots + a.outer % a.slots) * a.cap_flat + (f0 - ns)) * 3; c[0] = valid ? p.x : -1; c[1] = valid ? p.y : -1; c[2] = valid ? p.z : -1; }
        if (valid) { if (corner) made_c++; else made_p++; }
      } else need = true;
    }
    const unsigned m = __ballot_sync(0xffffffffu, need);
    int off = 0;
    if ((threadIdx.x & 31) == 0 && m) off = atomicAdd(&s_n, __popc(m));
    off = __shfl_sync(0xffffffffu, off, 0);
    if (need) s_list[off + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = f0;
    __syncthreads();
    f = (int)threadIdx.x < s_n ? s_list[threadIdx.x] : ns + nf;
    // A handful of features left in this block (typical from the third iteration on): one thread each would walk its searches as a
    // chain of ~100 dependent loads with nothing else in flight — ~130 us of pure latency per launch.  They go to the warp-per-feature
    // kernel, which is launched anyway.
    if (s_n <= LVO_ODO_FEW) {
      if (f < ns + nf) {
        a.slow_list[(size_t)lane * (a.cap_sharp + a.cap_flat) + atomicAdd(&a.slow_cnt[lane], 1)] = f;
        atomicAdd(&s.stats.odo_slow[a.outer], 1); atomicAdd(&s.stats.odo_slow_why[5], 1);
      }
      f = ns + nf;
    }
  }
  if (f < ns + nf) {
    const bool corner = f < ns;
    const float4* C = corner ? a.corner_last + (size_t)lane * a.cap_lsharp : a.surf_last + (size_t)lane * a.P;
    const GridView& g = gv[corner ? 0 : 1];
    const GridView& gaz = gv[corner ? 2 : 3];
    const float4 pt = corner ? a.sharp[(size_t)lane * a.cap_sharp + f] : a.flat[(size_t)lane * a.cap_flat + (f - ns)];
    const float4 sel = transform_to_start(s.para_q, s.para_t, pt, a.distortion);
    int pc = -1, pA = -1, pB = -1;
    if (a.outer > 0) {
      if (a.reuse) {   // what the last full association chose, also when it produced no factor (any of them is a valid bound)
        const int4 p = a.sel[(size_t)lane * (a.cap_sharp + a.cap_flat) + f];
        pc = p.x; pA = p.y; pB = p.z;
      } else if (corner) { const int* c = a.corner_corr + (((size_t)lane * a.slots + (a.outer - 1) % a.slots) * a.cap_sharp + f) * 2; pc = c[0]; pB = c[1]; }
      else { const int* c = a.plane_corr + (((size_t)lane * a.slots + (a.outer - 1) % a.slots) * a.cap_flat + (f - ns)) * 3; pc = c[0]; pA = c[1]; pB = c[2]; }
    }
    {
    float d = FLT_MAX, d2c = FLT_MAX; int id = INT_MAX;
    auto near = [&](float4 p) {
      const int i = __float_as_int(p.w);
      const float dd = sqdist3(p, sel.x, sel.y, sel.z);
      if (dd < d || (dd == d && i < id)) { if (id != INT_MAX) d2c = fminf(d2c, d); d = dd; id = i; }
      else if (i != id) d2c = fminf(d2c, dd);
    };
    const int cx = cell_coord(sel.x, g.inv_cell) - g.org[0], cy = cell_coord(sel.y, g.inv_cell) - g.org[1], cz = cell_coord(sel.z, g.inv_cell_z) - g.org[2];
    // ---- bound on the closest point: the previous iteration's closest point, else the best point of the query's own cell
    if (pc >= 0) { d = sqdist3(C[pc], sel.x, sel.y, sel.z); id = pc; }
    else if (g.dim[0] > 0) { unsigned b, e; row_bounds(g, cz, cy, cx, cx, b, e); scan_range4(g.pts, b, e, near); }
    d2c = FLT_MAX;   // the second-best distance is taken from the box query below, which sees every point inside the box (the bound itself again too)
    float rad = sqrtf(d) * 1.0001f + 1e-5f;
    if (a.reuse && rad + LVO_ODO_SLACK < g.cell) rad += LVO_ODO_SLACK;   // a little more than needed: room for the next iterations' certificates
    // (a box query on the 2 m middle grid for bounds between 0.5 and 2 m was tried here: it halves the list handed to the warp-per-feature
    // kernel but one thread then walks a (4 m)^3 box while its warp waits — association time went from 4.1 to 5.1 ms per 128-lane frame)
    bool fast = id != INT_MAX && rad < g.cell && (double)d < 25.0;
    int why = id == INT_MAX ? 0 : (!(rad < g.cell) ? 1 : 2);
    int closest = -1, same = -1, other = -1;
    float4 pj = make_float4(0.f, 0.f, 0.f, 0.f), guard = make_float4(0.f, 0.f, 0.f, 0.f);
    if (fast) {
      // ---- closest point: box query on the fine grid (every cell that intersects [q - rad, q + rad])
      const int x0 = cell_coord(sel.x - rad, g.inv_cell) - g.org[0], x1 = cell_coord(sel.x + rad, g.inv_cell) - g.org[0];
      const int y0 = cell_coord(sel.y - rad, g.inv_cell) - g.org[1], y1 = cell_coord(sel.y + rad, g.inv_cell) - g.org[1];
      const int z0 = cell_coord(sel.z - rad, g.inv_cell_z) - g.org[2], z1 = cell_coord(sel.z + rad, g.inv_cell_z) - g.org[2];
      unsigned rb[9], re[9];   // rad < cell: at most 3 x 3 rows; all bounds are fetched before the first candidate
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        rb[k] = re[k] = 0;
        const int z = z0 + k / 3, y = y0 + k % 3;
        if (z <= z1 && y <= y1) row_bounds(g, z, y, x0, x1, rb[k], re[k]);
      }
      // one copy of the scan body (the kernel is instruction-fetch bound when these loops are unrolled: 129 KB of SASS)
#pragma unroll 1
      for (int k = 0; k < 9; ++k) scan_range4(g.pts, rb[k], re[k], near);
      closest = id;
      pj = C[closest];
      const int cid = ring_clamped(pj.w);
      // ---- adjacent-ring searches.  Seeds: the previous iteration's points if they still pass the ring filter, else
      // the best points of the +-2 bucket windows.
      Best bA{25.0f, INT_MAX, -1}, bB{25.0f, INT_MAX, -1};
      float d2A = FLT_MAX, d2B = FLT_MAX;   // best distance among the OTHER eligible candidates of each search (guard radii)
      auto upd = [&](Best& b, float& d2, const Best& c) {
        if (c.j == b.j) return;   // the seed met again in its bucket
        if (c.d < b.d || (c.d == b.d && c.pos < b.pos)) { if (b.j >= 0) d2 = fminf(d2, b.d); b = c; }
        else d2 = fminf(d2, c.d);
      };
      auto seed = [&](int pidx, bool same_ring, Best& best) {
        if (pidx < 0 || pidx == closest) return;
        const float4 p = C[pidx];
        const int dr = ring_clamped(p.w) - cid;
        if (same_ring ? (dr != 0) : (dr == 0 || dr > 2 || dr < -2)) return;
        if ((pidx > closest && dr < 0) || (pidx < closest && dr > 0)) return;
        const float dd = (p.x - sel.x) * (p.x - sel.x) + (p.y - sel.y) * (p.y - sel.y) + (p.z - sel.z) * (p.z - sel.z);
        if (!(dd < 25.0f)) return;
        best = Best{dd, pidx > closest ? (pidx - closest) : ((closest - pidx) + (1 << 30)), pidx};
      };
      if (!corner) seed(pA, true, bA);
      seed(pB, false, bB);
      const float rho = sqrtf(sel.x * sel.x + sel.y * sel.y);
      const int bq = az_bucket(sel.x, sel.y);
      int dr_cur = 0;
      auto cand = [&](float4 p) {
        const int idx = __float_as_int(p.w);
        if (idx == closest) return;
        if ((idx > closest && dr_cur < 0) || (idx < closest && dr_cur > 0)) return;
        const float dd = (p.x - sel.x) * (p.x - sel.x) + (p.y - sel.y) * (p.y - sel.y) + (p.z - sel.z) * (p.z - sel.z);
        if (!(dd < 25.0f)) { if (dr_cur == 0) d2A = fminf(d2A, dd); else d2B = fminf(d2B, dd); return; }   // eligible, beyond the gate: only bounds the guard
        const Best c{dd, idx > closest ? (idx - closest) : ((closest - idx) + (1 << 30)), idx};
        if (dr_cur == 0) upd(bA, d2A, c); else upd(bB, d2B, c);
      };
      // window k = (ring slot r = k >> 1 <-> ring cid - 2 + r, side = k & 1); buckets with |offset| <= skip were scanned before
      auto window = [&](int k, int hA, int hB, int skipA, int skipB, int& lo, int& hi) -> bool {
        const int r = k >> 1, side = k & 1, ring = cid - 2 + r;
        if (ring < 0 || ring >= LVO_AZ_RINGS || (r == 2 && corner)) return false;
        const int h = r == 2 ? hA : hB, skip = r == 2 ? skipA : skipB;
        if (h <= skip) return false;
        if (skip < 0) { if (side) return false; lo = bq - h; hi = bq + h; }
        else if (side == 0) { lo = bq - h; hi = bq - skip - 1; }
        else { lo = bq + skip + 1; hi = bq + h; }
        return true;
      };
      int sA = -1, sB = -1;   // half-widths already scanned
      const bool first_needed = (!corner && bA.j < 0) || bB.j < 0;   // no seed for some target: first look at +-2 buckets
#pragma unroll 1
      for (int pass = first_needed ? 0 : 1; pass < 2; ++pass) {
        int hA, hB, skipA, skipB;
        if (pass == 0) {
          const int wA = (!corner && bA.j < 0) ? 2 : -1, wB = bB.j < 0 ? 2 : -1;
          hA = wA < 0 ? 0 : wA; hB = wB < 0 ? 0 : wB; skipA = wA < 0 ? 0 : -1; skipB = wB < 0 ? 0 : -1;
          if (wA >= 0) sA = wA;
          if (wB >= 0) sB = wB;
        } else {
          // with LVO_OPT_ODO_REUSE the windows reach LVO_ODO_SLACK beyond the best distances: room for the next iterations' certificates
          hA = corner ? 0 : (bA.j >= 0 ? (a.reuse ? az_halfwidth_slack(bA.d, rho) : az_halfwidth(bA.d, rho)) : LVO_AZ_BUCKETS);
          hB = bB.j >= 0 ? (a.reuse ? az_halfwidth_slack(bB.d, rho) : az_halfwidth(bB.d, rho)) : LVO_AZ_BUCKETS;
          if (hA > LVO_ODO_FAST_AZ_HALF || hB > LVO_ODO_FAST_AZ_HALF) {   // a target has no candidate nearby or its window is wide: leave it to the cooperative kernel
            fast = false; why = ((!corner && bA.j < 0) || bB.j < 0) ? 4 : 3; break;
          }
          skipA = corner ? hA : sA; skipB = sB;
          sA = max(sA, hA); sB = max(sB, hB);   // half-widths scanned completely once this pass is through
        }
        unsigned wb[10], we[10];   // part 0 of every bucket range; fetched together before any candidate
#pragma unroll
        for (int k = 0; k < 10; ++k) {
          wb[k] = we[k] = 0;
          int lo, hi;
          if (window(k, hA, hB, skipA, skipB, lo, hi)) az_bounds(gaz, cid - 2 + (k >> 1), lo, hi, 0, wb[k], we[k]);
        }
#pragma unroll 1
        for (int k = 0; k < 10; ++k) { dr_cur = (k >> 1) - 2; scan_range4(gaz.pts, wb[k], we[k], cand); }
        // wrapped windows (the range crosses bucket 0): second part, rare
        const int hmax = max(hA, hB);
        if (bq - hmax < 0 || bq + hmax >= LVO_AZ_BUCKETS) {
#pragma unroll 1
          for (int k = 0; k < 10; ++k) {
            int lo, hi;
            if (!window(k, hA, hB, skipA, skipB, lo, hi)) continue;
            unsigned b, e;
            az_bounds(gaz, cid - 2 + (k >> 1), lo, hi, 1, b, e);
            dr_cur = (k >> 1) - 2;
            scan_range4(gaz.pts, b, e, cand);
          }
        }
      }
      if (fast) {
        same = bA.j; other = bB.j;
        guard = make_float4(odo_guard_of(d2c, rad), corner ? 0.f : odo_guard_of(d2A, az_region(sA, rho)), odo_guard_of(d2B, az_region(sB, rho)), 1.f);
      }
    }
    if (fast) {
      const int type = odo_emit(a, lane, f, ns, corner, true, pt, C, closest, pj, same, other, sel, guard);
      if (type >= 0) { if (corner) made_c++; else made_p++; }
    } else {
      a.slow_list[(size_t)lane * (a.cap_sharp + a.cap_flat) + atomicAdd(&a.slow_cnt[lane], 1)] = f;
      atomicAdd(&s.stats.odo_slow[a.outer], 1); atomicAdd(&s.stats.odo_slow_why[why], 1);
    }
    }
  }
  const int nc = __reduce_add_sync(0xffffffffu, made_c), np = __reduce_add_sync(0xffffffffu, made_p);
  const int ncert = __popc(__ballot_sync(0xffffffffu, certified));
  if ((threadIdx.x & 31) == 0) {
    if (nc) atomicAdd(&s.stats.odo_corner_corr[a.outer], nc);
    if (np) atomicAdd(&s.stats.odo_plane_corr[a.outer], np);
    if (ncert) atomicAdd(&s.stats.odo_certified[a.outer], ncert);
  }
}

// tile-wide best (d, id) in every lane; a lane whose own best lost folds it into its second-best distance first
template <int TW>
__device__ __forceinline__ void tile_best_merge(float& d, int& id, float& d2) {
  const float dl = d; const int il = id;
  int key = id;
  tile_min3<TW>(d, key, id);
  if (il != id && il != INT_MAX) d2 = fminf(d2, dl);
}
template <int TW>
__device__ __forceinline__ void tile_best_merge(Best& b, float& d2) {
  const float dl = b.d; const int jl = b.j;
  tile_min3<TW>(b.d, b.pos, b.j);
  if (jl != b.j && jl >= 0) d2 = fminf(d2, dl);
}
template <int TW>
__device__ __forceinline__ float tile_min_f(float v) {
#pragma unroll
  for (int o = TW / 2; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o, TW));
  return v;
}

template <int TW>
__global__ void __launch_bounds__(256, 4) k_odo_assoc(OdoArgs a) {
  __shared__ GridView gv[LVO_ODO_GRIDS];
  const int lane = blockIdx.y;
  LaneState& s = a.ls[lane];
  if (!lane_active(a.lane_flags, lane) || !s.odo_inited || s.odo_done) return;   // idle / first frame / fixed point reached (LVO_OPT_FIXPOINT_SKIP)
  if (threadIdx.x < LVO_ODO_GRIDS) gv[threadIdx.x] = grid_view(a.grid, LVO_ODO_GRIDS * lane + threadIdx.x);
  __syncthreads();
  const int ns = s.n_sharp, nf = s.n_flat;
  const int tl = (int)tile_lane<TW>();
  // one tile per feature the fast kernel could not take
  const int nwork = a.slow_cnt[lane];   // the features the fast kernel could not take
  const int tiles_total = (gridDim.x * blockDim.x) / TW;
  for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) / TW;; slot += tiles_total) {
  if (__all_sync(0xffffffffu, slot >= nwork)) break;                // whole warp idle
  const bool have = slot < nwork;
  const int f = have ? a.slow_list[(size_t)lane * (a.cap_sharp + a.cap_flat) + slot] : ns + nf;
  const bool corner = f < ns;
  const double* q = s.para_q; const double* t = s.para_t;
  const float4* C = corner ? a.corner_last + (size_t)lane * a.cap_lsharp : a.surf_last + (size_t)lane * a.P;
  const GridView& gfine = gv[corner ? 0 : 1];
  const GridView& gaz = gv[corner ? 2 : 3];
  const GridView& gmid = gv[corner ? 4 : 5];
  float4 pt = make_float4(0.f, 0.f, 0.f, 0.f), sel = pt;
  if (have) {
    pt = corner ? a.sharp[(size_t)lane * a.cap_sharp + f] : a.flat[(size_t)lane * a.cap_flat + (f - ns)];
    sel = transform_to_start(q, t, pt, a.distortion);  // TransformToStart
  }
  // ---- closest point (laserOdometry.cpp:386 / :470, gate :389 / :473): the 27 cells around the query on the fine grid
  // (0.5 m) settle it when the best squared distance is below cell^2; otherwise the middle grid (2 m), then the coarse
  // grid (8 m, whose 27 cells cover the whole 5 m gate), then coarse shells if the cells had to be enlarged.
  float d = FLT_MAX, d2c = FLT_MAX, region_c = 0.f; int id = INT_MAX;
  // Upper bounds from the previous outer iteration of this frame (same clouds, slightly different pose): the points found
  // then still exist, so their distances to the new query bound the new minima and the searches shrink to a small box /
  // azimuth window.  Results are identical to the unbounded search.
  int pc = -1, pA = -1, pB = -1;
  if (have && a.outer > 0) {
    if (a.reuse) {   // what the last full association chose, also when it produced no factor
      const int4 p = a.sel[(size_t)lane * (a.cap_sharp + a.cap_flat) + f];
      pc = p.x; pA = p.y; pB = p.z;
    } else if (corner) { const int* c = a.corner_corr + (((size_t)lane * a.slots + (a.outer - 1) % a.slots) * a.cap_sharp + f) * 2; pc = c[0]; pB = c[1]; }
    else { const int* c = a.plane_corr + (((size_t)lane * a.slots + (a.outer - 1) % a.slots) * a.cap_flat + (f - ns)) * 3; pc = c[0]; pA = c[1]; pB = c[2]; }
  }
  bool boxed = false, boxed_mid = false;
  float rad = 0.f;
  if (pc >= 0) {
    const float dp = sqdist3(C[pc], sel.x, sel.y, sel.z);
    rad = sqrtf(dp) * 1.0001f + 1e-5f;
    if (rad < gfine.cell) { boxed = true; d = dp; id = pc; if (a.reuse && rad + LVO_ODO_SLACK < gfine.cell) rad += LVO_ODO_SLACK; }
    else if (rad < gmid.cell && gmid.dim[0] > 0) {   // bound between a fine and a middle cell: box on the 2 m grid
      boxed_mid = true; d = dp; id = pc;
      if (a.reuse && rad + LVO_ODO_SLACK < gmid.cell) rad += LVO_ODO_SLACK;
    }
  }
  // region_c: radius around the query inside which EVERY point of the cloud has been looked at (guard radius of LVO_OPT_ODO_REUSE)
  if (__any_sync(0xffffffffu, boxed)) {
    tile_box_nn1<TW>(gfine, boxed, sel, rad, d, id, d2c);
    tile_best_merge<TW>(d, id, d2c);
  }
  if (__any_sync(0xffffffffu, boxed_mid)) {
    tile_box_nn1<TW>(gmid, boxed_mid, sel, rad, d, id, d2c);
    tile_best_merge<TW>(d, id, d2c);
  }
  if (boxed || boxed_mid) region_c = rad;
  const bool unboxed = have && !boxed && !boxed_mid;
  if (__any_sync(0xffffffffu, unboxed)) {
    tile_block_nn1<TW>(gfine, unboxed, sel, d, id, d2c);
    tile_best_merge<TW>(d, id, d2c);
  }
  bool more = unboxed && !(d < gfine.cell * gfine.cell);
  if (unboxed && !more) region_c = gfine.cell;   // the 27 fine cells hold every point within one cell edge of the query
  if (__any_sync(0xffffffffu, more)) {
    tile_block_nn1<TW>(gmid, more, sel, d, id, d2c);
    tile_best_merge<TW>(d, id, d2c);
    const bool settled = more && d < gmid.cell * gmid.cell;
    more = more && !settled;
    if (settled) region_c = gmid.cell;
    // beyond the 27 middle cells: shells of the middle grid, pruned by min(best, gate)
    const float gate_r = a.reuse ? 5.0f + LVO_ODO_SLACK : 5.0f;   // with LVO_OPT_ODO_REUSE a little beyond the gate, so that "nothing inside" can be certified later
    const int R = (int)ceilf(gate_r * gmid.inv_cell);
    for (int r = 2; r <= R; ++r) {
      const float bound = (float)(r - 1) * gmid.cell;
      more = more && !(d < bound * bound);
      if (!__any_sync(0xffffffffu, more)) break;
      tile_shell_nn1<TW>(gmid, more, sel, r, gate_r * gate_r, d, id, d2c);
      tile_best_merge<TW>(d, id, d2c);
    }
    // pruned shells: only the ball of min(best distance, scanned gate) is certain
    if (unboxed && !settled && region_c == 0.f) region_c = sqrtf(fminf(d, gate_r * gate_r)) * 0.999f;
  }
  d2c = tile_min_f<TW>(d2c);
  const bool ok = have && id != INT_MAX && (double)d < 25.0;
  const int closest = ok ? id : 0;
  float4 pj = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ok) pj = C[closest];
  const int cid = ring_clamped(pj.w);
  // ---- adjacent-ring searches on the (ring, azimuth) grid
  const bool needA = !corner;
  Best bA{25.0f, INT_MAX, -1}, bB{25.0f, INT_MAX, -1};
  float d2A = FLT_MAX, d2B = FLT_MAX;   // per lane: best distance among the other eligible candidates it saw (guard radii)
  auto upd = [&](Best& b, float& d2, const Best& c) {
    if (c.j == b.j) return;   // the seed (or the best so far) met again
    if (c.d < b.d || (c.d == b.d && c.pos < b.pos)) { if (b.j >= 0) d2 = fminf(d2, b.d); b = c; }
    else d2 = fminf(d2, c.d);
  };
  const int bq = az_bucket(sel.x, sel.y);
  const float rho = sqrtf(sel.x * sel.x + sel.y * sel.y);
  auto consider = [&](float4 p, int r) {   // range r <-> ring cid - 2 + r
    const int idx = __float_as_int(p.w);
    const int dr = r - 2;
    if (idx == closest) return;
    // the walk is monotone in the ring id: above `closest` it only meets rings >= cid, below it rings <= cid
    if ((idx > closest && dr < 0) || (idx < closest && dr > 0)) return;
    const float dd = (p.x - sel.x) * (p.x - sel.x) + (p.y - sel.y) * (p.y - sel.y) + (p.z - sel.z) * (p.z - sel.z);
    if (!(dd < 25.0f)) { if (dr == 0) d2A = fminf(d2A, dd); else d2B = fminf(d2B, dd); return; }   // eligible, beyond the gate: only bounds the guard
    const int k2 = idx > closest ? (idx - closest) : ((closest - idx) + (1 << 30));
    const Best c{dd, k2, idx};
    if (dr == 0) upd(bA, d2A, c); else upd(bB, d2B, c);
  };
  const int ring = cid - 2 + tl;   // lanes 0..4 of the tile own rings cid-2 .. cid+2
  const bool ring_ok = ok && tl < 5 && ring >= 0 && ring < LVO_AZ_RINGS && (ring != cid || needA);
  // seeds from the previous outer iteration, if they still satisfy the ring filter relative to the new closest point
  auto seed = [&](int pidx, bool same_ring, Best& best) {
    if (!ok || pidx < 0 || pidx == closest) return;
    const float4 p = C[pidx];
    const int dr = ring_clamped(p.w) - cid;
    if (same_ring ? (dr != 0) : (dr == 0 || dr > 2 || dr < -2)) return;
    if ((pidx > closest && dr < 0) || (pidx < closest && dr > 0)) return;
    const float dd = (p.x - sel.x) * (p.x - sel.x) + (p.y - sel.y) * (p.y - sel.y) + (p.z - sel.z) * (p.z - sel.z);
    if (!(dd < 25.0f)) return;
    best = Best{dd, pidx > closest ? (pidx - closest) : ((closest - pidx) + (1 << 30)), pidx};
  };
  if (needA) seed(pA, true, bA);
  seed(pB, false, bB);
  // phase 1: +-2 buckets, or the window implied by the seed (part 1 only exists when the window wraps)
  // (bA, bB are the same in every lane of the tile here and after each merge, so every lane can evaluate both searches' windows;
  // with LVO_OPT_ODO_REUSE they reach LVO_ODO_SLACK beyond the best distances: room for the next iterations' certificates)
  auto halfw = [&](const Best& b) { return a.reuse ? az_halfwidth_slack(b.d, rho) : az_halfwidth(b.d, rho); };
  const int h1A = bA.j >= 0 ? halfw(bA) : 2, h1B = bB.j >= 0 ? halfw(bB) : 2;
  const int h1 = ring == cid ? h1A : h1B;
  for (int part = 0; part < 2; ++part) {
    unsigned b = 0, e = 0;
    if (ring_ok) az_bounds(gaz, ring, bq - h1, bq + h1, part, b, e);
    tile_scan_ranges<TW, 5>(gaz.pts, b, e, consider);
  }
  tile_best_merge<TW>(bA, d2A); tile_best_merge<TW>(bB, d2B);
  int hsA = h1A, hsB = h1B;   // half-widths scanned completely
  {  // phase 2: the rest of the window implied by the best distances so far (or by the 5 m gate)
    const int h2A = needA ? halfw(bA) : 0, h2B = halfw(bB);
    hsA = max(hsA, h2A); hsB = max(hsB, h2B);
    const int h = ring == cid ? h2A : h2B;
    const bool whole = 2 * h + 1 >= LVO_AZ_BUCKETS;
    const bool need2 = ring_ok && h > h1 && 2 * h1 + 1 < LVO_AZ_BUCKETS;
    if (__any_sync(0xffffffffu, need2)) {
      for (int sp = 0; sp < 4; ++sp) {   // side (bit 1), part (bit 0)
        unsigned b = 0, e = 0;
        if (need2) {
          if (whole) { if (sp == 0) az_bounds(gaz, ring, 0, LVO_AZ_BUCKETS - 1, 0, b, e); }
          else if ((sp >> 1) == 0) az_bounds(gaz, ring, bq - h, bq - h1 - 1, sp & 1, b, e);
          else az_bounds(gaz, ring, bq + h1 + 1, bq + h, sp & 1, b, e);
        }
        tile_scan_ranges<TW, 5>(gaz.pts, b, e, consider);
      }
      tile_best_merge<TW>(bA, d2A); tile_best_merge<TW>(bB, d2B);
    }
  }
  const int same = bA.j, other = bB.j;
  d2A = tile_min_f<TW>(d2A); d2B = tile_min_f<TW>(d2B);
  // ---- factor record (tile leader)
  bool made_c = false, made_p = false;
  if (have && tl == 0) {
    float4 guard = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.reuse) {
      // ok: the other points are at least min(second best, region) away.  Not ok: the nearest point itself lies beyond the gate (or there is none)
      if (ok) guard = make_float4(odo_guard_of(d2c, region_c), needA ? odo_guard_of(d2A, az_region(hsA, rho)) : 0.f, odo_guard_of(d2B, az_region(hsB, rho)), 1.f);
      else guard = make_float4(odo_guard_of(d, region_c), 0.f, 0.f, 1.f);
    }
    const int type = odo_emit(a, lane, f, ns, corner, ok, pt, C, closest, pj, same, other, sel, guard);
    made_c = corner && type >= 0; made_p = !corner && type >= 0;
  }
  const int nc = __popc(__ballot_sync(0xffffffffu, made_c)), np = __popc(__ballot_sync(0xffffffffu, made_p));
  if ((threadIdx.x & 31) == 0) {
    if (nc) atomicAdd(&s.stats.odo_corner_corr[a.outer], nc);
    if (np) atomicAdd(&s.stats.odo_plane_corr[a.outer], np);
  }
  }  // slot loop
}

// after the outer loop: few-correspondence warning (:566-568), pose integration (:581-582)
__global__ void k_odo_integrate(OdoArgs a, int outer_iters) {
  const int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= a.lanes || !lane_active(a.lane_flags, lane)) return;
  LaneState& s = a.ls[lane];
  if (s.odo_inited) {
    for (int o = 0; o < outer_iters; ++o)
      if (s.stats.odo_corner_corr[o] + s.stats.odo_plane_corr[o] < 10) s.odo_status = LVO_W_FEW_CORR;
    const d3 dt = quat_rotate(s.q_w, d3{s.para_t[0], s.para_t[1], s.para_t[2]});
    s.t_w[0] = s.t_w[0] + dt.x; s.t_w[1] = s.t_w[1] + dt.y; s.t_w[2] = s.t_w[2] + dt.z;
    double qn[4];
    quat_mul(s.q_w, s.para_q, qn);
    for (int k = 0; k < 4; ++k) s.q_w[k] = qn[k];
  }
  s.odo_inited = 1;
  s.n_corner_last = s.n_less_sharp;
  s.n_surf_last = s.n_less_flat;
  for (int r = 0; r < LVO_MAX_RINGS + 2; ++r) { s.corner_ring_first[r] = s.n_less_sharp; s.surf_ring_first[r] = s.n_less_flat; }
}
// distortion mode 2: the block :610-625 with its `if (0)` lifted — TransformToEnd (:176-191) of the less-sharp, less-flat and
// full-resolution clouds in place, on every frame (the first included: para = identity only strips the fractional intensity)
__global__ void k_odo_to_end(OdoArgs a) {
  const int lane = blockIdx.y;
  const LaneState& s = a.ls[lane];
  const int n0 = s.n_less_sharp, n1 = s.n_less_flat, n2 = s.n_kept;
  if (!lane_active(a.lane_flags, lane)) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1 + n2; i += gridDim.x * blockDim.x) {
    float4* p = i < n0 ? a.less_sharp + (size_t)lane * a.cap_lsharp + i
                       : (i < n0 + n1 ? a.less_flat + (size_t)lane * a.P + (i - n0) : a.full + (size_t)lane * a.P + (i - n0 - n1));
    *p = transform_to_end(s.para_q, s.para_t, *p);
  }
}
// copy less-sharp / less-flat into the "last" buffers (the pointer swap of :627-636) and build the ring-offset tables:
// ring_first[r] = first index whose ring id int(intensity) is >= r
__global__ void k_odo_swap(OdoArgs a) {
  const int lane = blockIdx.y;
  LaneState& s = a.ls[lane];
  const int nc = s.n_corner_last, nsf = s.n_surf_last;
  if (!lane_active(a.lane_flags, lane)) return;
  const int stride = gridDim.x * blockDim.x;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nc + nsf; i += stride) {
    const bool corner = i < nc;
    const int k = corner ? i : i - nc;
    const float4* src = corner ? a.less_sharp + (size_t)lane * a.cap_lsharp : a.less_flat + (size_t)lane * a.P;
    float4* dst = corner ? a.corner_last + (size_t)lane * a.cap_lsharp : a.surf_last + (size_t)lane * a.P;
    int* rf = corner ? s.corner_ring_first : s.surf_ring_first;
    const float4 p = src[k];
    dst[k] = p;
    const int r = min(max(int(p.w), 0), LVO_MAX_RINGS + 1);
    const int rp = k > 0 ? min(max(int(src[k - 1].w), 0), LVO_MAX_RINGS + 1) : -1;
    for (int x = rp + 1; x <= r; ++x) rf[x] = k;
  }
}

static inline void lvo_launch_odometry(cudaStream_t st, OdoArgs a, const SolveArgs& solve_proto, int outer_iters, int lanes, long long* launches, LvoStageTimer* tm = nullptr) {
  LVO_MARK(tm, LVO_ST_ODO_REST, st);
  k_odo_begin<<<lvo_div_up(lanes, 64), 64, 0, st>>>(a);
  if (launches) *launches += 1;
  const int nfeat_cap = a.cap_sharp + a.cap_flat;
  dim3 ga(max(1, lvo_div_up(nfeat_cap * 8, 256)), lanes);          // 8-lane tiles, every feature (outer iteration 0)
  dim3 gs(max(1, lvo_div_up(nfeat_cap * 32 / 8, 256)), lanes);     // full-warp tiles for the slow list (an eighth of the features per pass, grid-strided)
  dim3 gf(max(1, lvo_div_up(nfeat_cap, 128)), lanes);
  for (int o = 0; o < outer_iters; ++o) {
    a.outer = o;
    LVO_MARK(tm, LVO_ST_ODO_ASSOC, st);
    k_odo_assoc_fast<<<gf, 128, 0, st>>>(a);   // (slow_cnt is zero here: k_odo_begin before the loop, k_lm_solve after every iteration)
    if (launches) *launches += 1;
    if (o == 0) k_odo_assoc<8><<<ga, 256, 0, st>>>(a);   // first iteration: more features lack a nearby candidate
    else k_odo_assoc<32><<<gs, 256, 0, st>>>(a);
    SolveArgs sa = solve_proto;
    sa.lane_flags = a.lane_flags;
    sa.which = 0; sa.outer = o; sa.n_outer = outer_iters; sa.factors = a.factors; sa.factor_cap = a.factor_cap; sa.distort = a.distortion != 0; sa.reset_cnt = a.slow_cnt;
    LVO_MARK(tm, LVO_ST_ODO_SOLVER, st);
    lvo_launch_lm(st, sa, lanes, nfeat_cap);
    if (launches) *launches += 2;
  }
  LVO_MARK(tm, LVO_ST_ODO_REST, st);
  k_odo_integrate<<<lvo_div_up(lanes, 64), 64, 0, st>>>(a, outer_iters);
  if (a.distortion == 2) { k_odo_to_end<<<dim3(64, lanes), 256, 0, st>>>(a); if (launches) *launches += 1; }
  k_odo_swap<<<dim3(32, lanes), 256, 0, st>>>(a);
  if (launches) *launches += 2;
  // every lane's grids, an idle lane's included (rebuilt from its unchanged "last" clouds: the problem offsets are shared by all lanes)
  lvo_grid_build(st, a.grid, launches);
}
