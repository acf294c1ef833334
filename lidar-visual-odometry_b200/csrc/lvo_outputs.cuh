// lvo_outputs.cuh — the clouds the reference's mapping node publishes besides the pose, for any number of lanes in one call
// (lvo_map_cloud, lvo_map_cloud_batch*).
//
//   k_mapout_offsets     per slot: exclusive prefix of the corner + surf counts of its cubes, in the order of
//                        /laser_cloud_surround (the valid list, laserMapping.cpp:806-815) or /laser_cloud_map (all 4851 cubes, :823-836)
//   k_mapout_copy        per slot: each cube's corner points, then its surf points, to dst + offset
//   k_mapout_registered  per lane: the registered cloud of the last step (/velodyne_cloud_registered, :838-842) to dst
//
// A slot is a lane (slot s = lane first_lane + s).  The launch count is fixed: the grids are (x, slots).
#pragma once
#include "lvo_internal.h"
#include "lvo_mapping.cuh"

// One per slot, uploaded from pinned staging before the copy kernels.  dst == NULL: the slot is not copied.
struct MapOutDesc {
  float4* dst;
  unsigned n;          // k_mapout_registered: points to copy (host-recorded at the end of the step)
  unsigned pad;
};
static_assert(sizeof(MapOutDesc) == 16, "MapOutDesc layout");

#define LVO_MAPOUT_STRIDE (LVO_NCUBES + 1)   // offset-table entries per slot

struct MapOutArgs {
  const LaneState* ls;
  const unsigned* cube_start[2];   // [type] -> [lanes][LVO_NCUBES + 1] of the current generation
  const float4* map_pts[2];        // [type] -> [lanes][map_cap[type]] of the current generation
  int map_cap[2];
  int first_lane;
  int surround;                    // 1: the last frame's valid cubes, 0: all cubes
};

__device__ __forceinline__ int mapout_ncubes(const MapOutArgs& a, const LaneState& s) { return a.surround ? s.n_valid : LVO_NCUBES; }

// grid (slots), 256 threads.  off[s][k] = points of the slot's cubes before its k-th cube; tot[s] = all of them.
__global__ void __launch_bounds__(256) k_mapout_offsets(MapOutArgs a, unsigned* off, unsigned* tot) {
  __shared__ unsigned sm[33];
  const int slot = blockIdx.x, lane = a.first_lane + slot;
  const LaneState& s = a.ls[lane];
  const int n = mapout_ncubes(a, s);
  const unsigned* cs0 = a.cube_start[0] + (size_t)lane * (LVO_NCUBES + 1);
  const unsigned* cs1 = a.cube_start[1] + (size_t)lane * (LVO_NCUBES + 1);
  unsigned* o = off + (size_t)slot * LVO_MAPOUT_STRIDE;
  unsigned carry = 0;
  for (int base = 0; base < n; base += blockDim.x) {
    const int k = base + threadIdx.x;
    unsigned cnt = 0;
    if (k < n) { const int c = a.surround ? s.valid_cube[k] : k; cnt = (cs0[c + 1] - cs0[c]) + (cs1[c + 1] - cs1[c]); }
    unsigned t;
    const unsigned ex = block_excl_scan(cnt, sm, &t);
    if (k < n) o[k] = carry + ex;
    carry += t;
  }
  if (threadIdx.x == 0) tot[slot] = carry;
}

// grid (x, slots), 256 threads: CTA x walks cubes x, x + gridDim.x, ... of its slot
__global__ void __launch_bounds__(256) k_mapout_copy(MapOutArgs a, const MapOutDesc* desc, const unsigned* off) {
  const int slot = blockIdx.y, lane = a.first_lane + slot;
  float4* dst = desc[slot].dst;
  if (!dst) return;
  const LaneState& s = a.ls[lane];
  const int n = mapout_ncubes(a, s);
  const unsigned* cs0 = a.cube_start[0] + (size_t)lane * (LVO_NCUBES + 1);
  const unsigned* cs1 = a.cube_start[1] + (size_t)lane * (LVO_NCUBES + 1);
  const float4* M0 = a.map_pts[0] + (size_t)lane * a.map_cap[0];
  const float4* M1 = a.map_pts[1] + (size_t)lane * a.map_cap[1];
  const unsigned* o = off + (size_t)slot * LVO_MAPOUT_STRIDE;
  for (int k = blockIdx.x; k < n; k += gridDim.x) {
    const int c = a.surround ? s.valid_cube[k] : k;
    const unsigned b0 = cs0[c], n0 = cs0[c + 1] - b0, b1 = cs1[c], n1 = cs1[c + 1] - b1;
    float4* d = dst + o[k];
    for (unsigned i = threadIdx.x; i < n0 + n1; i += blockDim.x) d[i] = i < n0 ? __ldg(M0 + b0 + i) : __ldg(M1 + b1 + (i - n0));
  }
}

// grid (x, lanes), 256 threads: registered[lane][0 .. n) -> dst
__global__ void __launch_bounds__(256) k_mapout_registered(const float4* registered, int P, const MapOutDesc* desc) {
  const int lane = blockIdx.y;
  const MapOutDesc d = desc[lane];
  if (!d.dst) return;
  const float4* src = registered + (size_t)lane * P;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < d.n; i += gridDim.x * blockDim.x) d.dst[i] = __ldg(src + i);
}
