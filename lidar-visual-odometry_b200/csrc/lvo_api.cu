// lvo_api.cu — the C ABI of liblvo.so (include/lvo.h): context, device arenas, and the host-side enqueue logic.
// Single translation unit: the kernels live in the .cuh files included below.  Compiled with
//   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo
// (-fmad=false: the reference's x86 build has no FMA contraction, SURVEY §7 hard part 1).
#include "lvo_internal.h"
#include "lvo_prims.cuh"
#include "lvo_extract.cuh"
#include "lvo_voxel.cuh"
#include "lvo_knn.cuh"
#include "lvo_solver.cuh"
#include "lvo_odometry.cuh"
#include "lvo_mapping.cuh"
#include "lvo_depth.cuh"
#include "lvo_outputs.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <nvtx3/nvToolsExt.h>   // header-only; ranges under the reference's stage names show up in Nsight timelines

// lvo_lane_load: lvo_probe_fetch of the lane returns LVO_E_STATE for a probe until the stage that writes it has run for the lane
#define LVO_PROBE_GATE_EXTRACT 1  // LVO_P_FULL .. LVO_P_LESS_FLAT: its next active frame, or lvo_extract_features
#define LVO_PROBE_GATE_ODO 2      // LVO_P_ODO_*: its next active frame, or lvo_scan_to_scan
#define LVO_PROBE_GATE_MAP 4      // LVO_P_MAP_*, LVO_P_REGISTERED: its next mapping frame, or lvo_scan_to_map

// Owner of device and pinned allocations that are freed together: the context's buffers, and each arena of the stand-alone calls.
// A failed allocation puts the CUDA error text into the context's lvo_last_error; nothing is zero-filled here.
struct LvoArena {
  std::vector<void*> dev, pin;
  template <class T> int device(lvo_ctx* c, T** p, size_t bytes) { return get(c, (void**)p, bytes, false); }
  template <class T> int pinned(lvo_ctx* c, T** p, size_t bytes) { return get(c, (void**)p, bytes, true); }
  int get(lvo_ctx* c, void** p, size_t bytes, bool host) {
    bytes = std::max<size_t>(bytes, 16);
    const cudaError_t e = host ? cudaMallocHost(p, bytes) : cudaMalloc(p, bytes);
    if (e != cudaSuccess) { *p = nullptr; lvo_set_error(c, std::string(host ? "cudaMallocHost: " : "cudaMalloc: ") + cudaGetErrorString(e)); return LVO_E_CUDA; }
    (host ? pin : dev).push_back(*p);
    return LVO_OK;
  }
  void release() {
    for (void* p : dev) cudaFree(p);
    for (void* p : pin) cudaFreeHost(p);
    dev.clear(); pin.clear();
  }
};

struct lvo_ctx {
  lvo_config cfg;
  int lanes, P, cap_sharp, cap_lsharp, cap_flat;
  cudaStream_t st = nullptr;
  cudaStream_t own_st = nullptr;
  mutable std::string err;    // lvo_last_error; the const getters set it too (lvo_enter)
  LvoArena mem;               // every buffer allocated by lvo_create (dalloc / halloc) and after it for the context's lifetime
  LaneState* d_ls = nullptr;
  LaneState* h_ls = nullptr;  // pinned mirror
  ExtractArgs ex;
  OdoArgs odo;
  MapArgs map;
  SolveArgs solve;
  GridSet gknn;               // 1-problem grid for the stand-alone lvo_knn operator (shares storage with map.grid)
  GridProblem* d_knn_prob = nullptr;
  int* d_knn_n = nullptr;
  unsigned char* d_raw = nullptr;   // [lanes][P * 32] raw sweep records
  const lvo_cloud_view* pending_next = nullptr;  // lvo_step_batch_pipelined: frame to prefetch once this frame is enqueued
  unsigned char* d_raw2 = nullptr;  // second staging buffer for lvo_step_batch_pipelined (allocated on first use)
  cudaStream_t copy_st = nullptr;
  cudaEvent_t copy_ev = nullptr, compute_ev = nullptr;
  std::vector<lvo_cloud_view> prefetched;  // the sweep set sitting in the "next" staging buffer
  std::vector<const unsigned char*> next_in_ptr;  // its per-lane device pointers
  int opt_stage_timing = 1;         // LVO_OPT_STAGE_TIMING: sub-stage events in plain-launch steps
  int raw_cur = 0;                  // which staging buffer the current frame reads
  size_t raw_lane_bytes = 0;
  const unsigned char** d_in_ptr = nullptr; const unsigned char** h_in_ptr = nullptr;
  int* d_in_n = nullptr; int* h_in_n = nullptr;   // [2 * lanes]: sweep counts, then the LVO_LANE_* flags of the step (one upload)
  float4* d_upload = nullptr;       // scratch for strided uploads (P * 32 bytes)
  int* d_knn_ind = nullptr; float* d_knn_sq = nullptr;
  double* d_trace[2] = {nullptr, nullptr};
  long long launches = 0;
  std::vector<long long> lane_frame;  // frames a lane has processed since its creation / lvo_lane_reset (its skip_frame phase)
  // lvo_lane_configure: each lane's sensor settings (lvo_create gives every lane the context's); the kernels read d_lcfg, uploaded
  // from its pinned mirror h_lcfg; skip_frame stays on the host
  std::vector<lvo_lane_config> lane_cfg;
  LaneConfig* d_lcfg = nullptr; LaneConfig* h_lcfg = nullptr;
  std::vector<char> lane_active;      // lvo_set_lane_active
  std::vector<char> lane_map_update;  // lvo_set_lane_map_update (host state like activity: not in LaneState or a snapshot)
  std::vector<char> prefetched_active;  // the active set the prefetched sweeps were staged for
  std::vector<int> lane_status;
  // lvo_lane_load: a loaded lane's probe arrays belong to this context's earlier frames, its counts to the snapshot; LVO_PROBE_GATE_*
  // bits stay set until the stage that writes the probe has run for the lane
  std::vector<char> probe_gate;
  bool odo_grids_stale = false;     // lvo_lane_load: the odometry grids no longer match the "last" clouds (rebuilt by the next reader)
  cudaEvent_t ev[8];
  LvoStageTimer stage_tm;           // sub-stage CUDA events of plain-launch calls (reference TicToc names)
  lvo_timings tim;
  // lvo_step_batch*_async: what lvo_wait has to finish
  bool pending = false, pending_do_map = false, pending_graph = false;
  // merged host->device uploads (one copy per run of lanes that are adjacent in host memory)
  struct Span { const unsigned char* host; size_t bytes; size_t dev_off; };
  std::vector<Span> spans;
  std::vector<int> span_order;
  // CUDA graphs of the fused per-frame sequence: [mapping on/off][map generation]
  cudaGraphExec_t graph_exec[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  long long graph_launches[2][2] = {{0, 0}, {0, 0}};
  int graph_stride = -1, graph_off = -1;
  int opt_graphs = -1;
  // lvo_depth_associate*: the calls' own arena (DESIGN §3), allocated on the first call and grown, never shrunk, when a call
  // brings more points, keypoints or lanes; the step's buffers are not touched.  The single call is one slot of it.
  struct DepthArena {
    size_t cap_pts = 0, cap_raw = 0, cap_kp = 0; int cap_slots = 0;
    LvoArena mem;                      // all of the buffers below; growing releases and reallocates them
    unsigned char* raw = nullptr;      // [cap_raw] host-form sweep records, back to back in slot order
    unsigned* flag = nullptr;          // [cap_pts]
    float4* dc = nullptr;              // [cap_pts] depth clouds
    unsigned char* d_in = nullptr;     // slots, then the host form's keypoints (one upload)
    unsigned char* h_in = nullptr;     // its pinned staging
    unsigned* d_res = nullptr;         // host form: depth [K], valid [K], nn [3 K] (one download)
    unsigned* h_res = nullptr;
    unsigned* dc_off = nullptr; int* ndc = nullptr;   // [cap_slots]
    int* cnt = nullptr;                // scan length, depth-cloud total
    GridSet grid;                      // one problem per slot, LVO_DEPTH_CELLS cells each
  } depth;
  // lvo_map_cloud / lvo_map_cloud_batch*: the calls' own arena (DESIGN §3), allocated on the first call; the point buffer grows, never
  // shrinks, when a call brings more points; the step's buffers are not touched
  struct MapOutArena {
    LvoArena mem;                      // the per-slot part, sized for every lane of the context
    MapOutDesc* d_desc = nullptr; MapOutDesc* h_desc = nullptr;   // [lanes] copy descriptors and their pinned staging
    unsigned* off = nullptr;           // [lanes][LVO_NCUBES + 1] cube offsets of each slot's cloud
    unsigned* d_tot = nullptr; unsigned* h_tot = nullptr;         // [lanes] points of each slot's cloud
    size_t cap_pts = 0;
    LvoArena pts_mem;                  // the point buffer alone: growing releases and reallocates it
    float4* d_pts = nullptr;           // [cap_pts] host form: the selected lanes' clouds back to back
  } mapout;
  // lvo_map_cloud_batch* LVO_MAP_REGISTERED: points of each lane's registered cloud in the last lvo_step_batch* call (n_kept of that
  // frame for a lane that mapped, 0 otherwise), recorded by step_finish; reg_valid is false once lvo_scan_to_map or lvo_knn has
  // overwritten map.registered, until the next step completes
  std::vector<size_t> reg_n;
  bool reg_valid = true;
  // pose uncertainty (LVO_P_*_UNCERTAINTY): raw records [lanes][2] written by k_lm_solve; the derived records of every lane come to a
  // pinned mirror on the first fetch after unc_epoch moved (every call that can change a raw record bumps it); unc_frame is each
  // record's frame field, kept on the host (lane_frame of the step that wrote it, -1 otherwise)
  LvoUncRaw* d_unc = nullptr;
  lvo_pose_uncertainty* d_unc_out = nullptr; lvo_pose_uncertainty* h_unc = nullptr;
  std::vector<int64_t> unc_frame;
  long long unc_epoch = 0, unc_mirror_epoch = -1;
};

void lvo_set_error(lvo_ctx* ctx, const std::string& msg) { if (ctx) ctx->err = msg; }

namespace {

#define LVO_TRY(x) do { int _r = (x); if (_r != LVO_OK) return _r; } while (0)

// n elements of the context's own buffers (c->mem)
template <class T>
int dalloc(lvo_ctx* c, T** p, size_t n, bool zero = true) {
  const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
  LVO_TRY(c->mem.device(c, p, bytes));
  // stream-ordered with the kernels that follow (the context's stream is non-blocking: the legacy stream would not order with it)
  if (zero) LVO_CUDA_OK(c, cudaMemsetAsync(*p, 0, bytes, c->st));
  return LVO_OK;
}
template <class T>
int halloc(lvo_ctx* c, T** p, size_t n) {
  const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
  LVO_TRY(c->mem.pinned(c, p, bytes));
  memset(*p, 0, bytes);
  return LVO_OK;
}

int alloc_scan(lvo_ctx* c, LvoScanScratch* s, size_t n_cap) {
  s->cap_tiles = lvo_div_up((long long)n_cap, LVO_SCAN_TILE) + 2;
  return dalloc(c, &s->partial, (size_t)s->cap_tiles);
}
// table_cells: cells of the whole set (0 = nprob * cells_cap; smaller when the problems carry their own GridProblem::cells_cap shares)
int alloc_grid(lvo_ctx* c, GridSet* g, int nprob, int cells_cap, size_t pts_total, int pts_per_problem, size_t table_cells = 0) {
  g->nprob = nprob; g->cells_cap_per_problem = cells_cap; g->pts_cap_per_problem = pts_per_problem;
  if (table_cells == 0) table_cells = (size_t)nprob * cells_cap;
  g->table_cap_total = (long long)table_cells;
  LVO_TRY(dalloc(c, &g->prob, (size_t)nprob));
  LVO_TRY(dalloc(c, &g->table, table_cells + 1));
  LVO_TRY(dalloc(c, &g->d_table_len, 1));
  LVO_TRY(dalloc(c, &g->rank, pts_total));
  LVO_TRY(dalloc(c, &g->pt_off, (size_t)nprob + 1));
  LVO_TRY(dalloc(c, &g->sorted_pts, pts_total));
  LVO_TRY(dalloc(c, &g->sorted_id, pts_total));
  LVO_TRY(alloc_scan(c, &g->scan, table_cells + 1));
  return LVO_OK;
}

__global__ void k_unpack(const unsigned char* raw, int n, int stride, int off_xyz, int off_i, float4* out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float* p = reinterpret_cast<const float*>(raw + (size_t)i * stride + off_xyz);
    const float w = *reinterpret_cast<const float*>(raw + (size_t)i * stride + off_i);
    out[i] = make_float4(p[0], p[1], p[2], w);
  }
}
struct SetCounts { int what; int v[4]; double pose[7]; };
__global__ void k_set_lane(LaneState* ls, int lane, SetCounts sc) {
  LaneState& s = ls[lane];
  if (sc.what == 0) { s.n_sharp = sc.v[0]; s.n_less_sharp = sc.v[1]; s.n_flat = sc.v[2]; s.n_less_flat = sc.v[3]; }
  else if (sc.what == 1) { s.n_less_sharp = sc.v[0]; s.n_less_flat = sc.v[1]; s.n_kept = sc.v[2]; for (int k = 0; k < 4; ++k) s.q_wodom[k] = sc.pose[k]; for (int k = 0; k < 3; ++k) s.t_wodom[k] = sc.pose[4 + k]; }
  else if (sc.what == 2) { for (int k = 0; k < 4; ++k) s.q_wmap_wodom[k] = sc.pose[k]; for (int k = 0; k < 3; ++k) s.t_wmap_wodom[k] = sc.pose[4 + k]; }
  else if (sc.what == 3) { for (int k = 0; k < 4; ++k) s.para_q[k] = sc.pose[k]; for (int k = 0; k < 3; ++k) s.para_t[k] = sc.pose[4 + k]; }
  else if (sc.what == 4) { for (int k = 0; k < 4; ++k) s.q_w[k] = sc.pose[k]; for (int k = 0; k < 3; ++k) s.t_w[k] = sc.pose[4 + k]; }
  else if (sc.what == 5) { s.n_map[0] = sc.v[0]; s.n_map[1] = sc.v[1]; }
}
// lanes [first, first + n) of a zero-filled state array: the state of a freshly created context (lvo_create, lvo_lane_reset)
__global__ void k_init_lanes(LaneState* ls, int first, int n) {
  const int l = first + blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= first + n) return;
  LaneState& s = ls[l];
  s.para_q[3] = 1.0; s.q_w[3] = 1.0; s.map_x[3] = 1.0; s.q_wmap_wodom[3] = 1.0; s.q_wodom[3] = 1.0;
  s.cen[0] = 10; s.cen[1] = 10; s.cen[2] = 5;  // laserMapping.cpp:74-76
}
// which == 0: odometry, 8 problems per lane (corner / surf fine xyz, ring-azimuth, middle xyz, coarse xyz);
// which == 1: mapping, 2 problems per lane (corner / surf FromMap)
__global__ void k_setup_grid_problems(GridProblem* prob, int nprob, const float4* base0, size_t stride0, const float4* base1, size_t stride1,
                                      LaneState* ls, int which, float cell) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nprob) return;
  const int per = which == 0 ? LVO_ODO_GRIDS : 2;
  const int lane = p / per, t = p & 1;
  prob[p].pts = (t ? base1 + (size_t)lane * stride1 : base0 + (size_t)lane * stride0);
  if (which == 0) prob[p].d_n = t ? &ls[lane].n_surf_last : &ls[lane].n_corner_last;
  else prob[p].d_n = &ls[lane].from_off[t][LVO_MAX_VALID];
  const int k = p % per;
  // odometry: fine grid 0.5 x 0.5 x 2 m for the surf cloud (dense in x-y, sparse in z), 1 x 1 x 2 m for the corner cloud,
  // middle grids 2 m (their shells cover the 5 m gate; the former 8 m coarse grids were built every frame and never searched)
  prob[p].want_cell = which == 0 ? (k >= 4 ? 2.0f : (k == 1 ? 0.5f : 1.0f)) : cell;
  prob[p].want_cell_z = which == 0 ? 2.0f : 0.f;
  prob[p].mode = (which == 0 && (k == 2 || k == 3)) ? 1 : 0;
  // share of the cell table (lvo_odo_cells_cap): the fine grids get 4 M cells, the (ring, azimuth) grids their fixed size, the 2 m
  // and 8 m grids 1/8 and 1/64 of the fine share; a grid that does not fit doubles its cell edge (k_grid_setup)
  prob[p].cells_cap = which == 0 ? (k < 2 ? (1 << 22) : (k < 4 ? LVO_AZ_BUCKETS * LVO_AZ_RINGS : (1 << 19))) : 0;
  prob[p].clamp_xy = 0.f;
  prob[p].bbox_from = (which == 0 && k >= 4) ? p - k + (k & 1) : -1;   // middle / coarse grids reuse the fine grid's box
}
__global__ void k_setup_one_problem(GridProblem* prob, const float4* pts, const int* d_n, float cell) {
  prob[0].pts = pts; prob[0].d_n = d_n; prob[0].want_cell = cell; prob[0].want_cell_z = 0.f; prob[0].mode = 0; prob[0].cells_cap = 0; prob[0].clamp_xy = 0.f; prob[0].bbox_from = -1;
}
__global__ void k_vx_single_setup(VoxelEngine e, int n, float leaf) {
  if (blockIdx.x == 0 && threadIdx.x == 0) { *e.d_n = n; *e.d_nsegs = 1; e.seg_leaf[0] = leaf; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { e.in_seg[i] = 0; e.in_aux[i] = 0; }
}

// lvo_transform_cloud: TransformToStart / TransformToEnd of a packed cloud under (q, t) = pose or the lane's para_q / para_t
struct PoseArg { double q[4], t[3]; int use; };
__global__ void k_transform_cloud(const LaneState* ls, PoseArg pa, const float4* in, int n, int distortion, int to_end, float4* out) {
  const double* q = pa.use ? pa.q : ls[0].para_q;
  const double* t = pa.use ? pa.t : ls[0].para_t;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = to_end ? transform_to_end(q, t, in[i]) : transform_to_start(q, t, in[i], distortion);
}
// xyz_only: the cloud is a raw sweep, whose intensity the path never reads (scanRegistration.cpp:132-133 converts to pcl::PointXYZ):
// records of 12 bytes (packed x, y, z) are accepted and off_intensity is ignored.
int check_view(lvo_ctx* c, const lvo_cloud_view& v, size_t cap, bool xyz_only = false) {
  if (v.n == 0) return LVO_OK;
  const bool bad_i = !xyz_only && ((v.off_intensity & 3) || v.off_intensity + 4 > v.stride);
  if (!v.data || v.stride < (xyz_only ? 12u : 16u) || v.stride > 64 || (v.stride & 3) || (v.off_xyz & 3) || v.off_xyz + 12 > v.stride || bad_i) {
    lvo_set_error(c, "bad cloud view"); return LVO_E_BADARG;
  }
  if (v.n > cap) { lvo_set_error(c, "input cloud exceeds context capacity"); return LVO_E_CAPACITY; }
  return LVO_OK;
}
// strided host cloud -> packed float4 on device
int upload_cloud(lvo_ctx* c, const lvo_cloud_view& v, float4* dst) {
  if (v.n == 0) return LVO_OK;
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_upload, v.data, v.n * v.stride, cudaMemcpyHostToDevice, c->st));
  k_unpack<<<std::max(1, std::min(lvo_div_up((long long)v.n, 256), 592)), 256, 0, c->st>>>((const unsigned char*)c->d_upload, (int)v.n, (int)v.stride,
                                                                                             (int)v.off_xyz, (int)v.off_intensity, dst);
  c->launches++;
  return LVO_OK;
}
int download_cloud(lvo_ctx* c, const float4* src, size_t n, lvo_cloud_out* out) {
  if (!out) return LVO_OK;
  out->n = n;
  if (n > out->cap || (n && !out->data)) { lvo_set_error(c, "output cloud buffer too small"); return LVO_E_CAPACITY; }
  if (n) LVO_CUDA_OK(c, cudaMemcpyAsync(out->data, src, n * sizeof(float4), cudaMemcpyDeviceToHost, c->st));
  return LVO_OK;
}
int sync_state(lvo_ctx* c) {
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->h_ls, c->d_ls, sizeof(LaneState) * c->lanes, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}
// The odometry grids of frame k + 1 are built at the end of frame k for all lanes at once (the problems share one table).  After
// lvo_lane_load the loaded lane's grids are stale; the next call that searches them rebuilds every lane's grids once, however many
// lanes were loaded.  The other lanes' grids come out the same: they are built from the same clouds.
void rebuild_stale_grids(lvo_ctx* c) {
  if (!c->odo_grids_stale) return;
  lvo_grid_build(c->st, c->odo.grid, &c->launches);
  c->odo_grids_stale = false;
}
void pose_out(lvo_pose* p, const double* q, const double* t) {
  if (!p) return;
  for (int k = 0; k < 4; ++k) p->q[k] = q[k];
  for (int k = 0; k < 3; ++k) p->t[k] = t[k];
}
int* lane_flags(lvo_ctx* c) { return c->h_in_n + c->lanes; }
// capacities of the feature clouds of one sweep, which follow from n_scans (6 sectors per ring, at most 2 sharp, 20 less-sharp and 4
// flat points per sector: scanRegistration.cpp:293-370).  lvo_create sizes every lane's buffers for the context's n_scans, the largest
// a lane may take; a lane's own n_scans bounds what it can hold.
struct FeatureCaps { int sharp, lsharp, flat; };
FeatureCaps feature_caps(int n_scans) { return FeatureCaps{n_scans * LVO_SECTORS * 2, n_scans * LVO_SECTORS * 20, n_scans * LVO_SECTORS * 4}; }
// lane_cfg[lane] -> the device record of the lane, stream-ordered (the kernels of steps enqueued before it read the old one)
int upload_lane_config(lvo_ctx* c, int lane) {
  const lvo_lane_config& lc = c->lane_cfg[lane];
  c->h_lcfg[lane] = LaneConfig{lc.n_scans, (float)lc.minimum_range, {(float)lc.line_res, (float)lc.plane_res}};
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_lcfg + lane, c->h_lcfg + lane, sizeof(LaneConfig), cudaMemcpyHostToDevice, c->st));
  return LVO_OK;
}
// the stand-alone stage calls run their stage for every lane: its probes are this context's own again
void stage_ran_on_all_lanes(lvo_ctx* c, int gate) { for (char& g : c->probe_gate) g &= ~gate; }
// lvo_scan_to_scan (stage 0) / lvo_scan_to_map (stage 1) rewrite that stage's pose-uncertainty record of every lane; they keep no frame
// count, so the records' frame is -1
void uncertainty_written(lvo_ctx* c, int stage) {
  for (int l = 0; l < c->lanes; ++l) c->unc_frame[2 * l + stage] = -1;
  c->unc_epoch++;
}
// sweep pointers, counts and lane flags of the step
int set_inputs(lvo_ctx* c) {
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_in_ptr, c->h_in_ptr, sizeof(void*) * c->lanes, cudaMemcpyHostToDevice, c->st));
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_in_n, c->h_in_n, sizeof(int) * 2 * c->lanes, cudaMemcpyHostToDevice, c->st));
  return LVO_OK;
}
// lvo_extract_features / lvo_scan_to_scan / lvo_scan_to_map enqueue the batched kernels for every lane: all lanes active and mapping,
// whatever the last batched step left in the flags, each with its own map-update setting.  upload = false: set_inputs follows.
int flags_all_lanes(lvo_ctx* c, bool upload) {
  for (int l = 0; l < c->lanes; ++l) lane_flags(c)[l] = LVO_LANE_ACTIVE | LVO_LANE_MAPS | (c->lane_map_update[l] ? 0 : LVO_LANE_MAP_FIXED);
  if (upload) LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_in_n + c->lanes, lane_flags(c), sizeof(int) * c->lanes, cudaMemcpyHostToDevice, c->st));
  return LVO_OK;
}
void enqueue_extract(lvo_ctx* c, int stride, int off_xyz, int max_n, LvoStageTimer* tm) {
  ExtractArgs a = c->ex;
  a.in_stride = stride; a.in_off_xyz = off_xyz;
  nvtxRangePushA("scan registration");
  lvo_launch_extract(c->st, a, c->lanes, max_n, &c->launches, tm);
  nvtxRangePop();
}
void enqueue_odometry(lvo_ctx* c, LvoStageTimer* tm) {
  nvtxRangePushA("laserOdometry");
  lvo_launch_odometry(c->st, c->odo, c->solve, c->cfg.outer_iters, c->lanes, &c->launches, tm);
  nvtxRangePop();
}
void enqueue_mapping(lvo_ctx* c, int from_odo, bool want_registered, LvoStageTimer* tm) {
  MapArgs a = c->map;
  a.from_odo = from_odo;
  nvtxRangePushA("laserMapping");
  lvo_launch_mapping(c->st, a, c->solve, c->cfg.outer_iters, c->lanes, want_registered, &c->launches, tm);
  nvtxRangePop();
  c->map.gen ^= 1;
}
// plain-launch calls: begin / end of the sub-stage event list
LvoStageTimer* stage_timer_begin(lvo_ctx* c, bool on) {
  c->stage_tm.reset();
  c->stage_tm.on = on;
  return on ? &c->stage_tm : nullptr;
}
// after the stream has been synchronised: sub-stage sums into lvo_timings (stages that did not run keep 0)
void collect_stage_timing(lvo_ctx* c, bool mapped) {
  float ms[LVO_ST_COUNT]; int cnt[LVO_ST_COUNT];
  c->stage_tm.collect(ms, cnt);
  lvo_timings& t = c->tim;
  t.reg_prepare_ms = ms[LVO_ST_REG_PREPARE]; t.reg_sort_ms = ms[LVO_ST_REG_SORT]; t.reg_separate_ms = ms[LVO_ST_REG_SEPARATE];
  t.odo_association_ms = ms[LVO_ST_ODO_ASSOC]; t.odo_solver_ms = ms[LVO_ST_ODO_SOLVER]; t.odo_rest_ms = ms[LVO_ST_ODO_REST];
  t.map_prepare_ms = ms[LVO_ST_MAP_PREPARE]; t.map_build_tree_ms = ms[LVO_ST_MAP_TREE];
  t.map_association_ms = ms[LVO_ST_MAP_KNN] + ms[LVO_ST_MAP_FIT]; t.map_solver_ms = ms[LVO_ST_MAP_SOLVER];
  t.map_optimization_ms = ms[LVO_ST_MAP_KNN] + ms[LVO_ST_MAP_FIT] + ms[LVO_ST_MAP_SOLVER];
  t.map_add_points_ms = ms[LVO_ST_MAP_ADD]; t.map_filter_ms = ms[LVO_ST_MAP_FILTER]; t.map_pub_ms = ms[LVO_ST_MAP_PUB];
  t.knn_ms = ms[LVO_ST_MAP_KNN]; t.knn_launches = cnt[LVO_ST_MAP_KNN]; t.knn_bytes = 0;
  if (!mapped || !c->stage_tm.on) return;
  for (int l = 0; l < c->lanes; ++l) {
    const LaneState& s = c->h_ls[l];
    if (s.map_too_small || !(lane_flags(c)[l] & LVO_LANE_MAPS)) continue;
    const double M = (double)s.from_off[0][LVO_MAX_VALID] + (double)s.from_off[1][LVO_MAX_VALID];
    const double Q = (double)s.n_stack[0] + (double)s.n_stack[1];
    t.knn_bytes += s.stats.map_outer_executed * (16.0 * M + 56.0 * Q);   // iterations skipped at a fixed point search nothing
  }
}
// Host sweeps -> device staging buffer `buf` on stream `st`: lanes whose records are adjacent in host memory (one pinned slab per
// sequence or per context, the usual producer layout) go up in ONE cudaMemcpyAsync per run instead of one per lane; a gap of up to
// 64 KB between neighbours is copied along.  Sets h_in_ptr / h_in_n; idle lanes get no upload and a count of 0 (their views are not
// read).  The staging buffer holds lanes * P * 32 bytes.
int stage_sweeps(lvo_ctx* c, const lvo_cloud_view* sweeps, unsigned char* buf, cudaStream_t st) {
  const int L = c->lanes;
  c->span_order.clear();
  for (int l = 0; l < L; ++l) {
    if (c->lane_active[l]) c->span_order.push_back(l);
    else { c->h_in_n[l] = 0; c->h_in_ptr[l] = buf; }
  }
  std::sort(c->span_order.begin(), c->span_order.end(), [&](int a, int b) { return (uintptr_t)sweeps[a].data < (uintptr_t)sweeps[b].data; });
  c->spans.clear();
  const size_t cap = c->raw_lane_bytes * (size_t)L, max_gap = 64u << 10;
  size_t dev_off = 0;
  for (size_t k = 0; k < c->span_order.size(); ++k) {
    const int l = c->span_order[k];
    const lvo_cloud_view& v = sweeps[l];
    c->h_in_n[l] = (int)v.n;
    if (v.n == 0) { c->h_in_ptr[l] = buf; continue; }
    const unsigned char* h = (const unsigned char*)v.data;
    const size_t bytes = v.n * v.stride;
    bool merged = false;
    if (!c->spans.empty()) {
      lvo_ctx::Span& sp = c->spans.back();
      const unsigned char* end = sp.host + sp.bytes;
      if (h >= end && (size_t)(h - end) <= max_gap && sp.dev_off + (size_t)(h - sp.host) + bytes <= cap) {
        sp.bytes = (size_t)(h - sp.host) + bytes;
        c->h_in_ptr[l] = buf + sp.dev_off + (size_t)(h - sp.host);
        dev_off = sp.dev_off + ((sp.bytes + 255) & ~(size_t)255);
        merged = true;
      }
    }
    if (!merged) {
      if (dev_off + bytes > cap) { lvo_set_error(c, "sweeps exceed the staging buffer"); return LVO_E_CAPACITY; }
      c->spans.push_back(lvo_ctx::Span{h, bytes, dev_off});
      c->h_in_ptr[l] = buf + dev_off;
      dev_off += (bytes + 255) & ~(size_t)255;
    }
  }
  for (const lvo_ctx::Span& sp : c->spans) LVO_CUDA_OK(c, cudaMemcpyAsync(buf + sp.dev_off, sp.host, sp.bytes, cudaMemcpyHostToDevice, st));
  return LVO_OK;
}


// Every entry point makes the context's device current for its duration (a process may hold contexts on several GPUs and call them
// from any thread: kernels launched on a context's stream while another device is current fail with "invalid resource handle")
// and restores the caller's device on return.
struct LvoDeviceGuard {
  int prev = -1; bool switched = false;
  explicit LvoDeviceGuard(const lvo_ctx* c);
  ~LvoDeviceGuard() { if (switched) cudaSetDevice(prev); }
};
}  // namespace

LvoDeviceGuard::LvoDeviceGuard(const lvo_ctx* c) {
  if (!c) return;
  if (cudaGetDevice(&prev) == cudaSuccess && prev != c->cfg.device) switched = cudaSetDevice(c->cfg.device) == cudaSuccess;
}

// The checks every entry point that takes a context starts with, in this order: a context, no *_async step in flight (its kernels
// and its state download are still running on the context's stream, and lvo_wait finishes it), and for the per-lane calls a lane
// of the context.  Exempt: lvo_destroy and lvo_last_error (usable at any time) and lvo_wait (its own check is the inverse).
static int lvo_enter(const lvo_ctx* c, bool has_lane, int lane) {
  if (!c) return LVO_E_BADARG;
  if (c->pending) { c->err = "lvo_wait has not been called for the last *_async step"; return LVO_E_STATE; }
  if (has_lane && (lane < 0 || lane >= c->lanes)) { c->err = "lane out of range"; return LVO_E_BADARG; }
  return LVO_OK;
}
// The context's device is current until the entry point returns.
#define LVO_ENTER(c) LvoDeviceGuard _dev(c); LVO_TRY(lvo_enter((c), false, 0))
#define LVO_ENTER_LANE(c, lane) LvoDeviceGuard _dev(c); LVO_TRY(lvo_enter((c), true, (lane)))

static void destroy_graphs(lvo_ctx* c) {
  for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) if (c->graph_exec[a][b]) { cudaGraphExecDestroy(c->graph_exec[a][b]); c->graph_exec[a][b] = nullptr; }
}

extern "C" {

void lvo_default_config(lvo_config* cfg) {
  if (!cfg) return;
  memset(cfg, 0, sizeof(*cfg));
  cfg->n_scans = 64; cfg->minimum_range = 5.0; cfg->line_res = 0.4; cfg->plane_res = 0.8;  // launch/aloam_velodyne_HDL_64.launch:3-13
  cfg->skip_frame = 1; cfg->outer_iters = 10; cfg->lm_max_iters = 4; cfg->huber = 0.1; cfg->device = 0; cfg->lanes = 1;
  cfg->max_points = 0; cfg->max_map_corner = 0; cfg->max_map_surf = 0;
  cfg->distortion = 0;  // laserOdometry.cpp:67
  cfg->debug_probes = 0;
}

int lvo_create(const lvo_config* cfg, lvo_ctx** out) {
  if (!cfg || !out) return LVO_E_BADARG;
  *out = nullptr;
  if (cfg->n_scans != 16 && cfg->n_scans != 32 && cfg->n_scans != 64) return LVO_E_BADARG;  // "wrong scan number", scanRegistration.cpp:203
  if (cfg->distortion < 0 || cfg->distortion > 2) return LVO_E_BADARG;
  if (cfg->lanes < 1 || cfg->outer_iters < 1 || cfg->outer_iters > LVO_MAX_OUTER || cfg->lm_max_iters < 0 || cfg->lm_max_iters > LVO_MAX_LM) return LVO_E_BADARG;
  lvo_ctx* c = new (std::nothrow) lvo_ctx();
  if (!c) return LVO_E_CUDA;
  *out = c;  // returned even on failure so that lvo_last_error works; caller destroys it
  c->cfg = *cfg;
  if (c->cfg.skip_frame < 1) c->cfg.skip_frame = 1;
  c->lanes = cfg->lanes;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { lvo_set_error(c, "no CUDA device: liblvo has no CPU fallback"); return LVO_E_CUDA; }
  struct RestoreDevice { int prev = -1; ~RestoreDevice() { if (prev >= 0) cudaSetDevice(prev); } } restore;   // the caller's current device is left as it was
  cudaGetDevice(&restore.prev);
  LVO_CUDA_OK(c, cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  LVO_CUDA_OK(c, cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) { lvo_set_error(c, "liblvo is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor)); return LVO_E_CUDA; }
  LVO_CUDA_OK(c, cudaStreamCreateWithFlags(&c->own_st, cudaStreamNonBlocking));
  c->st = c->own_st;
  for (int i = 0; i < 8; ++i) LVO_CUDA_OK(c, cudaEventCreate(&c->ev[i]));
  memset(&c->tim, 0, sizeof(c->tim));

  const int L = c->lanes;
  const int P = c->P = cfg->max_points > 0 ? cfg->max_points : 262144;
  const FeatureCaps fc = feature_caps(cfg->n_scans);
  c->cap_sharp = fc.sharp; c->cap_lsharp = fc.lsharp; c->cap_flat = fc.flat;
  const int mapc[2] = {cfg->max_map_corner > 0 ? cfg->max_map_corner : (1 << 20), cfg->max_map_surf > 0 ? cfg->max_map_surf : (1 << 21)};
  c->lane_status.assign(L, 0);
  c->lane_frame.assign(L, 0);
  c->lane_active.assign(L, 1);
  c->lane_map_update.assign(L, 1);
  c->probe_gate.assign(L, 0);
  c->reg_n.assign(L, 0);
  c->unc_frame.assign(2 * (size_t)L, -1);
  c->lane_cfg.assign(L, lvo_lane_config{c->cfg.n_scans, c->cfg.minimum_range, c->cfg.line_res, c->cfg.plane_res, c->cfg.skip_frame});

  LVO_TRY(dalloc(c, &c->d_ls, (size_t)L));
  LVO_TRY(halloc(c, &c->h_ls, (size_t)L));
  k_init_lanes<<<lvo_div_up(L, 64), 64, 0, c->st>>>(c->d_ls, 0, L);
  LVO_TRY(dalloc(c, &c->d_lcfg, (size_t)L, false)); LVO_TRY(halloc(c, &c->h_lcfg, (size_t)L));
  for (int l = 0; l < L; ++l) LVO_TRY(upload_lane_config(c, l));
  c->raw_lane_bytes = (size_t)P * 32;
  LVO_TRY(dalloc(c, &c->d_raw, c->raw_lane_bytes * L, false));
  LVO_TRY(dalloc(c, &c->d_in_ptr, (size_t)L)); LVO_TRY(halloc(c, &c->h_in_ptr, (size_t)L));
  LVO_TRY(dalloc(c, &c->d_in_n, (size_t)2 * L)); LVO_TRY(halloc(c, &c->h_in_n, (size_t)2 * L));
  LVO_TRY(flags_all_lanes(c, true));
  LVO_TRY(dalloc(c, (unsigned char**)&c->d_upload, (size_t)std::max(P, std::max(mapc[0], mapc[1])) * 64, false));

  // ---- extract
  ExtractArgs& ex = c->ex;
  memset(&ex, 0, sizeof(ex));
  ex.in_ptr = c->d_in_ptr; ex.in_n = c->d_in_n; ex.lane_flags = c->d_in_n + L; ex.lcfg = c->d_lcfg; ex.max_scans = cfg->n_scans;
  ex.P = P; ex.nblk_cap = lvo_div_up(P, LVO_EX_THREADS); ex.ls = c->d_ls;
  LVO_TRY(dalloc(c, &ex.ring, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.ori, (size_t)L * P));
  LVO_TRY(dalloc(c, &ex.blkcnt, (size_t)L * ex.nblk_cap * LVO_MAX_RINGS));
  LVO_TRY(dalloc(c, &ex.full, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.curv, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.gapbig, (size_t)L * P));
  LVO_TRY(dalloc(c, &ex.sort_ind, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.picked, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.label, (size_t)L * P));
  const size_t nsec = (size_t)L * LVO_MAX_RINGS * LVO_SECTORS;
  LVO_TRY(dalloc(c, &ex.slot_sharp, nsec * 2)); LVO_TRY(dalloc(c, &ex.slot_lsharp, nsec * 20)); LVO_TRY(dalloc(c, &ex.slot_flat, nsec * 4));
  LVO_TRY(dalloc(c, &ex.slot_cnt, nsec * 3));
  LVO_TRY(dalloc(c, &ex.lf_ring, (size_t)L * P)); LVO_TRY(dalloc(c, &ex.lf_cnt, (size_t)L * LVO_MAX_RINGS));
  LVO_TRY(dalloc(c, &ex.sort_scratch, (size_t)L * 2 * P, false));
  LVO_TRY(dalloc(c, &ex.ring_done, (size_t)L * LVO_MAX_RINGS));
  LVO_TRY(dalloc(c, &ex.sharp, (size_t)L * c->cap_sharp)); LVO_TRY(dalloc(c, &ex.less_sharp, (size_t)L * c->cap_lsharp));
  LVO_TRY(dalloc(c, &ex.flat, (size_t)L * c->cap_flat)); LVO_TRY(dalloc(c, &ex.less_flat, (size_t)L * P));
  ex.cap_sharp = c->cap_sharp; ex.cap_lsharp = c->cap_lsharp; ex.cap_flat = c->cap_flat;

  // ---- solver
  SolveArgs& so = c->solve;
  memset(&so, 0, sizeof(so));
  so.ls = c->d_ls; so.max_iters = cfg->lm_max_iters; so.huber = cfg->huber;
  so.n_outer = cfg->outer_iters; so.fixpoint_skip = 1;
  LVO_TRY(dalloc(c, &c->d_unc, 2 * (size_t)L));
  LVO_TRY(dalloc(c, &c->d_unc_out, 2 * (size_t)L, false)); LVO_TRY(halloc(c, &c->h_unc, 2 * (size_t)L));
  so.unc = c->d_unc;
  const size_t trace_n = (size_t)L * LVO_MAX_OUTER * (LVO_MAX_LM + 1) * LVO_TRACE_W;
  LVO_TRY(dalloc(c, &c->d_trace[0], trace_n)); LVO_TRY(dalloc(c, &c->d_trace[1], trace_n));

  // ---- odometry
  OdoArgs& od = c->odo;
  memset(&od, 0, sizeof(od));
  od.ls = c->d_ls; od.lanes = L; od.distortion = cfg->distortion; od.full = ex.full; od.lane_flags = ex.lane_flags; od.unc = c->d_unc;
  od.sharp = ex.sharp; od.less_sharp = ex.less_sharp; od.flat = ex.flat; od.less_flat = ex.less_flat;
  od.cap_sharp = c->cap_sharp; od.cap_lsharp = c->cap_lsharp; od.cap_flat = c->cap_flat; od.P = P;
  // per-outer-iteration probe arrays: all LVO_MAX_OUTER iterations only when the parity probes are wanted, else the current and the previous one
  const int slots = cfg->debug_probes ? LVO_MAX_OUTER : 2;
  od.slots = slots;
  LVO_TRY(dalloc(c, &od.corner_last, (size_t)L * c->cap_lsharp)); LVO_TRY(dalloc(c, &od.surf_last, (size_t)L * P));
  od.factor_cap = std::max(c->cap_sharp + c->cap_flat, c->cap_lsharp + P);
  LVO_TRY(dalloc(c, &od.factors, (size_t)L * od.factor_cap));
  LVO_TRY(dalloc(c, &od.slow_list, (size_t)L * (c->cap_sharp + c->cap_flat))); LVO_TRY(dalloc(c, &od.slow_cnt, (size_t)L));
  od.reuse = 1;   // default: correspondences carried across the outer iterations with a certificate
  LVO_TRY(dalloc(c, &od.ref, (size_t)L * (c->cap_sharp + c->cap_flat))); LVO_TRY(dalloc(c, &od.guard, (size_t)L * (c->cap_sharp + c->cap_flat)));
  LVO_TRY(dalloc(c, &od.sel, (size_t)L * (c->cap_sharp + c->cap_flat)));
  LVO_TRY(dalloc(c, &od.corner_corr, (size_t)L * slots * c->cap_sharp * 2));
  LVO_TRY(dalloc(c, &od.plane_corr, (size_t)L * slots * c->cap_flat * 3));
  const size_t odo_cells = 2 * ((size_t)(1 << 22) + (size_t)LVO_AZ_BUCKETS * LVO_AZ_RINGS + (1 << 19));   // per lane, see k_setup_grid_problems
  LVO_TRY(alloc_grid(c, &od.grid, LVO_ODO_GRIDS * L, 1 << 22, (size_t)3 * L * (c->cap_lsharp + P), P, odo_cells * L));
  k_setup_grid_problems<<<lvo_div_up(LVO_ODO_GRIDS * L, 64), 64, 0, c->st>>>(od.grid.prob, LVO_ODO_GRIDS * L, od.corner_last, (size_t)c->cap_lsharp, od.surf_last, (size_t)P, c->d_ls, 0, 1.0f);

  // ---- mapping
  MapArgs& mp = c->map;
  memset(&mp, 0, sizeof(mp));
  mp.ls = c->d_ls; mp.lanes = L; mp.lane_flags = ex.lane_flags; mp.lcfg = c->d_lcfg; mp.unc = c->d_unc;
  mp.in_pts[0] = ex.less_sharp; mp.in_pts[1] = ex.less_flat; mp.in_cap[0] = c->cap_lsharp; mp.in_cap[1] = P;
  mp.full = ex.full; mp.P = P; mp.gen = 0; mp.slots = slots;
  mp.knn_reuse = 1;   // default: neighbour sets carried across the outer iterations with a certificate
  lvo_extract_kernel_attributes();
  for (int t = 0; t < 2; ++t) {
    mp.map_cap[t] = mapc[t];
    for (int g = 0; g < 2; ++g) {
      LVO_TRY(dalloc(c, &mp.map_pts[g][t], (size_t)L * mapc[t], false));
      LVO_TRY(dalloc(c, &mp.cube_start[g][t], (size_t)L * (LVO_NCUBES + 1)));
    }
    LVO_TRY(dalloc(c, &mp.from_map[t], (size_t)L * mapc[t], false));
    LVO_TRY(dalloc(c, &mp.stack[t], (size_t)L * mp.in_cap[t]));
    LVO_TRY(dalloc(c, &mp.knn_ind[t], (size_t)L * slots * mp.in_cap[t] * 5));
    LVO_TRY(dalloc(c, &mp.fac_valid[t], (size_t)L * slots * mp.in_cap[t]));
    LVO_TRY(dalloc(c, &mp.knn_ref[t], (size_t)L * mp.in_cap[t], false));
    LVO_TRY(dalloc(c, &mp.knn_sel[t], (size_t)L * mp.in_cap[t] * 5, false));
    LVO_TRY(dalloc(c, &mp.knn_flag[t], (size_t)L * mp.in_cap[t], false));
  }
  LVO_TRY(alloc_grid(c, &mp.grid, 2 * L, 1 << 21, (size_t)L * ((size_t)mapc[0] + mapc[1]), std::max(mapc[0], mapc[1])));   // 2 M cells of 1 m: a 250 x 250 x 32 m neighbourhood; larger boxes double the cell edge
  k_setup_grid_problems<<<lvo_div_up(2 * L, 64), 64, 0, c->st>>>(mp.grid.prob, 2 * L, mp.from_map[0], (size_t)mapc[0], mp.from_map[1], (size_t)mapc[1], c->d_ls, 1, 1.0f);
  LVO_TRY(dalloc(c, &mp.item_off, (size_t)2 * L + 1));
  LVO_TRY(dalloc(c, &mp.fit_list, (size_t)L * (mp.in_cap[0] + mp.in_cap[1]), false));
  LVO_TRY(dalloc(c, &mp.fit_cnt, (size_t)L * LVO_MAX_OUTER));
  mp.factors = od.factors; mp.factor_cap = od.factor_cap;
  LVO_TRY(dalloc(c, &mp.app_cnt, (size_t)2 * L * LVO_NCUBES)); LVO_TRY(dalloc(c, &mp.app_first, (size_t)2 * L * LVO_NCUBES));
  LVO_TRY(dalloc(c, &mp.new_cnt, (size_t)2 * L * (LVO_NCUBES + 1)));
  LVO_TRY(dalloc(c, &mp.registered, (size_t)L * P, false));
  // voxel engine shared by the stack downsample and the cube re-filter
  VoxelEngine& vx = mp.vx;
  vx.cap_items = (int)std::min<size_t>((size_t)L * ((size_t)mapc[0] + mapc[1] + c->cap_lsharp + P), (size_t)INT_MAX - 4096);
  vx.cap_segs = 2 * L * LVO_MSEGS;
  const size_t NI = (size_t)vx.cap_items, NS = (size_t)vx.cap_segs;
  LVO_TRY(dalloc(c, &vx.in_pts, NI, false)); LVO_TRY(dalloc(c, &vx.in_seg, NI)); LVO_TRY(dalloc(c, &vx.in_aux, NI));
  LVO_TRY(dalloc(c, &vx.d_n, 1)); LVO_TRY(dalloc(c, &vx.seg_leaf, NS)); LVO_TRY(dalloc(c, &vx.d_nsegs, 1));
  LVO_TRY(dalloc(c, &vx.seg_mn, 3 * NS)); LVO_TRY(dalloc(c, &vx.seg_mx, 3 * NS)); LVO_TRY(dalloc(c, &vx.seg_minb, 3 * NS));
  LVO_TRY(dalloc(c, &vx.seg_div, 2 * NS)); LVO_TRY(dalloc(c, &vx.seg_mode, NS)); LVO_TRY(dalloc(c, &vx.d_vbits, 1)); LVO_TRY(dalloc(c, &vx.d_bits, 1));
  for (int k = 0; k < 2; ++k) { LVO_TRY(dalloc(c, &vx.sort.keys[k], NI, false)); LVO_TRY(dalloc(c, &vx.sort.vals[k], NI, false)); }
  const size_t tiles = (size_t)lvo_div_up((long long)NI, LVO_SORT_TILE) + 1;
  LVO_TRY(dalloc(c, &vx.sort.ghist, (size_t)LVO_SORT_GHIST_WORDS)); LVO_TRY(dalloc(c, &vx.sort.d_epoch, 1));
  LVO_TRY(dalloc(c, &vx.sort.status, 256 * tiles));   // zero-filled once: epoch 0 never matches (k_sort_ghist bumps the epoch before the first pass)
  vx.sort.cap = vx.cap_items;
  LVO_TRY(dalloc(c, &vx.outpos, NI)); LVO_TRY(dalloc(c, &vx.out_pts, NI, false)); LVO_TRY(dalloc(c, &vx.out_aux, NI));
  LVO_TRY(dalloc(c, &vx.seg_out_cnt, NS)); LVO_TRY(dalloc(c, &vx.seg_out_start, NS + 1)); LVO_TRY(dalloc(c, &vx.d_n_out, 1));
  LVO_TRY(alloc_scan(c, &vx.scan, std::max(NI, NS + 1)));

  // stand-alone kNN operator: one problem, storage borrowed from the mapping grid
  c->gknn = mp.grid; c->gknn.nprob = 1;
  LVO_TRY(dalloc(c, &c->d_knn_prob, 1)); LVO_TRY(dalloc(c, &c->d_knn_n, 1));
  c->gknn.prob = c->d_knn_prob;
  LVO_TRY(dalloc(c, &c->d_knn_ind, (size_t)P * 5)); LVO_TRY(dalloc(c, &c->d_knn_sq, (size_t)P * 5));

  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

int lvo_destroy(lvo_ctx* c) {
  if (!c) return LVO_E_BADARG;
  LvoDeviceGuard _dev(c);
  if (c->st) cudaStreamSynchronize(c->st);
  c->mem.release();
  c->depth.mem.release();
  c->mapout.mem.release();
  c->mapout.pts_mem.release();
  destroy_graphs(c);
  if (c->copy_st) { cudaStreamSynchronize(c->copy_st); cudaStreamDestroy(c->copy_st); cudaEventDestroy(c->copy_ev); cudaEventDestroy(c->compute_ev); }
  if (c->own_st) { for (int i = 0; i < 8; ++i) cudaEventDestroy(c->ev[i]); c->stage_tm.destroy(); cudaStreamDestroy(c->own_st); }
  delete c;
  return LVO_OK;
}

const char* lvo_last_error(const lvo_ctx* c) { return c ? c->err.c_str() : "null context"; }

int lvo_get_stats(const lvo_ctx* c, int lane, lvo_stats* out, size_t bytes) {
  LVO_ENTER_LANE(c, lane);
  if (!out) return LVO_E_BADARG;
  memcpy(out, &c->h_ls[lane].stats, std::min(bytes, sizeof(lvo_stats)));
  return LVO_OK;
}
int lvo_lane_status(const lvo_ctx* c, int lane) {
  LVO_ENTER_LANE(c, lane);
  return c->lane_status[lane];
}
size_t lvo_state_bytes(void) { return sizeof(LaneState); }
int lvo_set_option(lvo_ctx* c, int option, int value) {
  LVO_ENTER(c);
  if (option == LVO_OPT_GRAPHS) { c->opt_graphs = value; return LVO_OK; }
  if (option == LVO_OPT_STAGE_TIMING) { c->opt_stage_timing = value ? 1 : 0; return LVO_OK; }
  if (option == LVO_OPT_ODO_REUSE) {
    if (c->st) cudaStreamSynchronize(c->st);
    destroy_graphs(c);
    c->odo.reuse = value ? 1 : 0;
    return LVO_OK;
  }
  if (option == LVO_OPT_KNN_REUSE) {
    if (c->st) cudaStreamSynchronize(c->st);
    destroy_graphs(c);
    c->map.knn_reuse = value ? 1 : 0;
    return LVO_OK;
  }
  if (option == LVO_OPT_FIXPOINT_SKIP) {   // a kernel argument: captured graphs hold the old value
    if (c->st) cudaStreamSynchronize(c->st);
    destroy_graphs(c);
    c->solve.fixpoint_skip = value ? 1 : 0;
    return LVO_OK;
  }
  return LVO_E_BADARG;
}
int lvo_set_stream(lvo_ctx* c, void* cuda_stream) {
  LVO_ENTER(c);
  cudaStreamSynchronize(c->st);
  destroy_graphs(c);
  c->st = cuda_stream ? (cudaStream_t)cuda_stream : c->own_st;
  return LVO_OK;
}
int lvo_get_timings(const lvo_ctx* c, lvo_timings* out) {
  LVO_ENTER(c);
  if (!out) return LVO_E_BADARG;
  *out = c->tim;
  out->kernel_launches = (int)c->launches;
  return LVO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
int lvo_extract_features(lvo_ctx* c, lvo_cloud_view sweep, lvo_cloud_out* full, lvo_cloud_out* sharp, lvo_cloud_out* less_sharp, lvo_cloud_out* flat,
                         lvo_cloud_out* less_flat) {
  LVO_ENTER(c);
  LVO_TRY(check_view(c, sweep, (size_t)c->P, true));
  c->launches = 0;
  cudaEventRecord(c->ev[0], c->st);
  if (sweep.n) LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_raw, sweep.data, sweep.n * sweep.stride, cudaMemcpyHostToDevice, c->st));
  for (int l = 0; l < c->lanes; ++l) { c->h_in_ptr[l] = c->d_raw + c->raw_lane_bytes * l; c->h_in_n[l] = l == 0 ? (int)sweep.n : 0; }
  LVO_TRY(flags_all_lanes(c, false));
  LVO_TRY(set_inputs(c));
  LvoStageTimer* tm = stage_timer_begin(c, true);
  enqueue_extract(c, sweep.n ? (int)sweep.stride : 16, sweep.n ? (int)sweep.off_xyz : 0, (int)sweep.n, tm);
  stage_ran_on_all_lanes(c, LVO_PROBE_GATE_EXTRACT);
  c->stage_tm.stop(c->st);
  cudaEventRecord(c->ev[1], c->st);
  LVO_TRY(sync_state(c));
  cudaEventElapsedTime(&c->tim.extract_ms, c->ev[0], c->ev[1]);
  collect_stage_timing(c, false);
  const LaneState& s = c->h_ls[0];
  int r = LVO_OK, q;
  if ((q = download_cloud(c, c->ex.full, (size_t)s.n_kept, full)) != LVO_OK) r = q;
  if ((q = download_cloud(c, c->ex.sharp, (size_t)s.n_sharp, sharp)) != LVO_OK) r = q;
  if ((q = download_cloud(c, c->ex.less_sharp, (size_t)s.n_less_sharp, less_sharp)) != LVO_OK) r = q;
  if ((q = download_cloud(c, c->ex.flat, (size_t)s.n_flat, flat)) != LVO_OK) r = q;
  if ((q = download_cloud(c, c->ex.less_flat, (size_t)s.n_less_flat, less_flat)) != LVO_OK) r = q;
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  c->lane_status[0] = r;
  return r;
}

int lvo_scan_to_scan(lvo_ctx* c, lvo_cloud_view sharp, lvo_cloud_view less_sharp, lvo_cloud_view flat, lvo_cloud_view less_flat, lvo_pose* T_last_curr,
                     lvo_pose* T_w_curr) {
  LVO_ENTER(c);
  const FeatureCaps fc = feature_caps(c->lane_cfg[0].n_scans);   // lane 0's n_scans
  LVO_TRY(check_view(c, sharp, (size_t)fc.sharp)); LVO_TRY(check_view(c, less_sharp, (size_t)fc.lsharp));
  LVO_TRY(check_view(c, flat, (size_t)fc.flat)); LVO_TRY(check_view(c, less_flat, (size_t)c->P));
  c->launches = 0;
  rebuild_stale_grids(c);
  cudaEventRecord(c->ev[2], c->st);
  LVO_TRY(upload_cloud(c, sharp, c->ex.sharp)); LVO_TRY(upload_cloud(c, less_sharp, c->ex.less_sharp));
  LVO_TRY(upload_cloud(c, flat, c->ex.flat)); LVO_TRY(upload_cloud(c, less_flat, c->ex.less_flat));
  SetCounts sc; memset(&sc, 0, sizeof(sc));
  sc.what = 0; sc.v[0] = (int)sharp.n; sc.v[1] = (int)less_sharp.n; sc.v[2] = (int)flat.n; sc.v[3] = (int)less_flat.n;
  k_set_lane<<<1, 1, 0, c->st>>>(c->d_ls, 0, sc);
  LVO_TRY(flags_all_lanes(c, true));
  c->solve.trace = c->d_trace[0];
  LvoStageTimer* tm = stage_timer_begin(c, true);
  enqueue_odometry(c, tm);
  stage_ran_on_all_lanes(c, LVO_PROBE_GATE_ODO);
  uncertainty_written(c, 0);
  c->stage_tm.stop(c->st);
  cudaEventRecord(c->ev[3], c->st);
  LVO_TRY(sync_state(c));
  cudaEventElapsedTime(&c->tim.odometry_ms, c->ev[2], c->ev[3]);
  collect_stage_timing(c, false);
  const LaneState& s = c->h_ls[0];
  pose_out(T_last_curr, s.para_q, s.para_t);
  pose_out(T_w_curr, s.q_w, s.t_w);
  c->lane_status[0] = s.odo_status;
  return s.odo_status;
}

int lvo_scan_to_map(lvo_ctx* c, lvo_cloud_view corner_last, lvo_cloud_view surf_last, lvo_cloud_view full_or_null, const lvo_pose* T_wodom_curr,
                    lvo_pose* T_wmap_curr, lvo_cloud_out* registered_or_null) {
  LVO_ENTER(c);
  if (!T_wodom_curr) return LVO_E_BADARG;
  LVO_TRY(check_view(c, corner_last, (size_t)feature_caps(c->lane_cfg[0].n_scans).lsharp)); LVO_TRY(check_view(c, surf_last, (size_t)c->P));
  LVO_TRY(check_view(c, full_or_null, (size_t)c->P));
  c->launches = 0;
  c->reg_valid = false;   // its k_register rewrites map.registered
  cudaEventRecord(c->ev[4], c->st);
  LVO_TRY(upload_cloud(c, corner_last, c->ex.less_sharp)); LVO_TRY(upload_cloud(c, surf_last, c->ex.less_flat));
  const bool want_reg = registered_or_null && full_or_null.n > 0;
  if (full_or_null.n) LVO_TRY(upload_cloud(c, full_or_null, c->ex.full));
  SetCounts sc; memset(&sc, 0, sizeof(sc));
  sc.what = 1; sc.v[0] = (int)corner_last.n; sc.v[1] = (int)surf_last.n; sc.v[2] = (int)full_or_null.n;
  for (int k = 0; k < 4; ++k) sc.pose[k] = T_wodom_curr->q[k];
  for (int k = 0; k < 3; ++k) sc.pose[4 + k] = T_wodom_curr->t[k];
  k_set_lane<<<1, 1, 0, c->st>>>(c->d_ls, 0, sc);
  LVO_TRY(flags_all_lanes(c, true));
  c->solve.trace = c->d_trace[1];
  LvoStageTimer* tm = stage_timer_begin(c, true);
  enqueue_mapping(c, 0, want_reg, tm);
  stage_ran_on_all_lanes(c, LVO_PROBE_GATE_MAP);
  uncertainty_written(c, 1);
  c->stage_tm.stop(c->st);
  cudaEventRecord(c->ev[5], c->st);
  LVO_TRY(sync_state(c));
  cudaEventElapsedTime(&c->tim.mapping_ms, c->ev[4], c->ev[5]);
  collect_stage_timing(c, true);
  const LaneState& s = c->h_ls[0];
  pose_out(T_wmap_curr, s.map_x, s.map_x + 4);
  int r = s.map_status;
  if (registered_or_null) {
    int q = download_cloud(c, c->map.registered, want_reg ? full_or_null.n : 0, registered_or_null);
    if (q != LVO_OK) r = q;
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  }
  if (r == LVO_E_CAPACITY) lvo_set_error(c, "map capacity exceeded (max_map_corner / max_map_surf)");
  c->lane_status[0] = r;
  return r;
}

// ---------------------------------------------------------------------------------------------------------------
// Upload of the next frame into the staging buffer that is not in use, on the copy stream (lvo_step_batch_pipelined).  That buffer
// was last read by the previous frame's kernels, which have completed (every call ends synchronised).  Issued BEFORE this frame's
// kernels are enqueued, so that the copy engine starts at once; the uploads are merged per run of adjacent lanes (stage_sweeps).
static int enqueue_prefetch(lvo_ctx* c) {
  const lvo_cloud_view* next = c->pending_next;
  c->pending_next = nullptr;
  if (!next) return LVO_OK;
  unsigned char* bufs[2] = {c->d_raw, c->d_raw2};
  // stage_sweeps fills h_in_ptr / h_in_n for the NEXT frame: keep this frame's, which set_inputs has not uploaded yet
  std::vector<const unsigned char*> keep_ptr(c->h_in_ptr, c->h_in_ptr + c->lanes);
  std::vector<int> keep_n(c->h_in_n, c->h_in_n + c->lanes);
  const int r = stage_sweeps(c, next, bufs[c->raw_cur ^ 1], c->copy_st);
  c->next_in_ptr.assign(c->h_in_ptr, c->h_in_ptr + c->lanes);
  std::copy(keep_ptr.begin(), keep_ptr.end(), c->h_in_ptr);
  std::copy(keep_n.begin(), keep_n.end(), c->h_in_n);
  if (r != LVO_OK) return r;
  LVO_CUDA_OK(c, cudaEventRecord(c->copy_ev, c->copy_st));
  c->prefetched.assign(c->lanes, lvo_cloud_view{});
  for (int l = 0; l < c->lanes; ++l) if (c->lane_active[l]) c->prefetched[l] = next[l];
  c->prefetched_active = c->lane_active;
  return LVO_OK;
}

// Enqueue one frame for every active lane (no host synchronisation).  h_in_ptr / h_in_n hold the sweeps, 0 points for idle lanes.
static int step_enqueue(lvo_ctx* c, int stride, int off_xyz, int max_n) {
  c->launches = 0;
  LVO_TRY(enqueue_prefetch(c));
  rebuild_stale_grids(c);             // outside the graph: a step without a preceding lvo_lane_load launches nothing more
  const long long pre_launches = c->launches;
  // a lane maps on its own frames 0, skip_frame, 2 skip_frame, ... of its own skip_frame (laserOdometry.cpp:643); the mapping stage
  // is enqueued when any lane maps, and the kernels pass the others through (LVO_LANE_MAPS)
  bool do_map = false;
  for (int l = 0; l < c->lanes; ++l) {
    const bool maps = c->lane_active[l] && (c->lane_frame[l] % c->lane_cfg[l].skip_frame) == 0;
    lane_flags(c)[l] = (c->lane_active[l] ? LVO_LANE_ACTIVE : 0) | (maps ? LVO_LANE_MAPS : 0) | (maps && !c->lane_map_update[l] ? LVO_LANE_MAP_FIXED : 0);
    do_map = do_map || maps;
  }
  LVO_TRY(set_inputs(c));
  const bool want_graph = c->opt_graphs == 1 || (c->opt_graphs < 0 && c->lanes <= 8);
  const bool use_graph = want_graph && c->st != nullptr;    // the legacy default stream cannot be captured
  nvtxRangePushA("lvo_step");
  if (use_graph) {
    if (c->graph_stride != stride || c->graph_off != off_xyz) { destroy_graphs(c); c->graph_stride = stride; c->graph_off = off_xyz; }
    const int gen = c->map.gen;
    stage_timer_begin(c, false);
    cudaEventRecord(c->ev[0], c->st);
    if (!c->graph_exec[do_map][gen]) {
      // capture one frame: the launch sequence is static (grids from capacities, sizes read from device memory)
      cudaGraph_t graph = nullptr;
      LVO_CUDA_OK(c, cudaStreamBeginCapture(c->st, cudaStreamCaptureModeThreadLocal));
      enqueue_extract(c, stride, off_xyz, c->P, nullptr);
      c->solve.trace = c->d_trace[0];
      enqueue_odometry(c, nullptr);
      if (do_map) { c->solve.trace = c->d_trace[1]; enqueue_mapping(c, 1, true, nullptr); }
      cudaError_t e = cudaStreamEndCapture(c->st, &graph);
      if (do_map) c->map.gen = gen;   // enqueue_mapping flipped it; the flip belongs to the execution below
      if (e != cudaSuccess || !graph) { nvtxRangePop(); lvo_set_error(c, std::string("graph capture: ") + cudaGetErrorString(e)); return LVO_E_CUDA; }
      e = cudaGraphInstantiate(&c->graph_exec[do_map][gen], graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { nvtxRangePop(); lvo_set_error(c, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e)); return LVO_E_CUDA; }
      c->graph_launches[do_map][gen] = c->launches - pre_launches;
    }
    cudaError_t ge = cudaGraphLaunch(c->graph_exec[do_map][gen], c->st);
    if (ge != cudaSuccess) { nvtxRangePop(); lvo_set_error(c, std::string("cudaGraphLaunch: ") + cudaGetErrorString(ge)); return LVO_E_CUDA; }
    c->launches = pre_launches + c->graph_launches[do_map][gen];
    if (do_map) c->map.gen = gen ^ 1;
    cudaEventRecord(c->ev[3], c->st);
  } else {
    LvoStageTimer* tm = stage_timer_begin(c, c->opt_stage_timing != 0);
    cudaEventRecord(c->ev[0], c->st);
    enqueue_extract(c, stride, off_xyz, max_n, tm);
    cudaEventRecord(c->ev[1], c->st);
    c->solve.trace = c->d_trace[0];
    enqueue_odometry(c, tm);
    cudaEventRecord(c->ev[2], c->st);
    if (do_map) { c->solve.trace = c->d_trace[1]; enqueue_mapping(c, 1, true, tm); }
    c->stage_tm.stop(c->st);
    cudaEventRecord(c->ev[3], c->st);
  }
  nvtxRangePop();
  for (int l = 0; l < c->lanes; ++l) {
    const int f = lane_flags(c)[l];
    if (f & LVO_LANE_ACTIVE) c->unc_frame[2 * l] = c->lane_frame[l];       // the frame index of this step
    if (f & LVO_LANE_MAPS) c->unc_frame[2 * l + 1] = c->lane_frame[l];
    if (f & LVO_LANE_ACTIVE) { c->lane_frame[l]++; c->probe_gate[l] &= ~(LVO_PROBE_GATE_EXTRACT | LVO_PROBE_GATE_ODO); }
    if (f & LVO_LANE_MAPS) c->probe_gate[l] = 0;
  }
  c->unc_epoch++;
  // the lane states come back on the same stream; lvo_wait only has to synchronise
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->h_ls, c->d_ls, sizeof(LaneState) * c->lanes, cudaMemcpyDeviceToHost, c->st));
  c->pending = true; c->pending_do_map = do_map; c->pending_graph = use_graph;
  return LVO_OK;
}

// Wait for the frame enqueued by step_enqueue and deliver its results.
static int step_finish(lvo_ctx* c, lvo_pose* T_wodom, lvo_pose* T_wmap) {
  if (!c->pending) { lvo_set_error(c, "lvo_wait without a step in flight"); return LVO_E_STATE; }
  c->pending = false;
  const bool do_map = c->pending_do_map;
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  // the registered clouds of this step (k_register ran for the lanes that mapped): their sizes are n_kept of this frame, read here
  // because a later extraction rewrites n_kept
  for (int l = 0; l < c->lanes; ++l) c->reg_n[l] = (lane_flags(c)[l] & LVO_LANE_MAPS) ? (size_t)c->h_ls[l].n_kept : 0;
  c->reg_valid = true;
  if (c->pending_graph) {
    c->tim.extract_ms = c->tim.odometry_ms = 0.f;     // per-stage times are only available with plain launches
    cudaEventElapsedTime(&c->tim.mapping_ms, c->ev[0], c->ev[3]);
  } else {
    cudaEventElapsedTime(&c->tim.extract_ms, c->ev[0], c->ev[1]);
    cudaEventElapsedTime(&c->tim.odometry_ms, c->ev[1], c->ev[2]);
    cudaEventElapsedTime(&c->tim.mapping_ms, c->ev[2], c->ev[3]);
  }
  collect_stage_timing(c, do_map);
  int worst = LVO_OK;
  for (int l = 0; l < c->lanes; ++l) {
    const int flags = lane_flags(c)[l];
    if (!(flags & LVO_LANE_ACTIVE)) continue;   // idle: poses not written, status unchanged
    const bool mapped = (flags & LVO_LANE_MAPS) != 0;
    const LaneState& s = c->h_ls[l];
    if (T_wodom) pose_out(&T_wodom[l], s.q_w, s.t_w);
    if (T_wmap) {
      if (mapped) pose_out(&T_wmap[l], s.map_x, s.map_x + 4);
      else {  // high-frequency pose: q_wmap_wodom * odom (laserMapping.cpp:214-215), evaluated on the host
        const double* a = s.q_wmap_wodom; const double* b = s.q_w;
        double q[4] = {a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1], a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2],
                       a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0], a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2]};
        const double v[3] = {s.t_w[0], s.t_w[1], s.t_w[2]};
        const double uv[3] = {2 * (a[1] * v[2] - a[2] * v[1]), 2 * (a[2] * v[0] - a[0] * v[2]), 2 * (a[0] * v[1] - a[1] * v[0])};
        const double t[3] = {v[0] + a[3] * uv[0] + (a[1] * uv[2] - a[2] * uv[1]) + s.t_wmap_wodom[0], v[1] + a[3] * uv[1] + (a[2] * uv[0] - a[0] * uv[2]) + s.t_wmap_wodom[1],
                             v[2] + a[3] * uv[2] + (a[0] * uv[1] - a[1] * uv[0]) + s.t_wmap_wodom[2]};
        pose_out(&T_wmap[l], q, t);
      }
    }
    int st = s.odo_status;
    if (mapped && s.map_status != LVO_OK) st = s.map_status < 0 ? s.map_status : std::max(st, s.map_status);
    c->lane_status[l] = st;
    if (st < 0) worst = st; else if (worst >= 0) worst = std::max(worst, st);
  }
  if (worst == LVO_E_CAPACITY) lvo_set_error(c, "map capacity exceeded (max_map_corner / max_map_surf)");
  return worst;
}

// Validates the views of the active lanes (idle lanes' views are not read) and returns their shared layout.  With no lane active the
// layout of the captured graphs is kept, so that a step of idle lanes does not force a new capture.
static int check_sweeps(lvo_ctx* c, const lvo_cloud_view* sweeps, int* max_n, int* stride, int* off_xyz) {
  *max_n = 0;
  int first = -1;
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l]) continue;
    if (first < 0) first = l;
    LVO_TRY(check_view(c, sweeps[l], (size_t)c->P, true));
    if (sweeps[l].stride != sweeps[first].stride || sweeps[l].off_xyz != sweeps[first].off_xyz) { lvo_set_error(c, "all lanes must share one point layout"); return LVO_E_BADARG; }
    if (sweeps[l].stride > 32) { lvo_set_error(c, "stride > 32 unsupported in lvo_step_batch"); return LVO_E_BADARG; }
    *max_n = std::max(*max_n, (int)sweeps[l].n);
  }
  if (first >= 0) { *stride = (int)sweeps[first].stride; *off_xyz = (int)sweeps[first].off_xyz; }
  else if (c->graph_stride >= 0) { *stride = c->graph_stride; *off_xyz = c->graph_off; }
  else { *stride = 16; *off_xyz = 0; }
  return LVO_OK;
}

int lvo_step_batch_async(lvo_ctx* c, const lvo_cloud_view* sweeps) {
  LVO_ENTER(c);
  if (!sweeps) return LVO_E_BADARG;
  int max_n = 0, stride = 0, off_xyz = 0;
  LVO_TRY(check_sweeps(c, sweeps, &max_n, &stride, &off_xyz));
  LVO_TRY(stage_sweeps(c, sweeps, c->d_raw, c->st));
  return step_enqueue(c, stride, off_xyz, max_n);
}
int lvo_wait(lvo_ctx* c, lvo_pose* T_wodom, lvo_pose* T_wmap) {
  LvoDeviceGuard _dev(c);
  if (!c) return LVO_E_BADARG;
  return step_finish(c, T_wodom, T_wmap);
}
int lvo_step_batch(lvo_ctx* c, const lvo_cloud_view* sweeps, lvo_pose* T_wodom, lvo_pose* T_wmap) {
  LVO_ENTER(c);
  LVO_TRY(lvo_step_batch_async(c, sweeps));
  return step_finish(c, T_wodom, T_wmap);
}

int lvo_step_batch_pipelined(lvo_ctx* c, const lvo_cloud_view* sweeps, const lvo_cloud_view* next, lvo_pose* T_wodom, lvo_pose* T_wmap) {
  LVO_ENTER(c);
  if (!sweeps) return LVO_E_BADARG;
  if (!c->copy_st) {
    LVO_CUDA_OK(c, cudaStreamCreateWithFlags(&c->copy_st, cudaStreamNonBlocking));
    LVO_CUDA_OK(c, cudaEventCreateWithFlags(&c->copy_ev, cudaEventDisableTiming));
    LVO_CUDA_OK(c, cudaEventCreateWithFlags(&c->compute_ev, cudaEventDisableTiming));
    LVO_TRY(dalloc(c, &c->d_raw2, c->raw_lane_bytes * c->lanes, false));
  }
  int max_n = 0, max_next = 0, stride = 0, off_xyz = 0, nstride = 0, noff = 0;
  LVO_TRY(check_sweeps(c, sweeps, &max_n, &stride, &off_xyz));
  if (next) LVO_TRY(check_sweeps(c, next, &max_next, &nstride, &noff));
  // a hit needs the prefetch to have been staged for the same active set, with the same views of the active lanes
  bool hit = (int)c->prefetched.size() == c->lanes && c->prefetched_active == c->lane_active;
  for (int l = 0; hit && l < c->lanes; ++l)
    hit = !c->lane_active[l] || (c->prefetched[l].data == sweeps[l].data && c->prefetched[l].n == sweeps[l].n && c->prefetched[l].stride == sweeps[l].stride);
  unsigned char* bufs[2] = {c->d_raw, c->d_raw2};
  if (hit) {
    c->raw_cur ^= 1;                                         // the prefetched buffer becomes current
    LVO_CUDA_OK(c, cudaStreamWaitEvent(c->st, c->copy_ev, 0));
    for (int l = 0; l < c->lanes; ++l) { c->h_in_ptr[l] = c->next_in_ptr[l]; c->h_in_n[l] = c->lane_active[l] ? (int)sweeps[l].n : 0; }
  } else {
    LVO_TRY(stage_sweeps(c, sweeps, bufs[c->raw_cur], c->st));
  }
  c->prefetched.clear();
  c->pending_next = next;
  int r = step_enqueue(c, stride, off_xyz, max_n);
  c->pending_next = nullptr;  // an early error return must not leave a pointer for a later call
  if (r != LVO_OK) return r;
  return step_finish(c, T_wodom, T_wmap);
}

int lvo_step_batch_dev_async(lvo_ctx* c, const lvo_point* const* d_sweeps, const size_t* n) {
  LVO_ENTER(c);
  if (!d_sweeps || !n) return LVO_E_BADARG;
  int max_n = 0;
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l]) { c->h_in_ptr[l] = c->d_raw; c->h_in_n[l] = 0; continue; }   // d_sweeps[l] / n[l] not read
    if (n[l] > (size_t)c->P) { lvo_set_error(c, "input cloud exceeds context capacity"); return LVO_E_CAPACITY; }
    c->h_in_ptr[l] = (const unsigned char*)d_sweeps[l]; c->h_in_n[l] = (int)n[l];
    max_n = std::max(max_n, (int)n[l]);
  }
  return step_enqueue(c, 16, 0, max_n);
}
int lvo_step_batch_dev(lvo_ctx* c, const lvo_point* const* d_sweeps, const size_t* n, lvo_pose* T_wodom, lvo_pose* T_wmap) {
  LVO_ENTER(c);
  LVO_TRY(lvo_step_batch_dev_async(c, d_sweeps, n));
  return step_finish(c, T_wodom, T_wmap);
}

// ---- per-lane lifecycle: the flags are data of the next step (set_inputs), so captured graphs stay valid
int lvo_set_lane_active(lvo_ctx* c, int lane, int active) {
  LVO_ENTER_LANE(c, lane);
  c->lane_active[lane] = active ? 1 : 0;
  return LVO_OK;
}
int lvo_set_lane_map_update(lvo_ctx* c, int lane, int update) {
  LVO_ENTER_LANE(c, lane);
  c->lane_map_update[lane] = update ? 1 : 0;
  return LVO_OK;
}

}  // extern "C"
// lvo_lane_reset, and lvo_lane_configure with cfg != NULL: the lane starts a new sequence (with the given settings)
static int reset_lane(lvo_ctx* c, int lane, const lvo_lane_config* cfg) {
  // the lane's device state as lvo_create leaves it: zeroed LaneState + k_init_lanes, an empty map in both generations (the points
  // behind an empty offset table are never read; the odometry "last" clouds are not read before the first frame replaces them)
  LVO_CUDA_OK(c, cudaMemsetAsync(c->d_ls + lane, 0, sizeof(LaneState), c->st));
  for (int g = 0; g < 2; ++g)
    for (int t = 0; t < 2; ++t)
      LVO_CUDA_OK(c, cudaMemsetAsync(c->map.cube_start[g][t] + (size_t)lane * (LVO_NCUBES + 1), 0, sizeof(unsigned) * (LVO_NCUBES + 1), c->st));
  k_init_lanes<<<1, 64, 0, c->st>>>(c->d_ls, lane, 1);
  LVO_CUDA_OK(c, cudaMemsetAsync(c->d_unc + 2 * (size_t)lane, 0, 2 * sizeof(LvoUncRaw), c->st));   // both pose-uncertainty records
  if (cfg) { c->lane_cfg[lane] = *cfg; LVO_TRY(upload_lane_config(c, lane)); }
  // and its host copies, so that lvo_get_stats / lvo_lane_status report the new sequence at once
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->h_ls + lane, c->d_ls + lane, sizeof(LaneState), cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  c->lane_status[lane] = LVO_OK;
  c->lane_frame[lane] = 0;
  c->probe_gate[lane] = 0;   // zero counts: every probe is empty, and in bounds
  c->reg_n[lane] = 0;
  c->unc_frame[2 * lane] = c->unc_frame[2 * lane + 1] = -1;
  c->unc_epoch++;
  return LVO_OK;
}
extern "C" {

int lvo_lane_reset(lvo_ctx* c, int lane) {
  LVO_ENTER_LANE(c, lane);
  return reset_lane(c, lane, nullptr);
}

int lvo_lane_configure(lvo_ctx* c, int lane, const lvo_lane_config* cfg) {
  LVO_ENTER_LANE(c, lane);
  const lvo_lane_config lc = cfg ? *cfg : lvo_lane_config{c->cfg.n_scans, c->cfg.minimum_range, c->cfg.line_res, c->cfg.plane_res, c->cfg.skip_frame};
  auto bad = [&](const char* what) { lvo_set_error(c, std::string("lvo_lane_config::") + what); return LVO_E_BADARG; };
  if (lc.n_scans != 16 && lc.n_scans != 32 && lc.n_scans != 64) return bad("n_scans must be 16, 32 or 64");   // scanRegistration.cpp:203
  if (lc.n_scans > c->cfg.n_scans) {
    lvo_set_error(c, "lvo_lane_config::n_scans " + std::to_string(lc.n_scans) + " exceeds the context's n_scans " + std::to_string(c->cfg.n_scans) +
                     ", which sizes the feature buffers and per-ring tables of every lane");
    return LVO_E_CAPACITY;
  }
  // the kernels see the values as float: check them as float too (a double that rounds to 0 or overflows is refused)
  const float range = (float)lc.minimum_range, line = (float)lc.line_res, plane = (float)lc.plane_res;
  if (!(std::isfinite(range) && range >= 0.f)) return bad("minimum_range must be finite and >= 0");
  if (!(std::isfinite(line) && line > 0.f)) return bad("line_res must be finite and > 0");
  if (!(std::isfinite(plane) && plane > 0.f)) return bad("plane_res must be finite and > 0");
  if (lc.skip_frame < 1) return bad("skip_frame must be >= 1");
  return reset_lane(c, lane, &lc);
}

int lvo_lane_get_config(const lvo_ctx* c, int lane, lvo_lane_config* out) {
  LVO_ENTER_LANE(c, lane);
  if (!out) return LVO_E_BADARG;
  *out = c->lane_cfg[lane];
  return LVO_OK;
}

// ---- lane snapshots (DESIGN §3 "Lane snapshot"): header | LaneState | cube_start corner | cube_start surf | corner_last | surf_last |
// map corner | map surf.  Everything before the point sections has a fixed size, so that a load can check it on the host first.
}  // extern "C"
namespace {
#define LVO_SNAP_VERSION 1u
static const char kSnapMagic[8] = {'L', 'V', 'O', 'L', 'A', 'N', 'E', '\0'};
struct LvoSnapHeader {
  char magic[8];
  uint32_t version, header_bytes, state_bytes, cube_entries;   // LVO_SNAP_VERSION, 128, sizeof(LaneState), LVO_NCUBES + 1
  uint64_t total_bytes;
  // every lvo_config field that changes results
  int32_t n_scans, skip_frame, outer_iters, lm_max_iters, distortion, reserved0;
  double minimum_range, line_res, plane_res, huber;
  // host-side lane data
  int64_t lane_frame;   // frames since the sequence started (its skip_frame phase)
  int32_t lane_status;
  uint32_t n_corner_last, n_surf_last, n_map[2];   // points in the four point sections
  uint8_t reserved1[12];
};
static_assert(sizeof(LvoSnapHeader) == 128, "lane snapshot header layout");
const size_t kSnapCubeBytes = sizeof(unsigned) * (LVO_NCUBES + 1);
const size_t kSnapPrefix = sizeof(LvoSnapHeader) + sizeof(LaneState) + 2 * kSnapCubeBytes;   // a multiple of 16: the points stay aligned
static_assert(kSnapPrefix % 16 == 0, "lane snapshot sections");
// LaneState::cen: cube_coord adds it to int((v + 25) / 50), and k_map_begin walks the centre cube back into the window one step at a
// time; a running lane keeps it near the cube of the world origin (50 m cubes: 2^20 of them span 52 000 km).  The poses bound v:
// every translation within 1e7 m and every quaternion component within [-2, 2] keep the map position that k_map_begin composes
// below 3e8 m, so the cube coordinate plus cen stays far from int overflow and the walk is finite.
#define LVO_SNAP_CEN_LIMIT (1 << 20)
#define LVO_SNAP_T_LIMIT 1.0e7
#define LVO_SNAP_Q_LIMIT 2.0

uint64_t snap_total(const LvoSnapHeader& h) {
  return kSnapPrefix + 16ull * ((uint64_t)h.n_corner_last + h.n_surf_last + h.n_map[0] + h.n_map[1]);
}
int snap_bad(lvo_ctx* c, const std::string& what) { lvo_set_error(c, "lane snapshot rejected: " + what); return LVO_E_BADARG; }
int snap_cap(lvo_ctx* c, const std::string& what) { lvo_set_error(c, "lane snapshot does not fit this context: " + what); return LVO_E_CAPACITY; }
// a (q, t) pair of doubles in LaneState: finite and inside the limits above
bool pose_ok(const double* q, const double* t) {
  for (int k = 0; k < 4; ++k) if (!std::isfinite(q[k]) || std::fabs(q[k]) > LVO_SNAP_Q_LIMIT) return false;
  for (int k = 0; k < 3; ++k) if (!std::isfinite(t[k]) || std::fabs(t[k]) > LVO_SNAP_T_LIMIT) return false;
  return true;
}
bool monotone(const int* v, int n, int lo, int hi) {   // lo <= v[0] <= ... <= v[n - 1] <= hi
  int prev = lo;
  for (int i = 0; i < n; ++i) { if (v[i] < prev || v[i] > hi) return false; prev = v[i]; }
  return true;
}
// the lane's sensor settings (lvo_lane_config) and the context's solver settings
void snap_fingerprint(const lvo_ctx* c, int lane, LvoSnapHeader& h) {
  const lvo_config& cfg = c->cfg; const lvo_lane_config& lc = c->lane_cfg[lane];
  h.n_scans = lc.n_scans; h.skip_frame = lc.skip_frame; h.outer_iters = cfg.outer_iters; h.lm_max_iters = cfg.lm_max_iters;
  h.distortion = cfg.distortion; h.minimum_range = lc.minimum_range; h.line_res = lc.line_res; h.plane_res = lc.plane_res; h.huber = cfg.huber;
}
// Every field of the fixed part that a kernel or an entry point later uses as an index, a loop bound or a size, checked against the
// destination lane and its context before anything is written.  `cs` = the two cube_start tables.
int snap_check(lvo_ctx* c, int lane, const LvoSnapHeader& h, const LaneState& s, const unsigned* const cs[2], size_t n_bytes) {
  if (memcmp(h.magic, kSnapMagic, sizeof(kSnapMagic)) != 0) return snap_bad(c, "not a lane snapshot (magic)");
  if (h.version != LVO_SNAP_VERSION) return snap_bad(c, "format version " + std::to_string(h.version) + ", this library reads " + std::to_string(LVO_SNAP_VERSION));
  if (h.header_bytes != sizeof(LvoSnapHeader) || h.state_bytes != sizeof(LaneState) || h.cube_entries != LVO_NCUBES + 1)
    return snap_bad(c, "header / LaneState / cube table size differs from this library's");
  if (h.total_bytes != snap_total(h) || n_bytes != h.total_bytes)
    return snap_bad(c, "byte length " + std::to_string(n_bytes) + ", the header describes " + std::to_string(snap_total(h)));
  LvoSnapHeader mine; memset(&mine, 0, sizeof(mine));
  snap_fingerprint(c, lane, mine);
#define LVO_SNAP_FIELD(f, owner) if (!(h.f == mine.f)) return snap_bad(c, #f " differs from the " owner);
  LVO_SNAP_FIELD(n_scans, "lane's (lvo_lane_config)") LVO_SNAP_FIELD(minimum_range, "lane's (lvo_lane_config)")
  LVO_SNAP_FIELD(line_res, "lane's (lvo_lane_config)") LVO_SNAP_FIELD(plane_res, "lane's (lvo_lane_config)")
  LVO_SNAP_FIELD(skip_frame, "lane's (lvo_lane_config)") LVO_SNAP_FIELD(outer_iters, "context's (lvo_config)")
  LVO_SNAP_FIELD(lm_max_iters, "context's (lvo_config)") LVO_SNAP_FIELD(huber, "context's (lvo_config)") LVO_SNAP_FIELD(distortion, "context's (lvo_config)")
#undef LVO_SNAP_FIELD
  const FeatureCaps fc = feature_caps(h.n_scans);   // the lane's n_scans
  if (h.lane_frame < 0) return snap_bad(c, "lane_frame < 0");
  // odometry: the "last" clouds and their ring-offset tables
  if ((int64_t)s.n_corner_last != h.n_corner_last || (int64_t)s.n_surf_last != h.n_surf_last) return snap_bad(c, "n_corner_last / n_surf_last disagree with the header");
  if (s.n_corner_last > fc.lsharp) return snap_bad(c, "n_corner_last exceeds the less-sharp capacity of n_scans");
  if (!monotone(s.corner_ring_first, LVO_MAX_RINGS + 2, 0, s.n_corner_last)) return snap_bad(c, "corner_ring_first");
  if (!monotone(s.surf_ring_first, LVO_MAX_RINGS + 2, 0, s.n_surf_last)) return snap_bad(c, "surf_ring_first");
  // poses: the odometry pose and its increment, the mapping pose, the map correction, the odometry pose the mapping stage last read
  if (!pose_ok(s.para_q, s.para_t) || !pose_ok(s.q_w, s.t_w) || !pose_ok(s.map_x, s.map_x + 4) || !pose_ok(s.q_wmap_wodom, s.t_wmap_wodom) ||
      !pose_ok(s.q_wodom, s.t_wodom))
    return snap_bad(c, "a pose is not finite or out of range (|t| <= 1e7 m, |q_i| <= 2)");
  // the counts of the source lane's last frame.  A batched step rewrites them before reading them, but lvo_scan_to_scan /
  // lvo_scan_to_map run their stage for every lane of the context from its stored counts: n_sharp, n_flat, n_less_sharp, n_less_flat
  // and n_kept bound the odometry kernels (association, k_odo_to_end, the swap into the "last" clouds), n_less_* and n_kept the stack
  // gather and the registered cloud of the mapping stage, n_stack the mapping association and solve.  Bounds that depend on the lane's
  // n_scans alone cannot be exceeded by a snapshot of a matching lane (LVO_E_BADARG); those set by max_points can (LVO_E_CAPACITY).  So
  // a lane accepts or refuses a snapshot as lane 0 of a context created with its settings and the same capacities does.
  const struct { int n; int cap; bool cap_is_P; const char* name; } counts[] = {
      {s.n_sharp, fc.sharp, false, "n_sharp"}, {s.n_less_sharp, fc.lsharp, false, "n_less_sharp"}, {s.n_flat, fc.flat, false, "n_flat"},
      {s.n_stack[0], fc.lsharp, false, "n_stack[0]"}, {s.n_kept, c->P, true, "n_kept"}, {s.n_less_flat, c->P, true, "n_less_flat"},
      {s.n_stack[1], c->map.in_cap[1], true, "n_stack[1]"}};
  for (const auto& k : counts) {
    if (k.n < 0) return snap_bad(c, std::string(k.name) + " < 0");
    if (k.n > k.cap && !k.cap_is_P) return snap_bad(c, std::string(k.name) + " exceeds its capacity for n_scans");
  }
  // mapping: cube window, valid list, FromMap offsets
  const int dims[3] = {LVO_CUBE_W, LVO_CUBE_H, LVO_CUBE_D};
  for (int k = 0; k < 3; ++k) {
    if (s.cen[k] < -LVO_SNAP_CEN_LIMIT || s.cen[k] > LVO_SNAP_CEN_LIMIT) return snap_bad(c, "cen out of range");
    if (s.center[k] < 0 || s.center[k] >= dims[k]) return snap_bad(c, "center out of range");
    if (s.shift[k] != 0) return snap_bad(c, "shift != 0 (k_map_end clears it after every mapping stage)");
  }
  if (s.n_valid < 0 || s.n_valid > LVO_MAX_VALID) return snap_bad(c, "n_valid out of range");
  for (int v = 0; v < s.n_valid; ++v) if (s.valid_cube[v] < 0 || s.valid_cube[v] >= LVO_NCUBES) return snap_bad(c, "valid_cube out of range");
  for (int t = 0; t < 2; ++t) {
    if (s.from_off[t][0] != 0 || !monotone(s.from_off[t], LVO_MAX_VALID + 1, 0, INT_MAX)) return snap_bad(c, "from_off");
    if (cs[t][0] != 0) return snap_bad(c, "cube_start does not start at 0");
    for (int k = 0; k < LVO_NCUBES; ++k) if (cs[t][k + 1] < cs[t][k]) return snap_bad(c, "cube_start decreases");
    if (cs[t][LVO_NCUBES] != h.n_map[t]) return snap_bad(c, "cube_start ends at a count other than the header's");
  }
  // capacities: may differ from the source context's as long as the saved counts fit
  if (s.n_surf_last > c->P) return snap_cap(c, "n_surf_last " + std::to_string(s.n_surf_last) + " > max_points " + std::to_string(c->P));
  for (const auto& k : counts)
    if (k.n > k.cap) return snap_cap(c, std::string(k.name) + " " + std::to_string(k.n) + " > max_points " + std::to_string(c->P));
  for (int t = 0; t < 2; ++t) {
    const char* nm = t ? "max_map_surf" : "max_map_corner";
    if (h.n_map[t] > (uint32_t)c->map.map_cap[t]) return snap_cap(c, std::to_string(h.n_map[t]) + " map points > " + nm + " " + std::to_string(c->map.map_cap[t]));
    // the mapping grid build of a step in which the lane does not map still reads FromMap up to from_off[t][LVO_MAX_VALID]
    if (s.from_off[t][LVO_MAX_VALID] > c->map.map_cap[t]) return snap_cap(c, std::string("FromMap count > ") + nm);
  }
  return LVO_OK;
}
}  // namespace
extern "C" {

int lvo_lane_save(lvo_ctx* c, int lane, void* dst, size_t cap, size_t* n_bytes) {
  LVO_ENTER_LANE(c, lane);
  // the fixed part is assembled on the host (the device holds no header); the points go straight from the arenas to dst
  std::vector<unsigned char> pre(kSnapPrefix, 0);
  LvoSnapHeader& h = *reinterpret_cast<LvoSnapHeader*>(pre.data());
  LaneState& s = *reinterpret_cast<LaneState*>(pre.data() + sizeof(LvoSnapHeader));
  unsigned* cs[2] = {reinterpret_cast<unsigned*>(pre.data() + sizeof(LvoSnapHeader) + sizeof(LaneState)), nullptr};
  cs[1] = cs[0] + (LVO_NCUBES + 1);
  const int gen = c->map.gen;
  LVO_CUDA_OK(c, cudaMemcpyAsync(&s, c->d_ls + lane, sizeof(LaneState), cudaMemcpyDeviceToHost, c->st));
  for (int t = 0; t < 2; ++t)
    LVO_CUDA_OK(c, cudaMemcpyAsync(cs[t], c->map.cube_start[gen][t] + (size_t)lane * (LVO_NCUBES + 1), kSnapCubeBytes, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  memcpy(h.magic, kSnapMagic, sizeof(kSnapMagic));
  h.version = LVO_SNAP_VERSION; h.header_bytes = sizeof(LvoSnapHeader); h.state_bytes = sizeof(LaneState); h.cube_entries = LVO_NCUBES + 1;
  snap_fingerprint(c, lane, h);
  h.lane_frame = c->lane_frame[lane]; h.lane_status = c->lane_status[lane];
  h.n_corner_last = (uint32_t)s.n_corner_last; h.n_surf_last = (uint32_t)s.n_surf_last;
  h.n_map[0] = cs[0][LVO_NCUBES]; h.n_map[1] = cs[1][LVO_NCUBES];
  h.total_bytes = snap_total(h);
  if (n_bytes) *n_bytes = (size_t)h.total_bytes;
  if (!dst || cap < h.total_bytes) { lvo_set_error(c, "snapshot buffer too small"); return LVO_E_CAPACITY; }
  // host or device memory of any device: UVA resolves the direction
  unsigned char* out = (unsigned char*)dst;
  LVO_CUDA_OK(c, cudaMemcpyAsync(out, pre.data(), kSnapPrefix, cudaMemcpyDefault, c->st));
  size_t off = kSnapPrefix;
  const float4* src[4] = {c->odo.corner_last + (size_t)lane * c->cap_lsharp, c->odo.surf_last + (size_t)lane * c->P,
                          c->map.map_pts[gen][0] + (size_t)lane * c->map.map_cap[0], c->map.map_pts[gen][1] + (size_t)lane * c->map.map_cap[1]};
  const size_t cnt[4] = {h.n_corner_last, h.n_surf_last, h.n_map[0], h.n_map[1]};
  for (int k = 0; k < 4; ++k) {
    if (cnt[k]) LVO_CUDA_OK(c, cudaMemcpyAsync(out + off, src[k], cnt[k] * sizeof(float4), cudaMemcpyDefault, c->st));
    off += cnt[k] * sizeof(float4);
  }
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));   // `pre` dies on return
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

int lvo_lane_load(lvo_ctx* c, int lane, const void* src, size_t n_bytes) {
  LVO_ENTER_LANE(c, lane);
  if (!src) return snap_bad(c, "null buffer");
  if (n_bytes < kSnapPrefix) return snap_bad(c, "truncated: " + std::to_string(n_bytes) + " bytes");
  // the fixed part comes to the host to be checked (from device memory too); nothing is written before every check has passed
  std::vector<unsigned char> pre(kSnapPrefix);
  LVO_CUDA_OK(c, cudaMemcpyAsync(pre.data(), src, kSnapPrefix, cudaMemcpyDefault, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LvoSnapHeader h; LaneState s;
  memcpy(&h, pre.data(), sizeof(h));
  memcpy(&s, pre.data() + sizeof(h), sizeof(s));
  const unsigned* cs[2] = {reinterpret_cast<const unsigned*>(pre.data() + sizeof(h) + sizeof(s)), nullptr};
  cs[1] = cs[0] + (LVO_NCUBES + 1);
  LVO_TRY(snap_check(c, lane, h, s, cs, n_bytes));
  // into the current map generation; the other one is rewritten by the next mapping stage before anything reads it
  const int gen = c->map.gen;
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_ls + lane, &s, sizeof(LaneState), cudaMemcpyHostToDevice, c->st));
  for (int t = 0; t < 2; ++t)
    LVO_CUDA_OK(c, cudaMemcpyAsync(c->map.cube_start[gen][t] + (size_t)lane * (LVO_NCUBES + 1), cs[t], kSnapCubeBytes, cudaMemcpyHostToDevice, c->st));
  float4* dst[4] = {c->odo.corner_last + (size_t)lane * c->cap_lsharp, c->odo.surf_last + (size_t)lane * c->P,
                    c->map.map_pts[gen][0] + (size_t)lane * c->map.map_cap[0], c->map.map_pts[gen][1] + (size_t)lane * c->map.map_cap[1]};
  const size_t cnt[4] = {h.n_corner_last, h.n_surf_last, h.n_map[0], h.n_map[1]};
  size_t off = kSnapPrefix;
  for (int k = 0; k < 4; ++k) {
    if (cnt[k]) LVO_CUDA_OK(c, cudaMemcpyAsync(dst[k], (const unsigned char*)src + off, cnt[k] * sizeof(float4), cudaMemcpyDefault, c->st));
    off += cnt[k] * sizeof(float4);
  }
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  c->h_ls[lane] = s;   // lvo_get_stats / lvo_get_map_correction / lvo_map_* see the snapshot at once
  c->lane_frame[lane] = h.lane_frame;
  c->lane_status[lane] = h.lane_status;
  c->probe_gate[lane] = LVO_PROBE_GATE_EXTRACT | LVO_PROBE_GATE_ODO | LVO_PROBE_GATE_MAP;
  c->odo_grids_stale = true;
  c->reg_n[lane] = 0;
  c->unc_frame[2 * lane] = c->unc_frame[2 * lane + 1] = -1;   // gated until the stage runs (probe_gate)
  c->unc_epoch++;
  return LVO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
int lvo_map_import(lvo_ctx* c, int lane, const lvo_point* corner, const int* corner_cube, size_t n_corner, const lvo_point* surf, const int* surf_cube,
                   size_t n_surf) {
  LVO_ENTER_LANE(c, lane);
  const lvo_point* pts[2] = {corner, surf}; const int* cubes[2] = {corner_cube, surf_cube}; const size_t ns[2] = {n_corner, n_surf};
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  for (int t = 0; t < 2; ++t) {
    if (ns[t] > (size_t)c->map.map_cap[t]) { lvo_set_error(c, "map import exceeds capacity"); return LVO_E_CAPACITY; }
    if (ns[t] && (!pts[t] || !cubes[t])) return LVO_E_BADARG;
    std::vector<unsigned> start(LVO_NCUBES + 1, 0);
    for (size_t i = 0; i < ns[t]; ++i) { if (cubes[t][i] < 0 || cubes[t][i] >= LVO_NCUBES) return LVO_E_BADARG; start[cubes[t][i] + 1]++; }
    for (int k = 0; k < LVO_NCUBES; ++k) start[k + 1] += start[k];
    std::vector<lvo_point> sorted(ns[t]);
    std::vector<unsigned> cur(start.begin(), start.end() - 1);
    for (size_t i = 0; i < ns[t]; ++i) sorted[cur[cubes[t][i]]++] = pts[t][i];  // stable inside a cube
    if (ns[t]) LVO_CUDA_OK(c, cudaMemcpyAsync(c->map.map_pts[c->map.gen][t] + (size_t)lane * c->map.map_cap[t], sorted.data(), ns[t] * sizeof(lvo_point), cudaMemcpyHostToDevice, c->st));
    LVO_CUDA_OK(c, cudaMemcpyAsync(c->map.cube_start[c->map.gen][t] + (size_t)lane * (LVO_NCUBES + 1), start.data(), sizeof(unsigned) * (LVO_NCUBES + 1), cudaMemcpyHostToDevice, c->st));
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));   // `sorted` / `start` die at the end of this iteration
  }
  SetCounts sc; memset(&sc, 0, sizeof(sc));
  sc.what = 5; sc.v[0] = (int)n_corner; sc.v[1] = (int)n_surf;
  k_set_lane<<<1, 1, 0, c->st>>>(c->d_ls, lane, sc);
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  return LVO_OK;
}

int lvo_map_export(lvo_ctx* c, int lane, int which, lvo_cloud_out* pts, int* cube_out) {
  LVO_ENTER_LANE(c, lane);
  if (which < 0 || which > 1 || !pts) return LVO_E_BADARG;
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  std::vector<unsigned> start(LVO_NCUBES + 1);
  LVO_CUDA_OK(c, cudaMemcpyAsync(start.data(), c->map.cube_start[c->map.gen][which] + (size_t)lane * (LVO_NCUBES + 1), sizeof(unsigned) * (LVO_NCUBES + 1), cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  const size_t n = start[LVO_NCUBES];
  pts->n = n;
  if (n > pts->cap) return LVO_E_CAPACITY;
  if (n) {
    LVO_CUDA_OK(c, cudaMemcpyAsync(pts->data, c->map.map_pts[c->map.gen][which] + (size_t)lane * c->map.map_cap[which], n * sizeof(lvo_point), cudaMemcpyDeviceToHost, c->st));
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  }
  if (cube_out) for (int k = 0; k < LVO_NCUBES; ++k) for (unsigned i = start[k]; i < start[k + 1]; ++i) cube_out[i] = k;
  return LVO_OK;
}

// ---- map outputs (DESIGN §3 "Map-output arena"): one launch sequence for any number of lanes, slot s = lane first_lane + s
// The per-slot part, allocated on the first call for every lane of the context (d_desc last: it marks the part as complete).
static int mapout_reserve_slots(lvo_ctx* c) {
  lvo_ctx::MapOutArena& m = c->mapout;
  if (m.d_desc) return LVO_OK;
  const size_t L = (size_t)c->lanes;
  int r = m.mem.device(c, &m.off, L * LVO_MAPOUT_STRIDE * sizeof(unsigned));
  if (r == LVO_OK) r = m.mem.device(c, &m.d_tot, L * sizeof(unsigned));
  if (r == LVO_OK) r = m.mem.pinned(c, &m.h_desc, L * sizeof(MapOutDesc));
  if (r == LVO_OK) r = m.mem.pinned(c, &m.h_tot, L * sizeof(unsigned));
  if (r == LVO_OK) r = m.mem.device(c, &m.d_desc, L * sizeof(MapOutDesc));
  if (r != LVO_OK) m.mem.release();
  return r;
}
// The host form's point buffer, grown to `pts`.  Every call ends synchronised, so the old buffer can be freed at once.
static int mapout_reserve_points(lvo_ctx* c, size_t pts) {
  lvo_ctx::MapOutArena& m = c->mapout;
  LVO_TRY(mapout_reserve_slots(c));
  if (m.d_pts && pts <= m.cap_pts) return LVO_OK;
  pts = std::max<size_t>({pts, m.cap_pts + m.cap_pts / 2, 1024});   // a growing map does not reallocate on every call
  m.pts_mem.release();
  m.cap_pts = 0;
  LVO_TRY(m.pts_mem.device(c, &m.d_pts, pts * sizeof(float4)));
  m.cap_pts = pts;
  return LVO_OK;
}

static MapOutArgs mapout_args(const lvo_ctx* c, int which, int first_lane) {
  MapOutArgs a;
  memset(&a, 0, sizeof(a));
  a.ls = c->d_ls;
  for (int t = 0; t < 2; ++t) { a.cube_start[t] = c->map.cube_start[c->map.gen][t]; a.map_pts[t] = c->map.map_pts[c->map.gen][t]; a.map_cap[t] = c->map.map_cap[t]; }
  a.first_lane = first_lane;
  a.surround = which == LVO_MAP_SURROUND;
  return a;
}

// which 0 / 1: the cloud sizes of S slots (one launch and the call's only synchronisation)
static int mapout_count(lvo_ctx* c, const MapOutArgs& a, int S, size_t* n) {
  lvo_ctx::MapOutArena& m = c->mapout;
  k_mapout_offsets<<<S, 256, 0, c->st>>>(a, m.off, m.d_tot);
  c->launches++;
  LVO_CUDA_OK(c, cudaMemcpyAsync(m.h_tot, m.d_tot, sizeof(unsigned) * S, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  for (int s = 0; s < S; ++s) n[s] = m.h_tot[s];
  return LVO_OK;
}

// Uploads the descriptors staged in h_desc[0, S) and enqueues the copy kernel (not synchronised).
static int mapout_copy(lvo_ctx* c, int which, const MapOutArgs& a, int S) {
  lvo_ctx::MapOutArena& m = c->mapout;
  LVO_CUDA_OK(c, cudaMemcpyAsync(m.d_desc, m.h_desc, sizeof(MapOutDesc) * S, cudaMemcpyHostToDevice, c->st));
  if (which == LVO_MAP_REGISTERED) k_mapout_registered<<<dim3(64, S), 256, 0, c->st>>>(c->map.registered, c->P, m.d_desc);
  else k_mapout_copy<<<dim3(which == LVO_MAP_SURROUND ? LVO_MAX_VALID : 296, S), 256, 0, c->st>>>(a, m.d_desc, m.off);
  c->launches++;
  return LVO_OK;
}

// Host form: the selected slots' clouds (dst[s] != NULL) are gathered back to back into the arena, and each goes to the caller's
// buffer in one cudaMemcpyAsync.  profiles/map_outputs.md compares this with one packed download into pinned memory followed by a
// host scatter.
static int mapout_host(lvo_ctx* c, int which, const MapOutArgs& a, int S, const size_t* n, lvo_point* const* dst) {
  lvo_ctx::MapOutArena& m = c->mapout;
  size_t total = 0; bool any = false;
  for (int s = 0; s < S; ++s) if (dst[s]) { total += n[s]; any = true; }
  if (!any) return LVO_OK;
  LVO_TRY(mapout_reserve_points(c, total));
  size_t o = 0;
  for (int s = 0; s < S; ++s) {
    m.h_desc[s] = MapOutDesc{dst[s] ? m.d_pts + o : nullptr, (unsigned)n[s], 0u};
    if (dst[s]) o += n[s];
  }
  LVO_TRY(mapout_copy(c, which, a, S));
  o = 0;
  for (int s = 0; s < S; ++s) {
    if (!dst[s]) continue;
    if (n[s]) LVO_CUDA_OK(c, cudaMemcpyAsync(dst[s], m.d_pts + o, n[s] * sizeof(float4), cudaMemcpyDeviceToHost, c->st));
    o += n[s];
  }
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

// Checks shared by the batch forms; n[l] gets every lane's count.  Nothing is written to a destination before it returns.
static int mapout_batch_begin(lvo_ctx* c, int which, size_t* n, MapOutArgs* a) {
  if (which < LVO_MAP_SURROUND || which > LVO_MAP_REGISTERED) { lvo_set_error(c, "bad `which`: LVO_MAP_SURROUND, LVO_MAP_WHOLE or LVO_MAP_REGISTERED"); return LVO_E_BADARG; }
  if (which == LVO_MAP_REGISTERED && !c->reg_valid) {
    lvo_set_error(c, "the registered clouds were overwritten by lvo_scan_to_map or lvo_knn; the next lvo_step_batch* call makes them available again");
    return LVO_E_STATE;
  }
  c->launches = 0;
  *a = mapout_args(c, which, 0);
  if (which == LVO_MAP_REGISTERED) { for (int l = 0; l < c->lanes; ++l) n[l] = c->reg_n[l]; return LVO_OK; }
  LVO_TRY(mapout_reserve_slots(c));
  return mapout_count(c, *a, c->lanes, n);
}

static int map_cloud_one(lvo_ctx* c, int lane, int which, lvo_cloud_out* pts) {
  LVO_TRY(mapout_reserve_slots(c));
  const MapOutArgs a = mapout_args(c, which, lane);
  size_t n = 0;
  LVO_TRY(mapout_count(c, a, 1, &n));
  pts->n = n;
  if (n > pts->cap || (n && !pts->data)) { lvo_set_error(c, "output cloud buffer too small"); return LVO_E_CAPACITY; }
  lvo_point* dst = pts->data;
  return mapout_host(c, which, a, 1, &n, &dst);
}
int lvo_map_cloud(lvo_ctx* c, int lane, int which, lvo_cloud_out* pts) {
  LVO_ENTER_LANE(c, lane);
  if (which < 0 || which > 1 || !pts) return LVO_E_BADARG;
  const long long launches = c->launches;   // lvo_timings::kernel_launches keeps reporting the last step / stage call
  const int r = map_cloud_one(c, lane, which, pts);
  c->launches = launches;
  return r;
}

int lvo_map_cloud_batch(lvo_ctx* c, int which, lvo_cloud_out* outs) {
  LVO_ENTER(c);
  if (!outs) { lvo_set_error(c, "NULL array"); return LVO_E_BADARG; }
  const int L = c->lanes;
  std::vector<size_t> n(L);
  MapOutArgs a;
  LVO_TRY(mapout_batch_begin(c, which, n.data(), &a));
  std::vector<lvo_point*> dst(L);
  int short_lane = -1;
  for (int l = 0; l < L; ++l) {
    outs[l].n = n[l];
    dst[l] = outs[l].data;
    if (dst[l] && outs[l].cap < n[l] && short_lane < 0) short_lane = l;
  }
  if (short_lane >= 0) { lvo_set_error(c, "output buffer of lane " + std::to_string(short_lane) + " too small"); return LVO_E_CAPACITY; }
  return mapout_host(c, which, a, L, n.data(), dst.data());
}

int lvo_map_cloud_batch_dev(lvo_ctx* c, int which, lvo_point* const* d_out, const size_t* cap, size_t* n_out) {
  LVO_ENTER(c);
  if (!d_out || !cap || !n_out) { lvo_set_error(c, "NULL array"); return LVO_E_BADARG; }
  const int L = c->lanes;
  std::vector<size_t> n(L);
  MapOutArgs a;
  LVO_TRY(mapout_batch_begin(c, which, n.data(), &a));
  int short_lane = -1;
  bool any = false;
  for (int l = 0; l < L; ++l) {
    n_out[l] = n[l];
    any = any || d_out[l];
    if (d_out[l] && cap[l] < n[l] && short_lane < 0) short_lane = l;
  }
  if (short_lane >= 0) { lvo_set_error(c, "output buffer of lane " + std::to_string(short_lane) + " too small"); return LVO_E_CAPACITY; }
  if (!any) return LVO_OK;
  LVO_TRY(mapout_reserve_slots(c));
  for (int l = 0; l < L; ++l) c->mapout.h_desc[l] = MapOutDesc{(float4*)d_out[l], (unsigned)n[l], 0u};
  LVO_TRY(mapout_copy(c, which, a, L));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

int lvo_transform_cloud(lvo_ctx* c, lvo_cloud_view in, const lvo_pose* T, int to_end, lvo_cloud_out* out) {
  LVO_ENTER(c);
  if (!out) return LVO_E_BADARG;
  const size_t cap = (size_t)std::max(c->P, std::max(c->map.map_cap[0], c->map.map_cap[1]));
  LVO_TRY(check_view(c, in, cap));
  if (in.n * in.stride > cap * 32) { lvo_set_error(c, "input cloud exceeds the staging buffer"); return LVO_E_CAPACITY; }
  float4* d_in = (float4*)c->d_upload + 2 * cap;   // d_upload holds 4 * cap points; the first half stages strided uploads
  float4* d_out = d_in + cap;
  if (in.n) {
    LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_upload, in.data, in.n * in.stride, cudaMemcpyHostToDevice, c->st));
    k_unpack<<<std::max(1, std::min(lvo_div_up((long long)in.n, 256), 592)), 256, 0, c->st>>>((const unsigned char*)c->d_upload, (int)in.n, (int)in.stride,
                                                                                                 (int)in.off_xyz, (int)in.off_intensity, d_in);
    PoseArg pa; memset(&pa, 0, sizeof(pa));
    if (T) { pa.use = 1; for (int k = 0; k < 4; ++k) pa.q[k] = T->q[k]; for (int k = 0; k < 3; ++k) pa.t[k] = T->t[k]; }
    k_transform_cloud<<<std::max(1, std::min(lvo_div_up((long long)in.n, 256), 592)), 256, 0, c->st>>>(c->d_ls, pa, d_in, (int)in.n, c->cfg.distortion, to_end, d_out);
  }
  const int r = download_cloud(c, d_out, in.n, out);
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return r;
}

static int set_pose(lvo_ctx* c, int lane, int what, const lvo_pose* p) {
  if (!p) return LVO_E_BADARG;
  SetCounts sc; memset(&sc, 0, sizeof(sc));
  sc.what = what;
  for (int k = 0; k < 4; ++k) sc.pose[k] = p->q[k];
  for (int k = 0; k < 3; ++k) sc.pose[4 + k] = p->t[k];
  k_set_lane<<<1, 1, 0, c->st>>>(c->d_ls, lane, sc);
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  return LVO_OK;
}
int lvo_set_map_correction(lvo_ctx* c, int lane, const lvo_pose* T) {
  LVO_ENTER_LANE(c, lane);
  return set_pose(c, lane, 2, T);
}
int lvo_get_map_correction(lvo_ctx* c, int lane, lvo_pose* T) {
  LVO_ENTER_LANE(c, lane);
  if (!T) return LVO_E_BADARG;
  LVO_TRY(sync_state(c));
  pose_out(T, c->h_ls[lane].q_wmap_wodom, c->h_ls[lane].t_wmap_wodom);
  return LVO_OK;
}
int lvo_set_odometry_state(lvo_ctx* c, int lane, const lvo_pose* T_last_curr, const lvo_pose* T_w_curr) {
  LVO_ENTER_LANE(c, lane);
  int r = LVO_OK;
  if (T_last_curr) r = set_pose(c, lane, 3, T_last_curr);
  if (r == LVO_OK && T_w_curr) r = set_pose(c, lane, 4, T_w_curr);
  return r;
}

// ---------------------------------------------------------------------------------------------------------------
}  // extern "C"
// LVO_P_ODO_UNCERTAINTY / LVO_P_MAP_UNCERTAINTY: one launch of k_pose_uncertainty and one copy bring every lane's records into the
// pinned mirror when a raw record may have changed since the last fetch; otherwise the mirror answers.  The launch is not counted in
// lvo_timings::kernel_launches, which keeps reporting the last step or stage call.
static int fetch_uncertainty(lvo_ctx* c, int lane, int stage, void* out, size_t cap_bytes, size_t* n_bytes) {
  if (c->probe_gate[lane] & (stage ? LVO_PROBE_GATE_MAP : LVO_PROBE_GATE_ODO)) {
    lvo_set_error(c, "the lane was loaded from a snapshot and the stage that writes this probe has not run for it since");
    return LVO_E_STATE;
  }
  const size_t bytes = sizeof(lvo_pose_uncertainty);
  if (n_bytes) *n_bytes = bytes;
  if (!out) return LVO_OK;  // size query
  if (cap_bytes < bytes) return LVO_E_CAPACITY;
  if (c->unc_mirror_epoch != c->unc_epoch) {
    const int n = 2 * c->lanes;
    k_pose_uncertainty<<<lvo_div_up(n, 64), 64, 0, c->st>>>(c->d_unc, c->d_unc_out, n);
    LVO_CUDA_OK(c, cudaGetLastError());
    LVO_CUDA_OK(c, cudaMemcpyAsync(c->h_unc, c->d_unc_out, bytes * n, cudaMemcpyDeviceToHost, c->st));
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
    c->unc_mirror_epoch = c->unc_epoch;
  }
  lvo_pose_uncertainty r = c->h_unc[2 * lane + stage];
  r.frame = c->unc_frame[2 * lane + stage];
  memcpy(out, &r, bytes);
  return LVO_OK;
}
extern "C" {

int lvo_probe_fetch(lvo_ctx* c, int lane, int what, void* out, size_t cap_bytes, size_t* n_bytes) {
  LVO_ENTER_LANE(c, lane);
  if (what == LVO_P_ODO_UNCERTAINTY || what == LVO_P_MAP_UNCERTAINTY) return fetch_uncertainty(c, lane, what == LVO_P_MAP_UNCERTAINTY ? 1 : 0, out, cap_bytes, n_bytes);
  LVO_TRY(sync_state(c));
  const LaneState& s = c->h_ls[lane];
  const ExtractArgs& ex = c->ex;
  const int P = c->P, O = c->cfg.outer_iters;
  const void* src = nullptr; size_t bytes = 0;
  // 2-D probes (outer x rows) are gathered row block by row block below
  size_t row_bytes = 0, row_stride = 0; int rows = 1;
  bool per_outer = false;   // probe arrays that keep every outer iteration only with lvo_config::debug_probes
  switch (what) {
    case LVO_P_FULL: src = ex.full + (size_t)lane * P; bytes = (size_t)s.n_kept * 16; break;
    case LVO_P_CURVATURE: src = ex.curv + (size_t)lane * P; bytes = (size_t)s.n_kept * 4; break;
    case LVO_P_SORT_IND: src = ex.sort_ind + (size_t)lane * P; bytes = (size_t)s.n_kept * 4; break;
    case LVO_P_LABEL: src = ex.label + (size_t)lane * P; bytes = (size_t)s.n_kept * 4; break;
    case LVO_P_PICKED: src = ex.picked + (size_t)lane * P; bytes = (size_t)s.n_kept * 4; break;
    case LVO_P_SCAN_START: src = (const char*)(c->d_ls + lane) + offsetof(LaneState, scan_start); bytes = (size_t)c->lane_cfg[lane].n_scans * 4; break;
    case LVO_P_SCAN_END: src = (const char*)(c->d_ls + lane) + offsetof(LaneState, scan_end); bytes = (size_t)c->lane_cfg[lane].n_scans * 4; break;
    case LVO_P_SHARP: src = ex.sharp + (size_t)lane * c->cap_sharp; bytes = (size_t)s.n_sharp * 16; break;
    case LVO_P_LESS_SHARP: src = ex.less_sharp + (size_t)lane * c->cap_lsharp; bytes = (size_t)s.n_less_sharp * 16; break;
    case LVO_P_FLAT: src = ex.flat + (size_t)lane * c->cap_flat; bytes = (size_t)s.n_flat * 16; break;
    case LVO_P_LESS_FLAT: src = ex.less_flat + (size_t)lane * P; bytes = (size_t)s.n_less_flat * 16; break;
    case LVO_P_ODO_CORNER_CORR: src = c->odo.corner_corr + (size_t)lane * c->odo.slots * c->cap_sharp * 2; rows = O; per_outer = true; row_bytes = (size_t)s.n_sharp * 8; row_stride = (size_t)c->cap_sharp * 8; break;
    case LVO_P_ODO_PLANE_CORR: src = c->odo.plane_corr + (size_t)lane * c->odo.slots * c->cap_flat * 3; rows = O; per_outer = true; row_bytes = (size_t)s.n_flat * 12; row_stride = (size_t)c->cap_flat * 12; break;
    case LVO_P_ODO_LM_TRACE: case LVO_P_MAP_LM_TRACE: {
      const double* base = c->d_trace[what == LVO_P_ODO_LM_TRACE ? 0 : 1] + (size_t)lane * LVO_MAX_OUTER * (LVO_MAX_LM + 1) * LVO_TRACE_W;
      src = base; rows = O; row_bytes = (size_t)(c->cfg.lm_max_iters + 1) * LVO_TRACE_W * 8; row_stride = (size_t)(LVO_MAX_LM + 1) * LVO_TRACE_W * 8; break;
    }
    case LVO_P_MAP_CORNER_STACK: src = c->map.stack[0] + (size_t)lane * c->map.in_cap[0]; bytes = (size_t)s.n_stack[0] * 16; break;
    case LVO_P_MAP_SURF_STACK: src = c->map.stack[1] + (size_t)lane * c->map.in_cap[1]; bytes = (size_t)s.n_stack[1] * 16; break;
    case LVO_P_MAP_CORNER_FROM_MAP: src = c->map.from_map[0] + (size_t)lane * c->map.map_cap[0]; bytes = (size_t)s.from_off[0][LVO_MAX_VALID] * 16; break;
    case LVO_P_MAP_SURF_FROM_MAP: src = c->map.from_map[1] + (size_t)lane * c->map.map_cap[1]; bytes = (size_t)s.from_off[1][LVO_MAX_VALID] * 16; break;
    case LVO_P_MAP_CORNER_KNN: case LVO_P_MAP_SURF_KNN: {
      const int t = what == LVO_P_MAP_CORNER_KNN ? 0 : 1;
      src = c->map.knn_ind[t] + (size_t)lane * c->map.slots * c->map.in_cap[t] * 5; rows = O; per_outer = true; row_bytes = (size_t)s.n_stack[t] * 20; row_stride = (size_t)c->map.in_cap[t] * 20; break;
    }
    case LVO_P_MAP_CORNER_VALID: case LVO_P_MAP_SURF_VALID: {
      const int t = what == LVO_P_MAP_CORNER_VALID ? 0 : 1;
      src = c->map.fac_valid[t] + (size_t)lane * c->map.slots * c->map.in_cap[t]; rows = O; per_outer = true; row_bytes = (size_t)s.n_stack[t] * 4; row_stride = (size_t)c->map.in_cap[t] * 4; break;
    }
    case LVO_P_REGISTERED: src = c->map.registered + (size_t)lane * P; bytes = (size_t)s.n_kept * 16; break;
    default: return LVO_E_BADARG;
  }
  if (per_outer && !c->cfg.debug_probes) { lvo_set_error(c, "per-outer-iteration probes need lvo_config::debug_probes = 1"); return LVO_E_STATE; }
  const int gate = what <= LVO_P_LESS_FLAT ? LVO_PROBE_GATE_EXTRACT : (what <= LVO_P_ODO_LM_TRACE ? LVO_PROBE_GATE_ODO : LVO_PROBE_GATE_MAP);
  if (c->probe_gate[lane] & gate) {
    lvo_set_error(c, "the lane was loaded from a snapshot and the stage that writes this probe has not run for it since");
    return LVO_E_STATE;
  }
  if (rows > 1 || row_bytes) bytes = row_bytes * rows;
  if (n_bytes) *n_bytes = bytes;
  if (!out) return LVO_OK;  // size query
  if (cap_bytes < bytes) return LVO_E_CAPACITY;
  if (bytes == 0) return LVO_OK;
  if (row_bytes) {
    LVO_CUDA_OK(c, cudaMemcpy2DAsync(out, row_bytes, src, row_stride, row_bytes, rows, cudaMemcpyDeviceToHost, c->st));
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
    // LVO_OPT_FIXPOINT_SKIP: the outer iterations after a fixed point did not run; each of them would have reproduced the last
    // one that did, so its rows are that iteration's rows
    const bool odo = what == LVO_P_ODO_CORNER_CORR || what == LVO_P_ODO_PLANE_CORR || what == LVO_P_ODO_LM_TRACE;
    const int ran = odo ? s.stats.odo_outer_executed : s.stats.map_outer_executed;
    if (ran >= 1 && ran < rows)   // 0: the stage did not run at all (first frame / map too small)
      for (int o = ran; o < rows; ++o) memcpy((char*)out + (size_t)o * row_bytes, (const char*)out + (size_t)(ran - 1) * row_bytes, row_bytes);
  } else {
    LVO_CUDA_OK(c, cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, c->st));
    LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  }
  return LVO_OK;
}

// ---------------------------------------------------------------------------------------------------------------
int lvo_voxel_downsample(lvo_ctx* c, lvo_cloud_view in, float leaf, lvo_cloud_out* out) {
  LVO_ENTER(c);
  if (!out || !(leaf > 0.f)) return LVO_E_BADARG;
  LVO_TRY(check_view(c, in, (size_t)c->map.vx.cap_items));
  if (in.n * in.stride > (size_t)std::max(c->P, std::max(c->map.map_cap[0], c->map.map_cap[1])) * 64) return LVO_E_CAPACITY;
  c->launches = 0;
  VoxelEngine& vx = c->map.vx;
  LVO_TRY(upload_cloud(c, in, vx.in_pts));
  k_vx_single_setup<<<std::max(1, std::min(lvo_div_up((long long)in.n, 256), 592)), 256, 0, c->st>>>(vx, (int)in.n, leaf);
  lvo_voxel_run(c->st, vx, (int)std::max<size_t>(in.n, 1), 1, 1, &c->launches);
  unsigned n_out = 0;
  LVO_CUDA_OK(c, cudaMemcpyAsync(&n_out, vx.d_n_out, 4, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  if (in.n == 0) n_out = 0;
  int r = download_cloud(c, vx.out_pts, n_out, out);
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  return r;
}

int lvo_voxel_downsample_dev(lvo_ctx* c, const lvo_point* d_in, size_t n, float leaf, lvo_point* d_out, size_t* n_out, float* ms) {
  LVO_ENTER(c);
  if (!d_in || !d_out || !n_out || !(leaf > 0.f)) return LVO_E_BADARG;
  if (n > (size_t)c->map.vx.cap_items) { lvo_set_error(c, "input cloud exceeds the voxel engine capacity"); return LVO_E_CAPACITY; }
  c->launches = 0;
  VoxelEngine& vx = c->map.vx;
  LVO_CUDA_OK(c, cudaMemcpyAsync(vx.in_pts, d_in, n * sizeof(lvo_point), cudaMemcpyDeviceToDevice, c->st));
  k_vx_single_setup<<<std::max(1, std::min(lvo_div_up((long long)n, 256), 592)), 256, 0, c->st>>>(vx, (int)n, leaf);
  cudaEventRecord(c->ev[6], c->st);
  lvo_voxel_run(c->st, vx, (int)std::max<size_t>(n, 1), 1, 1, &c->launches);
  cudaEventRecord(c->ev[7], c->st);
  unsigned cnt = 0;
  LVO_CUDA_OK(c, cudaMemcpyAsync(&cnt, vx.d_n_out, 4, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  if (n == 0) cnt = 0;
  *n_out = cnt;
  if (cnt) LVO_CUDA_OK(c, cudaMemcpyAsync(d_out, vx.out_pts, (size_t)cnt * sizeof(lvo_point), cudaMemcpyDeviceToDevice, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  if (ms) cudaEventElapsedTime(ms, c->ev[6], c->ev[7]);
  return LVO_OK;
}

int lvo_knn(lvo_ctx* c, lvo_cloud_view cloud, lvo_cloud_view queries, int K, float max_sq, int* ind, float* sq) {
  LVO_ENTER(c);
  if (!ind || !sq || (K != 1 && K != 5)) return LVO_E_BADARG;
  LVO_TRY(check_view(c, cloud, (size_t)c->map.map_cap[1])); LVO_TRY(check_view(c, queries, (size_t)c->P));
  c->launches = 0;
  float4* d_cloud = c->map.from_map[1];
  float4* d_q = c->map.registered;
  c->reg_valid = false;   // the queries are staged in map.registered
  LVO_TRY(upload_cloud(c, cloud, d_cloud)); LVO_TRY(upload_cloud(c, queries, d_q));
  const int n = (int)cloud.n;
  LVO_CUDA_OK(c, cudaMemcpyAsync(c->d_knn_n, &n, 4, cudaMemcpyHostToDevice, c->st));
  // cell size: the smallest power of two >= sqrt(max_sq), at least 1/16 m, so that 27 cells cover the gate
  float cell = 0.0625f;
  while (cell * cell < max_sq && cell < 64.f) cell *= 2.f;
  if (K == 1 && cell > 2.f) cell = 2.f;  // 1-NN with a wide gate: small cells + expanding rings (as the odometry stage)
  k_setup_one_problem<<<1, 1, 0, c->st>>>(c->d_knn_prob, d_cloud, c->d_knn_n, cell);
  lvo_grid_build(c->st, c->gknn, &c->launches);
  const int nq = (int)queries.n;
  const int blocks = std::max(1, std::min(lvo_div_up((long long)nq, 8), 1184));
  if (K == 5) k_knn_queries<5><<<blocks, 256, 0, c->st>>>(c->gknn, d_q, nq, max_sq, c->d_knn_ind, c->d_knn_sq);
  else k_knn_queries<1><<<blocks, 256, 0, c->st>>>(c->gknn, d_q, nq, max_sq, c->d_knn_ind, c->d_knn_sq);
  c->launches += 2;
  if (nq) {
    LVO_CUDA_OK(c, cudaMemcpyAsync(ind, c->d_knn_ind, (size_t)nq * K * 4, cudaMemcpyDeviceToHost, c->st));
    LVO_CUDA_OK(c, cudaMemcpyAsync(sq, c->d_knn_sq, (size_t)nq * K * 4, cudaMemcpyDeviceToHost, c->st));
  }
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

// ---- depth association: one problem ("slot") per active lane of the batched calls, or the single call's one slot, solved by one
// launch sequence (lvo_launch_depth) in the calls' own arena
static size_t depth_slot_bytes(int slots) { return ((size_t)slots * sizeof(DepthSlot) + 15) & ~(size_t)15; }

static int depth_alloc(lvo_ctx* c, lvo_ctx::DepthArena& d, size_t pts, size_t raw, size_t kp, int slots) {
  LvoArena& m = d.mem;
  const size_t cells = (size_t)slots * LVO_DEPTH_CELLS + 1;
  LVO_TRY(m.device(c, &d.raw, raw)); LVO_TRY(m.device(c, &d.flag, 4 * pts)); LVO_TRY(m.device(c, &d.dc, 16 * pts));
  LVO_TRY(m.device(c, &d.d_in, depth_slot_bytes(slots) + 8 * kp)); LVO_TRY(m.pinned(c, &d.h_in, depth_slot_bytes(slots) + 8 * kp));
  LVO_TRY(m.device(c, &d.d_res, 20 * kp)); LVO_TRY(m.pinned(c, &d.h_res, 20 * kp));
  LVO_TRY(m.device(c, &d.dc_off, 4 * (size_t)slots)); LVO_TRY(m.device(c, &d.ndc, 4 * (size_t)slots));
  GridSet& g = d.grid;
  memset(&g, 0, sizeof(g));
  g.cells_cap_per_problem = LVO_DEPTH_CELLS;
  LVO_TRY(m.device(c, &g.prob, sizeof(GridProblem) * slots)); LVO_TRY(m.device(c, &g.table, 4 * cells)); LVO_TRY(m.device(c, &g.d_table_len, 4));
  LVO_TRY(m.device(c, &g.rank, 4 * pts)); LVO_TRY(m.device(c, &g.pt_off, 4 * ((size_t)slots + 1)));
  LVO_TRY(m.device(c, &g.sorted_pts, 16 * pts));   // sorted_id: no search reads it
  g.scan.cap_tiles = lvo_div_up((long long)std::max(pts, cells), LVO_SCAN_TILE) + 2;
  LVO_TRY(m.device(c, &g.scan.partial, 4 * (size_t)g.scan.cap_tiles));
  return m.device(c, &d.cnt, 8);   // last: a non-NULL cnt marks the arena as complete
}

// Grows the depth arena to hold `pts` points (`raw` bytes of host-form records), `kp` host-form keypoints and `slots` slots.  The
// stream is idle here (every call ends synchronised), so the old buffers can be freed at once.
static int depth_reserve(lvo_ctx* c, size_t pts, size_t raw, size_t kp, int slots) {
  lvo_ctx::DepthArena& d = c->depth;
  if (d.cnt && pts <= d.cap_pts && raw <= d.cap_raw && kp <= d.cap_kp && slots <= d.cap_slots) return LVO_OK;
  pts = std::max(pts, d.cap_pts); raw = std::max(raw, d.cap_raw); kp = std::max(kp, d.cap_kp); slots = std::max(slots, d.cap_slots);
  d.mem.release(); d.cnt = nullptr;
  d.cap_pts = d.cap_raw = d.cap_kp = 0; d.cap_slots = 0;
  const int r = depth_alloc(c, d, pts, raw, kp, slots);
  if (r != LVO_OK) { d.mem.release(); return r; }
  d.cap_pts = pts; d.cap_raw = raw; d.cap_kp = kp; d.cap_slots = slots;
  return LVO_OK;
}

// Per active lane: keypoint counts within the single call's limit, and the pointers a lane with keypoints needs.
static int depth_check_keypoints(lvo_ctx* c, const void* const* kp, const size_t* n_kp, const void* const* depth, const void* const* valid, const void* const* nn) {
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l] || n_kp[l] == 0) continue;
    if (2 * n_kp[l] > (size_t)c->P) { lvo_set_error(c, "too many keypoints"); return LVO_E_CAPACITY; }
    if (!kp[l] || !depth[l] || !valid[l] || (nn && !nn[l])) { lvo_set_error(c, "NULL keypoint or output pointer of an active lane"); return LVO_E_BADARG; }
  }
  return LVO_OK;
}

// Uploads the slots (and the host form's keypoints behind them) staged in h_in, then enqueues the kernels.
static int depth_enqueue(lvo_ctx* c, int nslot, size_t n_total, size_t kp_total, int max_n, int stride, int off_xyz, size_t in_bytes) {
  lvo_ctx::DepthArena& d = c->depth;
  LVO_CUDA_OK(c, cudaMemcpyAsync(d.d_in, d.h_in, in_bytes, cudaMemcpyHostToDevice, c->st));
  DepthArgs a;
  memset(&a, 0, sizeof(a));
  a.slot = (const DepthSlot*)d.d_in; a.nslot = nslot; a.stride = stride; a.off_xyz = off_xyz;
  a.n_total = (int)n_total; a.kp_total = (int)kp_total;
  a.flag = d.flag; a.d_n = d.cnt; a.d_total = (unsigned*)(d.cnt + 1); a.dc_off = d.dc_off; a.ndc = d.ndc; a.dc = d.dc;
  a.grid = d.grid;
  a.grid.nprob = nslot; a.grid.table_cap_total = (long long)nslot * LVO_DEPTH_CELLS; a.grid.pts_cap_per_problem = std::max(max_n, 1);
  lvo_launch_depth(c->st, a, max_n, d.grid.scan, &c->launches);
  return LVO_OK;
}

static void depth_slot_camera(DepthSlot& s, const lvo_camera& cam) { for (int k = 0; k < 12; ++k) s.extr[k] = cam.extrinsic[k]; }

// One slot of the host form: its sweep (records of the call's layout), keypoints and outputs.
struct DepthHostSlot { const lvo_camera* cam; const lvo_cloud_view* sweep; const float* uv; size_t nkp; float* depth; int* valid; int* nn; };

// Host form over the slots `in`, in an arena reserved for them: the sweeps back to back in slot order (exactly the bytes of each
// view, one copy per run of views that are contiguous in host memory), the keypoints behind the slot records (one upload), the
// results in one download, copied to each slot's outputs once the stream has synchronised.  ndc_or_null gets each slot's
// depth-cloud size.
static int depth_host(lvo_ctx* c, const std::vector<DepthHostSlot>& in, int stride, int off_xyz, bool want_nn, int* ndc_or_null) {
  lvo_ctx::DepthArena& d = c->depth;
  const int S = (int)in.size();
  size_t N = 0, K = 0; int max_n = 0;
  for (const DepthHostSlot& s : in) { N += s.sweep->n; K += s.nkp; max_n = std::max(max_n, (int)s.sweep->n); }
  DepthSlot* hs = (DepthSlot*)d.h_in;
  float* huv = (float*)(d.h_in + depth_slot_bytes(S));
  const float* d_uv = (const float*)(d.d_in + depth_slot_bytes(S));
  float* r_depth = (float*)d.d_res; int* r_valid = (int*)d.d_res + K; int* r_nn = (int*)d.d_res + 2 * K;
  struct Run { const unsigned char* host; size_t bytes; size_t dev_off; };
  std::vector<Run> runs;
  size_t po = 0, ko = 0;
  for (int s = 0; s < S; ++s) {
    const lvo_cloud_view& v = *in[s].sweep;
    DepthSlot& t = hs[s];
    memset(&t, 0, sizeof(t));
    t.pts = d.raw + po * stride; t.n = (int)v.n; t.pt_off = (unsigned)po;
    t.uv = d_uv + 2 * ko; t.nkp = (int)in[s].nkp; t.kp_off = (unsigned)ko;
    t.depth = r_depth + ko; t.valid = r_valid + ko; t.nn = want_nn ? r_nn + 3 * ko : nullptr;
    depth_slot_camera(t, *in[s].cam);
    if (in[s].nkp) memcpy(huv + 2 * ko, in[s].uv, 8 * in[s].nkp);
    if (v.n) {
      const unsigned char* h = (const unsigned char*)v.data;
      const size_t bytes = v.n * stride;
      if (!runs.empty() && runs.back().host + runs.back().bytes == h) runs.back().bytes += bytes;
      else runs.push_back(Run{h, bytes, po * stride});
    }
    po += v.n; ko += in[s].nkp;
  }
  for (const Run& r : runs) LVO_CUDA_OK(c, cudaMemcpyAsync(d.raw + r.dev_off, r.host, r.bytes, cudaMemcpyHostToDevice, c->st));
  LVO_TRY(depth_enqueue(c, S, N, K, max_n, stride, off_xyz, depth_slot_bytes(S) + 8 * K));
  const size_t res_words = (want_nn ? 5 : 2) * K;
  if (res_words) LVO_CUDA_OK(c, cudaMemcpyAsync(d.h_res, d.d_res, 4 * res_words, cudaMemcpyDeviceToHost, c->st));
  if (ndc_or_null) LVO_CUDA_OK(c, cudaMemcpyAsync(ndc_or_null, d.ndc, sizeof(int) * S, cudaMemcpyDeviceToHost, c->st));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  const float* h_depth = (const float*)d.h_res; const int* h_valid = (const int*)d.h_res + K; const int* h_nn = (const int*)d.h_res + 2 * K;
  ko = 0;
  for (const DepthHostSlot& s : in) {
    if (s.nkp) {
      memcpy(s.depth, h_depth + ko, 4 * s.nkp);
      memcpy(s.valid, h_valid + ko, 4 * s.nkp);
      if (want_nn) memcpy(s.nn, h_nn + 3 * ko, 12 * s.nkp);
    }
    ko += s.nkp;
  }
  return LVO_OK;
}

int lvo_depth_associate(lvo_ctx* c, lvo_cloud_view sweep, const lvo_camera* cam, const float* keypoints_uv, size_t n_kp, float* depth_out, int* valid_out,
                        int* nn_out, lvo_cloud_out* depth_cloud_or_null) {
  LVO_ENTER(c);
  if (!cam || (n_kp && (!keypoints_uv || !depth_out || !valid_out))) return LVO_E_BADARG;
  LVO_TRY(check_view(c, sweep, (size_t)c->P));
  if (2 * n_kp > (size_t)c->P) { lvo_set_error(c, "too many keypoints"); return LVO_E_CAPACITY; }
  c->launches = 0;
  // one slot of the batched calls' arena, reserved on first use at this call's limits (max_points points of the view's stride,
  // max_points / 2 keypoints): no later call within them reallocates
  const int stride = sweep.n ? (int)sweep.stride : 16, off_xyz = sweep.n ? (int)sweep.off_xyz : 0;
  LVO_TRY(depth_reserve(c, (size_t)c->P, (size_t)c->P * stride, (size_t)c->P / 2, 1));
  int ndc = 0;
  LVO_TRY(depth_host(c, {DepthHostSlot{cam, &sweep, keypoints_uv, n_kp, depth_out, valid_out, nn_out}}, stride, off_xyz, nn_out != nullptr, &ndc));
  if (sweep.n == 0) ndc = 0;
  const int r = download_cloud(c, c->depth.dc, (size_t)ndc, depth_cloud_or_null);   // slot 0's depth cloud starts the array
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  return r;
}

int lvo_depth_associate_batch(lvo_ctx* c, const lvo_camera* cams, const lvo_cloud_view* sweeps, const float* const* keypoints_uv, const size_t* n_kp,
                              float* const* depth_out, int* const* valid_out, int* const* nn_out_or_null) {
  LVO_ENTER(c);
  if (!cams || !sweeps || !keypoints_uv || !n_kp || !depth_out || !valid_out) { lvo_set_error(c, "NULL array"); return LVO_E_BADARG; }
  int max_n = 0, stride = 16, off_xyz = 0;
  LVO_TRY(check_sweeps(c, sweeps, &max_n, &stride, &off_xyz));
  LVO_TRY(depth_check_keypoints(c, (const void* const*)keypoints_uv, n_kp, (const void* const*)depth_out, (const void* const*)valid_out,
                                (const void* const*)nn_out_or_null));
  std::vector<DepthHostSlot> in;
  size_t N = 0, K = 0;
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l]) continue;
    in.push_back(DepthHostSlot{&cams[l], &sweeps[l], keypoints_uv[l], n_kp[l], depth_out[l], valid_out[l], nn_out_or_null ? nn_out_or_null[l] : nullptr});
    N += sweeps[l].n; K += n_kp[l];
  }
  if (N > INT_MAX || K > INT_MAX) { lvo_set_error(c, "too many points or keypoints in one call"); return LVO_E_CAPACITY; }
  c->launches = 0;
  if (in.empty()) return LVO_OK;
  LVO_TRY(depth_reserve(c, N, N * stride, K, (int)in.size()));
  return depth_host(c, in, stride, off_xyz, nn_out_or_null != nullptr, nullptr);
}

int lvo_depth_associate_batch_dev(lvo_ctx* c, const lvo_camera* cams, const lvo_point* const* d_sweeps, const size_t* n, const float* const* d_keypoints_uv,
                                  const size_t* n_kp, float* const* d_depth_out, int* const* d_valid_out, int* const* d_nn_out_or_null) {
  LVO_ENTER(c);
  if (!cams || !d_sweeps || !n || !d_keypoints_uv || !n_kp || !d_depth_out || !d_valid_out) { lvo_set_error(c, "NULL array"); return LVO_E_BADARG; }
  int A = 0, max_n = 0; size_t N = 0, K = 0;
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l]) continue;
    if (n[l] > (size_t)c->P) { lvo_set_error(c, "input cloud exceeds context capacity"); return LVO_E_CAPACITY; }
    if (n[l] && !d_sweeps[l]) { lvo_set_error(c, "NULL sweep of an active lane"); return LVO_E_BADARG; }
    A++; N += n[l]; K += n_kp[l]; max_n = std::max(max_n, (int)n[l]);
  }
  LVO_TRY(depth_check_keypoints(c, (const void* const*)d_keypoints_uv, n_kp, (const void* const*)d_depth_out, (const void* const*)d_valid_out,
                                (const void* const*)d_nn_out_or_null));
  if (N > INT_MAX || K > INT_MAX) { lvo_set_error(c, "too many points or keypoints in one call"); return LVO_E_CAPACITY; }
  c->launches = 0;
  if (A == 0) return LVO_OK;
  LVO_TRY(depth_reserve(c, N, 0, 0, A));
  DepthSlot* hs = (DepthSlot*)c->depth.h_in;
  int s = 0; size_t po = 0, ko = 0;
  for (int l = 0; l < c->lanes; ++l) {
    if (!c->lane_active[l]) continue;
    DepthSlot& t = hs[s++];
    memset(&t, 0, sizeof(t));
    t.pts = (const unsigned char*)d_sweeps[l]; t.n = (int)n[l]; t.pt_off = (unsigned)po;
    t.uv = d_keypoints_uv[l]; t.nkp = (int)n_kp[l]; t.kp_off = (unsigned)ko;
    t.depth = d_depth_out[l]; t.valid = d_valid_out[l]; t.nn = d_nn_out_or_null ? d_nn_out_or_null[l] : nullptr;
    depth_slot_camera(t, cams[l]);
    po += n[l]; ko += n_kp[l];
  }
  LVO_TRY(depth_enqueue(c, A, N, K, max_n, 16, 0, depth_slot_bytes(A)));
  LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
  LVO_CUDA_OK(c, cudaGetLastError());
  return LVO_OK;
}

__global__ void k_setup_batch_problems(GridProblem* prob, int S, const float4* maps, const unsigned* m_off, const int* m_cnt, float cell) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= S) return;
  prob[p].pts = maps + m_off[p]; prob[p].d_n = m_cnt + p; prob[p].want_cell = cell; prob[p].want_cell_z = 0.f; prob[p].mode = 0; prob[p].cells_cap = 0; prob[p].clamp_xy = 0.f; prob[p].bbox_from = -1;
}

int lvo_knn5_throughput(lvo_ctx* c, const lvo_point* d_maps, const int* map_counts, const lvo_point* d_queries, const int* query_counts, int S, int reps,
                        int* d_ind_out, float* d_sq_out, float* ms) {
  LVO_ENTER(c);
  if (!d_maps || !map_counts || !d_queries || !query_counts || S < 1 || reps < 1 || !d_ind_out || !d_sq_out || !ms) return LVO_E_BADARG;
  std::vector<unsigned> moff(S + 1, 0), qoff(S + 1, 0);
  int maxm = 1, maxq = 1;
  for (int p = 0; p < S; ++p) {
    if (map_counts[p] < 0 || query_counts[p] < 0) return LVO_E_BADARG;
    moff[p + 1] = moff[p] + (unsigned)map_counts[p]; qoff[p + 1] = qoff[p] + (unsigned)query_counts[p];
    maxm = std::max(maxm, map_counts[p]); maxq = std::max(maxq, query_counts[p]);
  }
  // temporary grid set and L2 flush buffer, zero-filled on the stream; released once the stream is idle, on every return path
  LvoArena tmp;
  auto talloc = [&](auto** p, size_t bytes) { LVO_TRY(tmp.device(c, p, bytes)); LVO_CUDA_OK(c, cudaMemsetAsync(*p, 0, bytes, c->st)); return LVO_OK; };
  const int r = [&]() -> int {
    GridSet g; memset(&g, 0, sizeof(g));
    const int cells_cap = 1 << 21;
    g.nprob = S; g.cells_cap_per_problem = cells_cap; g.pts_cap_per_problem = maxm;
    unsigned* d_moff = nullptr; unsigned* d_qoff = nullptr; int* d_mcnt = nullptr;
    const size_t total_m = moff[S];
    const size_t table_n = (size_t)S * cells_cap + 1;
    g.scan.cap_tiles = lvo_div_up((long long)table_n, LVO_SCAN_TILE) + 2;
    LVO_TRY(talloc(&g.prob, sizeof(GridProblem) * S)); LVO_TRY(talloc(&g.table, 4 * table_n)); LVO_TRY(talloc(&g.d_table_len, 4));
    LVO_TRY(talloc(&g.rank, 4 * total_m)); LVO_TRY(talloc(&g.pt_off, 4 * (size_t)(S + 1))); LVO_TRY(talloc(&g.sorted_pts, 16 * total_m));
    LVO_TRY(talloc(&g.sorted_id, 4 * total_m)); LVO_TRY(talloc(&g.scan.partial, 4 * (size_t)g.scan.cap_tiles));
    LVO_TRY(talloc(&d_moff, 4 * (size_t)(S + 1))); LVO_TRY(talloc(&d_qoff, 4 * (size_t)(S + 1))); LVO_TRY(talloc(&d_mcnt, 4 * (size_t)S));
    LVO_CUDA_OK(c, cudaMemcpyAsync(d_moff, moff.data(), 4 * (size_t)(S + 1), cudaMemcpyHostToDevice, c->st));
    LVO_CUDA_OK(c, cudaMemcpyAsync(d_qoff, qoff.data(), 4 * (size_t)(S + 1), cudaMemcpyHostToDevice, c->st));
    LVO_CUDA_OK(c, cudaMemcpyAsync(d_mcnt, map_counts, 4 * (size_t)S, cudaMemcpyHostToDevice, c->st));
    k_setup_batch_problems<<<lvo_div_up(S, 64), 64, 0, c->st>>>(g.prob, S, (const float4*)d_maps, d_moff, d_mcnt, 1.0f);
    c->launches = 0;
    lvo_grid_build(c->st, g, &c->launches);
    dim3 grid(std::max(1, std::min(lvo_div_up(maxq, 128), 256)), S);
    k_knn5_batch<<<grid, 128, 0, c->st>>>(g, (const float4*)d_queries, d_qoff, 1.0f, d_ind_out, d_sq_out);  // warm-up
    // every timed launch starts with a cold L2: a 256 MB scratch buffer (> 126 MB L2) is overwritten in between
    void* flush = nullptr;
    const size_t flush_bytes = 256u << 20;
    LVO_TRY(talloc(&flush, flush_bytes));
    float t = 0;
    for (int k = 0; k < reps; ++k) {
      cudaMemsetAsync(flush, k & 0xff, flush_bytes, c->st);
      cudaEventRecord(c->ev[6], c->st);
      k_knn5_batch<<<grid, 128, 0, c->st>>>(g, (const float4*)d_queries, d_qoff, 1.0f, d_ind_out, d_sq_out);
      cudaEventRecord(c->ev[7], c->st);
      LVO_CUDA_OK(c, cudaStreamSynchronize(c->st));
      float tr = 0;
      if (cudaEventElapsedTime(&tr, c->ev[6], c->ev[7]) == cudaSuccess) t += tr;
    }
    LVO_CUDA_OK(c, cudaGetLastError());
    *ms = t / reps;
    return LVO_OK;
  }();
  cudaStreamSynchronize(c->st);
  tmp.release();
  return r;
}

}  // extern "C"
