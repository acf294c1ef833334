/* lvo.h — C ABI of liblvo.so: the B200 (sm_100a) drop-in for the per-frame hot path of the reference
 * A-LOAM fork (ucmmesa/Lidar-Visual-Odometry).
 *
 * The reference exposes this path only as three ROS callback / loop bodies.  Each entry point below replaces
 * exactly one of them (citations are into the reference tree):
 *
 *   lvo_extract_features  <-  laserCloudHandler body            src/scanRegistration.cpp:127-411
 *   lvo_scan_to_scan      <-  odometry frame body               src/laserOdometry.cpp:353-641
 *   lvo_scan_to_map       <-  mapping process() body            src/laserMapping.cpp:307-848
 *
 * Payload type is the reference's PointType = pcl::PointXYZI (include/aloam_velodyne/common.h:43); a
 * lvo_cloud_view describes its memory without naming PCL (stride 32, xyz at 0, intensity at 16), or a packed
 * float4 (stride 16, xyz at 0, intensity at 12).  Poses are (quaternion x,y,z,w ; translation) in double, the
 * layout of the reference's `para_q/para_t` (laserOdometry.cpp:131-137) and `parameters[7]`
 * (laserMapping.cpp:110-112).
 *
 * No exceptions cross this boundary; no torch / PCL / Eigen / ROS types appear in it.  All arithmetic runs in
 * hand-written CUDA kernels; there is no CPU fallback: lvo_create fails with LVO_E_CUDA when no sm_100 device
 * (or no CUDA device at all) is usable.
 */
#ifndef LVO_H_
#define LVO_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ---------------------------------------------------------------------------------------- */
#define LVO_OK 0
#define LVO_E_BADARG (-1)   /* null pointer, bad stride, unsupported n_scans (reference: ROS_BREAK, scanRegistration.cpp:203) */
#define LVO_E_CAPACITY (-2) /* an input exceeds the context's capacities, or an output buffer is too small          */
#define LVO_E_CUDA (-3)     /* CUDA error (sticky); text through lvo_last_error                                    */
#define LVO_E_STATE (-4)    /* call order violated (e.g. lane out of range)                                        */
/* positive = the reference's soft conditions; outputs are still valid */
#define LVO_W_FIRST_FRAME 1   /* laserOdometry.cpp:355-358: first frame only initialises                           */
#define LVO_W_FEW_CORR 2      /* laserOdometry.cpp:566-568: < 10 correspondences in some outer iteration           */
#define LVO_W_MAP_TOO_SMALL 3 /* laserMapping.cpp:554,730-733: map too small, pose = initial guess, map updated    */

/* ---- plain data ------------------------------------------------------------------------------------------ */
typedef struct lvo_point { float x, y, z, intensity; } lvo_point; /* device + output layout: packed float4 */

typedef struct lvo_cloud_view { /* borrowed for the duration of the call */
  const void* data;
  size_t n;             /* number of points */
  size_t stride;        /* bytes between points: 32 for pcl::PointXYZI, 16 for lvo_point; raw sweeps (lvo_extract_features,
                         * lvo_step_batch*) may also be packed x,y,z records of 12 bytes: the path never reads a sweep's intensity
                         * (scanRegistration.cpp:132-133 converts the message to pcl::PointXYZ), off_intensity is then ignored */
  size_t off_xyz;       /* byte offset of x (y, z follow) */
  size_t off_intensity; /* byte offset of intensity */
} lvo_cloud_view;

typedef struct lvo_cloud_out { /* caller-owned; n is written back; LVO_E_CAPACITY if cap < n */
  lvo_point* data;
  size_t cap;
  size_t n;
} lvo_cloud_out;

typedef struct lvo_pose { double q[4]; /* x,y,z,w */ double t[3]; } lvo_pose;

typedef struct lvo_config {
  int n_scans;           /* 16 | 32 | 64                        scanRegistration.cpp:466                   */
  double minimum_range;  /* m                                   scanRegistration.cpp:468                   */
  double line_res;       /* corner voxel leaf, m                laserMapping.cpp:902                        */
  double plane_res;      /* surf voxel leaf, m                  laserMapping.cpp:903                        */
  int skip_frame;        /* mapping_skip_frame                  laserOdometry.cpp:274                       */
  int outer_iters;       /* 10                                  laserOdometry.cpp:364, laserMapping.cpp:562 */
  int lm_max_iters;      /* 4                                   laserOdometry.cpp:573, laserMapping.cpp:715 */
  double huber;          /* 0.1                                 laserOdometry.cpp:369, laserMapping.cpp:565 */
  int device;            /* CUDA ordinal                                                                    */
  int lanes;             /* independent sequences advanced in lock-step by the *_batch entry points (>=1)  */
  int max_points;        /* capacity per sweep (reference: 400000, scanRegistration.cpp:66); 0 = 262144    */
  int max_map_corner;    /* capacity of the whole corner map per lane, points; 0 = 1<<20                   */
  int max_map_surf;      /* capacity of the whole surf map per lane, points;   0 = 1<<21                   */
  int distortion;        /* the compile-time switch `#define DISTORTION` of laserOdometry.cpp:67 made a run-time option:
                          * 0 = DISTORTION 0 (the shipped value): s = 1 everywhere;
                          * 1 = DISTORTION 1 as the file is written: s = (intensity - int(intensity)) / SCAN_PERIOD per point in
                          *     TransformToStart (:157-163) and in LidarEdgeFactor / LidarPlaneFactor (:455-459, :549-553;
                          *     lidarFactor.hpp:27-30, 79-82); the TransformToEnd block (:610-625) stays off (`if (0)`);
                          * 2 = 1 plus that block: less-sharp, less-flat and full clouds are moved to the sweep end (:176-191)
                          *     before they become the "last" clouds and the mapping input.                                   */
  int debug_probes;      /* 1 = keep the per-outer-iteration parity probes (LVO_P_ODO_*_CORR, LVO_P_MAP_*_KNN / _VALID) of ALL outer
                          * iterations (16 slots per lane: ~50 MB per lane at the default capacities); 0 (default) = only what the path
                          * itself needs (the current and the previous iteration), and lvo_probe_fetch of those probes returns
                          * LVO_E_STATE.  Results are identical either way.                                                         */
} lvo_config;

/* Per-call counters, also the parity probes (SURVEY §5 "Metrics / logging").  One record per lane. */
typedef struct lvo_stats {
  /* lvo_extract_features */
  int n_in, n_kept, n_sharp, n_less_sharp, n_flat, n_less_flat;
  /* lvo_scan_to_scan: per outer iteration */
  int odo_corner_corr[16], odo_plane_corr[16], odo_lm_iters[16];
  double odo_final_cost[16];
  /* lvo_scan_to_map */
  int map_corner_from_map, map_surf_from_map, map_corner_stack, map_surf_stack;
  int map_corner_corr[16], map_surf_corr[16], map_lm_iters[16];
  double map_final_cost[16];
  int map_corner_total, map_surf_total; /* points in all 4851 cubes after insertion + re-filter */
  int center_cube[3], cen[3];           /* centerCubeI/J/K and laserCloudCen{Width,Height,Depth} after shifting */
  /* outer iterations that actually ran (== outer_iters unless LVO_OPT_FIXPOINT_SKIP cut the loop short; the per-iteration
   * entries above are then filled with the values of the last iteration that ran, which every later one would reproduce) */
  int odo_outer_executed, map_outer_executed;
  /* LVO_OPT_KNN_REUSE: queries of lvo_scan_to_map that were searched in full per outer iteration (iteration 0: all of them; later
   * ones: those whose neighbour set could not be carried over with a certificate).  Diagnostic only. */
  int map_knn_full[16];
  /* scan-to-scan features per outer iteration that the thread-per-feature association handed to the warp-per-feature kernel, and why
   * (summed over the iterations of the frame): 0 no bound on the closest point, 1 bound wider than a fine cell, 2 closest point beyond the
   * 5 m gate, 3 an adjacent-ring target exists but its azimuth window is wider than the fast limit, 4 an adjacent-ring target has no
   * candidate nearby, 5 too few uncertified features left in a block to keep one thread busy each.  Diagnostic only. */
  int odo_slow[16], odo_slow_why[6];
  /* LVO_OPT_ODO_REUSE: scan-to-scan features per outer iteration whose correspondence was carried over under the certificate */
  int odo_certified[16];
} lvo_stats;

typedef struct lvo_ctx lvo_ctx; /* one per (GPU, group of lanes); owns streams, device arenas, cross-frame state */

/* ---- lifetime -------------------------------------------------------------------------------------------- */
void lvo_default_config(lvo_config* cfg); /* HDL-64 launch values: 64, 5.0, 0.4, 0.8, 1, 10, 4, 0.1, dev 0, 1 lane */
int lvo_create(const lvo_config* cfg, lvo_ctx** out);
int lvo_destroy(lvo_ctx* ctx);
const char* lvo_last_error(const lvo_ctx* ctx);
int lvo_get_stats(const lvo_ctx* ctx, int lane, lvo_stats* out, size_t bytes);

/* ---- the three drop-in entry points (lane 0 with lane 0's lvo_lane_config; synchronous on return) ----------- */

/* scanRegistration.cpp:127-411.  `sweep` = /velodyne_points; outputs = /velodyne_cloud_2, /laser_cloud_sharp,
 * /laser_cloud_less_sharp, /laser_cloud_flat, /laser_cloud_less_flat (:413-441).  Any output may be NULL. */
int lvo_extract_features(lvo_ctx* ctx, lvo_cloud_view sweep, lvo_cloud_out* full, lvo_cloud_out* sharp,
                         lvo_cloud_out* less_sharp, lvo_cloud_out* flat, lvo_cloud_out* less_flat);

/* laserOdometry.cpp:353-641.  Keeps para_q/para_t, q_w_curr/t_w_curr and the two "last" clouds in ctx.
 * T_last_curr = (para_q, para_t) after the solve; T_w_curr = accumulated odometry pose (:581-582). */
int lvo_scan_to_scan(lvo_ctx* ctx, lvo_cloud_view sharp, lvo_cloud_view less_sharp, lvo_cloud_view flat,
                     lvo_cloud_view less_flat, lvo_pose* T_last_curr, lvo_pose* T_w_curr);

/* laserMapping.cpp:307-848.  corner_last / surf_last are what laserOdometry publishes (:646-656), i.e. the
 * current frame's less-sharp / less-flat clouds; full_or_null is /velodyne_cloud_3; T_wodom_curr is
 * /laser_odom_to_init.  Writes /aft_mapped_to_init to T_wmap_curr and, if requested, /velodyne_cloud_registered. */
int lvo_scan_to_map(lvo_ctx* ctx, lvo_cloud_view corner_last, lvo_cloud_view surf_last, lvo_cloud_view full_or_null,
                    const lvo_pose* T_wodom_curr, lvo_pose* T_wmap_curr, lvo_cloud_out* registered_or_null);

/* ---- device-resident, batched pipeline (SURVEY §8f rank 1: no host hops between the three stages) --------- */

/* One frame for every lane: extract -> scan-to-scan -> scan-to-map, all on device.  sweeps[l] is the sweep of
 * lane l (host memory; copied through pinned staging).  Poses may be NULL.  Returns the max status over lanes;
 * per-lane statuses through lvo_lane_status. */
int lvo_step_batch(lvo_ctx* ctx, const lvo_cloud_view* sweeps, lvo_pose* T_wodom_curr, lvo_pose* T_wmap_curr);

/* Pipelined form of lvo_step_batch for a host loop: computes the frame `sweeps` and, while it runs, uploads `next_sweeps`
 * (may be NULL) on a copy stream into a second staging buffer, the way the reference's ROS nodes overlap transport and
 * compute.  If `sweeps` is the set that the previous call prefetched (same pointers and sizes) no copy is issued for it.
 * The buffers of next_sweeps must stay valid and unchanged until the next call. */
int lvo_step_batch_pipelined(lvo_ctx* ctx, const lvo_cloud_view* sweeps, const lvo_cloud_view* next_sweeps_or_null, lvo_pose* T_wodom_curr,
                             lvo_pose* T_wmap_curr);

/* Asynchronous forms (SURVEY §8b "Threading": `_async` + lvo_wait, for pipelining a host loop the way the reference's three ROS
 * processes overlap): lvo_step_batch_async copies and enqueues one frame for every lane and returns without waiting for the GPU;
 * lvo_wait blocks until that frame is done and delivers its poses / statuses (same return value as lvo_step_batch).  The sweep
 * buffers must stay valid and unchanged until lvo_wait returns; exactly one step may be in flight per context; every other entry
 * point returns LVO_E_STATE while one is.  Lanes whose host buffers are adjacent in memory (one slab) are uploaded in one copy. */
int lvo_step_batch_async(lvo_ctx* ctx, const lvo_cloud_view* sweeps);
int lvo_step_batch_dev_async(lvo_ctx* ctx, const lvo_point* const* d_sweeps, const size_t* n);
int lvo_wait(lvo_ctx* ctx, lvo_pose* T_wodom_curr, lvo_pose* T_wmap_curr);

/* Same, with sweeps already resident in device memory as packed lvo_point arrays (d_sweeps[l] is a device
 * pointer with n[l] points).  This is what bench.py's device-resident `value` times. */
int lvo_step_batch_dev(lvo_ctx* ctx, const lvo_point* const* d_sweeps, const size_t* n, lvo_pose* T_wodom_curr,
                       lvo_pose* T_wmap_curr);
int lvo_lane_status(const lvo_ctx* ctx, int lane);

/* ---- per-lane lifecycle: sequences of unequal length, or started at different times, share one context ----- */

/* Lane activity (default: every lane active).  The lvo_step_batch* calls skip an idle lane entirely: its sweep view / device
 * pointer / count is not read, validated or uploaded (may be NULL / 0); its poses, odometry state and "last" clouds, map
 * (both generations as seen through lvo_map_export / lvo_map_cloud), map correction, lvo_stats, probes, lvo_lane_status and
 * skip_frame phase are left exactly as they were; its entries of T_wodom_curr / T_wmap_curr are not written; it does not
 * contribute to the returned status.  A step in which no lane is active returns LVO_OK.  Resuming the lane continues its
 * sequence bit for bit as if the idle steps had not happened.  Each lane maps on its own frames 0, skip_frame, 2 skip_frame, ...
 * An idle lane is not free: its odometry grids are rebuilt and its map is copied into the other generation.  Measured on a B200
 * (1000 W, 128 lanes): with 1/4, 1/2, 3/4 of the lanes idle a step takes 0.95, 0.77, 0.64 of its all-active time
 * (profiles/lane_lifecycle.md); the cost of an idle lane by itself is not measured.
 * LVO_E_STATE while an *_async step is in flight, LVO_E_BADARG for a bad lane.  Captured CUDA graphs stay valid. */
int lvo_set_lane_active(lvo_ctx* ctx, int lane, int active);
/* Map updates of `lane` (default: on).  update != 0: every mapping frame inserts the frame's stack into the cubes and re-filters the
 * valid cubes (laserMapping.cpp:737-801), as the reference does.  update == 0, localisation in a fixed prior map: the lane runs
 * process() (:307-848) with the insertion (:737-783) and the per-cube re-filter (:788-801) skipped; everything else runs unchanged:
 * transformAssociateToMap, the cube-window shift (:312-507), the valid list, the FromMap gather, the stack downsample, the 5-NN
 * search and the fits, the LM solve over every outer iteration, transformUpdate (the map correction keeps being refined) and the
 * registered cloud.  The reference has no such mode.  Consequences:
 *   - The map does not change while updates are off, except by the cube-window shift: cubes that leave the 21 x 21 x 11 window are
 *     dropped, as always, so a fixed map is bounded by the window (about 1050 x 1050 x 550 m around where it sits).
 *     lvo_stats::map_corner_total / map_surf_total report the stored map after any such drop.
 *   - An empty or too-small map gives LVO_W_MAP_TOO_SMALL on every mapping frame, with the initial guess as the pose.
 *   - A lane with updates off never returns LVO_E_CAPACITY from the map.
 *   - skip_frame, the high-frequency pose of non-mapping frames, statuses, probes and lvo_map_cloud[_batch] behave as for a lane
 *     with updates on.
 * Takes effect from the next call that runs the mapping stage (the lvo_step_batch* calls, and lvo_scan_to_map for lane 0) and may
 * change between any two steps.  It is host state, like activity: not part of lvo_config, lvo_lane_config or a snapshot (the bytes
 * of lvo_lane_save do not depend on it), and lvo_lane_reset, lvo_lane_configure, lvo_lane_load and lvo_set_lane_active leave it as
 * it is.  LVO_E_STATE while an *_async step is in flight, LVO_E_BADARG for a bad lane.  Captured CUDA graphs stay valid, and a step
 * launches the same kernels whatever the lanes' settings.  INTEGRATION.md, "Localisation in a prior map", gives the recipe. */
int lvo_set_lane_map_update(lvo_ctx* ctx, int lane, int update);
/* Return `lane` to the state of a freshly created context: next active step is its first frame (LVO_W_FIRST_FRAME), empty map,
 * identity poses and map correction, cen = (10, 10, 5), zero lvo_stats, status LVO_OK, skip_frame phase 0.  Other lanes are
 * untouched, and so are the lane's activity and its settings (lvo_lane_configure).  Stream-ordered (returns when done); LVO_E_STATE while an *_async step is in flight,
 * LVO_E_BADARG for a bad lane.  Captured CUDA graphs stay valid.  To resume a saved sequence exactly, use lvo_lane_load instead; to
 * start a new sequence from a pre-built map, follow the reset with lvo_map_import / lvo_set_odometry_state. */
int lvo_lane_reset(lvo_ctx* ctx, int lane);

/* ---- per-lane sensor settings: sequences of VLP-16, HDL-32 and HDL-64 sensors side by side in one context ---------------- */

/* The values the reference's launch files set per sensor model (launch/aloam_velodyne_VLP_16.launch: 16, 0.3, 0.2, 0.4;
 * aloam_velodyne_HDL_64.launch: 64, 5.0, 0.4, 0.8; both with mapping_skip_frame 1).  Same meaning and units as in lvo_config. */
typedef struct lvo_lane_config {
  int n_scans;           /* 16 | 32 | 64, and <= the context's lvo_config::n_scans   scan_line               */
  double minimum_range;  /* m, finite and >= 0                                        minimum_range           */
  double line_res;       /* corner voxel leaf, m, finite and > 0                      mapping_line_resolution  */
  double plane_res;      /* surf voxel leaf, m, finite and > 0                        mapping_plane_resolution */
  int skip_frame;        /* >= 1                                                      mapping_skip_frame       */
} lvo_lane_config;
/* Start a new sequence in `lane` with the settings `cfg` (NULL: the context's own values): everything lvo_lane_reset does (the next
 * active step is the lane's first frame, its skip_frame phase 0), then the lane takes the settings.  They change only here, at the
 * start of a sequence, as the reference reads them once at start-up.  Every other lane and the lane's activity are untouched.
 *   - A lane that was never configured has the context's lvo_config values; lvo_lane_reset and lvo_lane_load keep a lane's settings.
 *   - A lane computes bit for bit what lane 0 of a context created with its settings computes; the context's n_scans, the largest a
 *     lane may take, only sizes the buffers: a 16-beam lane of a 64-beam context holds 64-beam feature buffers (DESIGN.md §1).
 *   - outer_iters, lm_max_iters, huber and distortion are solver settings and stay per context.
 *   - Errors, all checked before anything is written (the lane's state and settings are left as they were; lvo_last_error names the
 *     field): LVO_E_BADARG for n_scans not 16, 32 or 64, a minimum_range that is not finite or is negative, a resolution that is not
 *     finite or is <= 0 (each as the float the kernels use), skip_frame < 1, or a bad lane; LVO_E_CAPACITY for n_scans above the
 *     context's; LVO_E_STATE while an *_async step is in flight.
 *   - Stream-ordered, returns when done.  Captured CUDA graphs stay valid, and a step launches the same kernels whatever the lanes'
 *     settings. */
int lvo_lane_configure(lvo_ctx* ctx, int lane, const lvo_lane_config* cfg_or_null);
/* The settings of `lane`.  LVO_E_BADARG for a bad lane or a NULL `out`. */
int lvo_lane_get_config(const lvo_ctx* ctx, int lane, lvo_lane_config* out);

/* ---- lane snapshots: checkpoint / resume, and moving a running lane to another lane, context or GPU -------- */

/* Snapshot of everything `lane` carries into its next frame: its device state (poses, map correction, cube window, lvo_stats, ...),
 * the odometry "last" clouds, the current map with its cube offset tables, its skip_frame phase and lvo_lane_status, and as a
 * fingerprint the settings it ran with (the lane's lvo_lane_config, the context's solver settings).  Per-frame
 * intermediates (probes, the registered cloud) are not included.  The format is versioned and documented in DESIGN.md §3; it holds
 * no lane index, device or pointer, so two lanes that ran the same sequence give the same bytes.  `dst` may be host memory
 * (pageable or pinned) or device memory of any device.  dst == NULL or cap too small: LVO_E_CAPACITY with *n_bytes = the size
 * needed (n_bytes may be NULL).  Changes nothing; synchronous on return.  LVO_E_STATE while an *_async step is in flight,
 * LVO_E_BADARG for a bad lane. */
int lvo_lane_save(lvo_ctx* ctx, int lane, void* dst, size_t cap, size_t* n_bytes);
/* Replace the state of `lane` with a snapshot (host or device memory, any device): its next active step continues the saved
 * sequence exactly as the source lane would have.  The destination may be any lane of any context whose lane settings (n_scans,
 * minimum_range, line_res, plane_res, skip_frame: lvo_lane_get_config) and context settings (outer_iters, lm_max_iters, huber,
 * distortion) equal the source's (else LVO_E_BADARG, and lvo_last_error names the field).  The load does not change the lane's
 * settings: to move a 16-beam lane into a lane of a 64-beam context, lvo_lane_configure that lane first.  Its capacities may differ as long as the saved clouds and map, and the point counts of the
 * lane's last frame, fit (else LVO_E_CAPACITY).  The snapshot is checked in full before anything is written: a malformed one
 * returns LVO_E_BADARG and leaves the lane as it was.
 * lvo_get_stats, lvo_lane_status, lvo_map_export, lvo_map_cloud and lvo_get_map_correction report the snapshot at once;
 * lvo_probe_fetch of the lane returns LVO_E_STATE for a probe until the stage that writes it has run for the lane: extraction and
 * odometry probes until its next active frame (or lvo_extract_features / lvo_scan_to_scan), LVO_P_MAP_* and LVO_P_REGISTERED until
 * its next mapping frame (or lvo_scan_to_map).  The
 * lane's activity is unchanged.  The next lvo_step_batch* / lvo_scan_to_scan call first rebuilds the odometry search grids of the
 * context once, however many lanes were loaded.  Synchronous on return; LVO_E_STATE while an *_async step is in flight, LVO_E_BADARG
 * for a bad lane.  Captured CUDA graphs stay valid. */
int lvo_lane_load(lvo_ctx* ctx, int lane, const void* src, size_t n_bytes);

/* ---- state export / import (start from a pre-filled map; exact checkpoint / resume: lvo_lane_save / lvo_lane_load) */

/* Replace the map of `lane` with the given cubes.  cube_ind[i] is the reference's array index
 * i + 21*j + 441*k (laserMapping.cpp:522) of point i; points of one cube keep their relative order. */
int lvo_map_import(lvo_ctx* ctx, int lane, const lvo_point* corner, const int* corner_cube, size_t n_corner,
                   const lvo_point* surf, const int* surf_cube, size_t n_surf);
/* which: 0 = corner, 1 = surf.  Points are returned cube-major in array-index order; cube_out may be NULL. */
int lvo_map_export(lvo_ctx* ctx, int lane, int which, lvo_cloud_out* pts, int* cube_out);
/* Map outputs of laserMapping.cpp:806-836.  which: 0 = "surround" cloud (:806-815: the cubes of the last frame's valid list in
 * i,j,k loop order, corner points then surf points of each cube), 1 = whole map (:823-836: all 4851 cubes in array order, corner
 * then surf).  The reference publishes them every 5th / 20th mapping frame; the schedule is the caller's (host/lvo_handlers.hpp).
 * Synchronous; runs the kernels of lvo_map_cloud_batch for one lane, in the arena of those calls, and leaves
 * lvo_timings::kernel_launches as it was.  n > cap, or data == NULL with n > 0: LVO_E_CAPACITY with pts->n = n. */
int lvo_map_cloud(lvo_ctx* ctx, int lane, int which, lvo_cloud_out* pts);

/* Map outputs of every lane of the context in one call: what the reference's mapping node publishes besides the pose. */
#define LVO_MAP_SURROUND 0   /* as lvo_map_cloud which = 0: /laser_cloud_surround, laserMapping.cpp:806-815              */
#define LVO_MAP_WHOLE 1      /* as lvo_map_cloud which = 1: /laser_cloud_map, :823-836                                   */
#define LVO_MAP_REGISTERED 2 /* registered full-resolution cloud of the last step: /velodyne_cloud_registered, :838-842    */
/* outs[l] is lane l's output, for every lane of the context.
 *   - Lane selection.  outs[l].n is written for every lane.  Points are copied only for lanes whose outs[l].data is non-NULL; a call
 *     whose destinations are all NULL is a size query (which = 0 / 1: one launch; which = 2: none).  So a caller can keep the
 *     reference's 5th / 20th-frame schedule for each lane.
 *   - LVO_MAP_SURROUND / LVO_MAP_WHOLE: every lane, active or idle, gets exactly the points, in the same order, that
 *     lvo_map_cloud(ctx, l, which, ...) returns, from the current map.  A freshly created or reset lane has an empty map (n = 0); a
 *     lane loaded with lvo_lane_load gets its snapshot's map at once.
 *   - LVO_MAP_REGISTERED reports the lanes that mapped in the last lvo_step_batch* call: each gets the n_kept points of that frame
 *     moved into the map frame, bit for bit what lvo_probe_fetch(LVO_P_REGISTERED) returns right after that step.  Every other lane
 *     gets n = 0 and its destination is not written: lanes that did not map (off their skip_frame phase or idle), and lanes reset or
 *     loaded since the step.  The counts are recorded on the host when the step completes.  lvo_scan_to_map, lvo_knn and
 *     lvo_depth_associate overwrite the registered clouds; after any of them which = 2 returns LVO_E_STATE (lvo_last_error says
 *     why) until the next lvo_step_batch* call completes.
 *   - Errors, each checked before any destination is written: LVO_E_BADARG for a NULL array or a bad `which`; LVO_E_STATE while an
 *     *_async step is in flight, or after the invalidation above; LVO_E_CAPACITY when a selected lane's cap is below its n (every n
 *     is still written, and no point is copied for any lane).
 *   - Synchronous on return, on the context's stream (lvo_set_stream).  which = 0 / 1 count the lanes' clouds in one launch and copy
 *     them in a second one; one small device-to-host copy of the per-lane totals between the two is the only synchronisation inside
 *     the call.  which = 2 is one launch.  These launch counts do not depend on the number of lanes (lvo_timings::kernel_launches
 *     reports them).  The host form gathers the selected clouds back to back on the device and copies each to its buffer once.
 *   - The calls use their own device arena: per-lane descriptors, offset tables and totals, allocated on the first call, and a point
 *     buffer on the device that grows, never shrinks, when a host-form call brings more points; lvo_destroy frees it.
 *     They read and write no state of the step: lane states, maps, probes, staging buffers, the prefetch of
 *     lvo_step_batch_pipelined and captured CUDA graphs are left as they were. */
int lvo_map_cloud_batch(lvo_ctx* ctx, int which, lvo_cloud_out* outs);
/* Same, into device memory of the context's device: d_out[l] (NULL = lane not copied) holds cap[l] points; n_out[l] gets every
 * lane's count.  The arena's point buffer is neither allocated nor used by this form. */
int lvo_map_cloud_batch_dev(lvo_ctx* ctx, int which, lvo_point* const* d_out, const size_t* cap, size_t* n_out);
/* (q_wmap_wodom, t_wmap_wodom), laserMapping.cpp:116-117 */
int lvo_get_map_correction(lvo_ctx* ctx, int lane, lvo_pose* T_wmap_wodom);
int lvo_set_map_correction(lvo_ctx* ctx, int lane, const lvo_pose* T_wmap_wodom);
/* (para_q, para_t) and (q_w_curr, t_w_curr) of the odometry stage */
int lvo_set_odometry_state(lvo_ctx* ctx, int lane, const lvo_pose* T_last_curr, const lvo_pose* T_w_curr);

/* ---- parity probes: copy an intermediate device array of `lane` to host ----------------------------------- */
enum lvo_probe {
  LVO_P_FULL = 0,          /* lvo_point[n_kept]  ring-ordered cloud                       scanRegistration.cpp:246-252 */
  LVO_P_CURVATURE = 1,     /* float[n_kept]      cloudCurvature                           :262                        */
  LVO_P_SORT_IND = 2,      /* int[n_kept]        cloudSortInd after all sector sorts      :288                        */
  LVO_P_LABEL = 3,         /* int[n_kept]        cloudLabel                               :303,309,355                */
  LVO_P_PICKED = 4,        /* int[n_kept]        cloudNeighborPicked                      :317-342                    */
  LVO_P_SCAN_START = 5,    /* int[n_scans]       scanStartInd (the lane's n_scans)        :249                        */
  LVO_P_SCAN_END = 6,      /* int[n_scans]       scanEndInd (the lane's n_scans)          :251                        */
  LVO_P_SHARP = 7, LVO_P_LESS_SHARP = 8, LVO_P_FLAT = 9, LVO_P_LESS_FLAT = 10, /* lvo_point[]                          */
  LVO_P_ODO_CORNER_CORR = 11, /* int[outer][n_sharp][2]  (closestPointInd, minPointInd2) or -1  laserOdometry.cpp:388-442 */
  LVO_P_ODO_PLANE_CORR = 12,  /* int[outer][n_flat][3]   (closest, minPointInd2, minPointInd3)   :472-534             */
  LVO_P_ODO_LM_TRACE = 13,    /* double[outer][lm_max_iters+1][10]: x(7), cost, radius, flags    ceres::Solve :576    */
  LVO_P_MAP_CORNER_STACK = 14, LVO_P_MAP_SURF_STACK = 15, /* lvo_point[]                         laserMapping.cpp:542-550 */
  LVO_P_MAP_CORNER_FROM_MAP = 16, LVO_P_MAP_SURF_FROM_MAP = 17, /* lvo_point[] in gather order    :531-537             */
  LVO_P_MAP_CORNER_KNN = 18,  /* int[outer][n_corner_stack][5], -1 row if d5^2 >= 1.0             :582-584             */
  LVO_P_MAP_SURF_KNN = 19,    /* int[outer][n_surf_stack][5]                                      :648-652             */
  LVO_P_MAP_CORNER_VALID = 20,/* int[outer][n_corner_stack]  1 if an edge factor was added        :611                 */
  LVO_P_MAP_SURF_VALID = 21,  /* int[outer][n_surf_stack]    1 if a plane factor was added        :681                 */
  LVO_P_MAP_LM_TRACE = 22,    /* as LVO_P_ODO_LM_TRACE                                            ceres::Solve :720    */
  LVO_P_REGISTERED = 23       /* lvo_point[n_kept]                                                :838-842             */
};
/* Copies up to cap_bytes; *n_bytes gets the full size (so a too-small buffer can be detected). */
int lvo_probe_fetch(lvo_ctx* ctx, int lane, int what, void* out, size_t cap_bytes, size_t* n_bytes);

/* Stand-alone operators (used by parity tests and by bench.py's per-kernel roofline; lane 0 scratch). */
/* TransformToStart (to_end = 0, laserOdometry.cpp:154-172) / TransformToEnd (to_end = 1, :176-191) of a cloud under T_last_curr
 * (NULL = lane 0's current para_q / para_t) with the context's distortion mode (to_end always interpolates, as :176-191 does
 * whenever its block is enabled).  In distortion mode 2 a host that drives the three entry points separately uses it to obtain
 * the full-resolution cloud that :610-625 would publish. */
int lvo_transform_cloud(lvo_ctx* ctx, lvo_cloud_view in, const lvo_pose* T_last_curr_or_null, int to_end, lvo_cloud_out* out);
/* pcl::VoxelGrid::filter restated (scanRegistration.cpp:401-405, laserMapping.cpp:543-549,793-799). */
int lvo_voxel_downsample(lvo_ctx* ctx, lvo_cloud_view in, float leaf, lvo_cloud_out* out);
/* Device-resident form for kernel measurements: d_in / d_out are device pointers (packed points, d_out capacity >= n);
 * *ms gets the CUDA-event time of the downsample kernels alone (no copies). */
int lvo_voxel_downsample_dev(lvo_ctx* ctx, const lvo_point* d_in, size_t n, float leaf, lvo_point* d_out, size_t* n_out, float* ms);
/* Exact K-NN (K<=5) of queries in cloud, squared-distance gate `max_sq`; ind/sq are [nq][K]; -1 when fewer
 * than K points lie inside the gate.  Replaces pcl::KdTreeFLANN::nearestKSearch + the d^2 gate
 * (laserMapping.cpp:582-584; laserOdometry.cpp:386-389). */
int lvo_knn(lvo_ctx* ctx, lvo_cloud_view cloud, lvo_cloud_view queries, int K, float max_sq, int* ind, float* sq);

/* Camera-lidar depth association (BASELINE config 5; reference src/vloam/Frame.cpp:289-352 + src/vloam/Frontend.cpp:223-301).
 * The sweep is moved into the camera frame by the 3x4 extrinsic, every point with z > 0 becomes a depth-cloud point
 * (10 x/z, 10 y/z, 10, intensity = z); each keypoint (normalised coordinates u = (px - cx)/fx, v = (py - cy)/fy) gets the
 * depth of the plane through its 3 nearest depth-cloud points when the nearest lies within d^2 < 0.5, with the reference's
 * clamps.  depth_out / valid_out are [n_kp]; nn_out (optional) is [n_kp][3] indices into the depth cloud (-1 if rejected). */
typedef struct lvo_camera { float fx, fy, cx, cy; int width, height; float extrinsic[12]; /* row-major 3x4 lidar -> camera */ } lvo_camera;
int lvo_depth_associate(lvo_ctx* ctx, lvo_cloud_view sweep, const lvo_camera* cam, const float* keypoints_uv, size_t n_kp, float* depth_out,
                        int* valid_out, int* nn_out, lvo_cloud_out* depth_cloud_or_null);

/* Depth association for every active lane of the context in one call (a fleet of lidar-visual front ends).  Lane l gets, bit for
 * bit, what lvo_depth_associate(sweeps[l], &cams[l], keypoints_uv[l], n_kp[l], ...) returns: depth_out[l] / valid_out[l] are
 * [n_kp[l]], nn_out_or_null[l] is [n_kp[l]][3] indices into that lane's depth cloud.  Only cams[l].extrinsic is read, and no
 * lane's result depends on another lane's inputs.  Idle lanes (lvo_set_lane_active) are skipped: none of their entries is read or
 * written, and they may be NULL / 0.
 *   - Sweep views follow lvo_step_batch: one layout for all active lanes, stride <= 32, packed 12-byte x, y, z records allowed.
 *   - Limits of the single call: n <= max_points and 2 n_kp <= max_points (LVO_E_CAPACITY).  NULL arrays, or a NULL keypoint /
 *     output pointer of an active lane with n_kp > 0: LVO_E_BADARG.  nn_out_or_null may be NULL as a whole.  LVO_E_STATE while an
 *     *_async step is in flight.  All of this is checked before anything is enqueued; on an error no output is written.
 *   - Synchronous on return, on the context's stream (lvo_set_stream).  One launch sequence for all lanes; its length does not
 *     depend on the number of lanes or keypoints.
 *   - The calls use their own device arena, allocated on the first call and grown when a call brings more points, keypoints or
 *     lanes (freed by lvo_destroy).  They read and write no state of the step: lane states, maps, probes, staging buffers, the
 *     prefetch of lvo_step_batch_pipelined and captured CUDA graphs are left as they were.
 * No depth cloud is returned; lvo_depth_associate remains the way to get one. */
int lvo_depth_associate_batch(lvo_ctx* ctx, const lvo_camera* cams, const lvo_cloud_view* sweeps, const float* const* keypoints_uv,
                              const size_t* n_kp, float* const* depth_out, int* const* valid_out, int* const* nn_out_or_null);
/* Same, with sweeps (packed lvo_point, n[l] points), keypoints and outputs in device memory of the context's device. */
int lvo_depth_associate_batch_dev(lvo_ctx* ctx, const lvo_camera* cams, const lvo_point* const* d_sweeps, const size_t* n,
                                  const float* const* d_keypoints_uv, const size_t* n_kp, float* const* d_depth_out, int* const* d_valid_out,
                                  int* const* d_nn_out_or_null);

/* Throughput-mode 5-NN benchmark entry (SURVEY §8d): S independent (map, query) problems in ONE launch.
 * d_maps / d_queries are device pointers to packed points, problems laid out back to back with the given
 * per-problem counts.  Builds the cell grids (untimed part) on first call with build != 0, then runs the search
 * kernel `reps` times; returns the average kernel milliseconds in *ms (CUDA events on the ctx stream). */
int lvo_knn5_throughput(lvo_ctx* ctx, const lvo_point* d_maps, const int* map_counts, const lvo_point* d_queries,
                        const int* query_counts, int S, int reps, int* d_ind_out, float* d_sq_out, float* ms);

/* ---- timing: the reference's TicToc stage names (SURVEY §5), CUDA-event milliseconds of the last call ------ */
typedef struct lvo_timings {
  float extract_ms;       /* "scan registration time"   scanRegistration.cpp:456 */
  float odometry_ms;      /* "whole laserOdometry time" laserOdometry.cpp:665    */
  float mapping_ms;       /* "whole mapping time"       laserMapping.cpp:852     */
  float knn_ms;           /* sum of the 5-NN kernels of the last scan-to-map call */
  int knn_launches;
  int kernel_launches;    /* kernels launched by the last call (for bench.py's gpu_launches) */
  double knn_bytes;       /* algorithmic bytes of those 5-NN launches: 16 M + 56 Q each (SURVEY §8d) */
  /* sub-stages under the reference's TicToc printf names (CUDA events between the kernels of plain-launch calls; 0 when the frame
   * was replayed from a CUDA graph or LVO_OPT_STAGE_TIMING is off).  Per-iteration stages are summed over the outer iterations. */
  float reg_prepare_ms;      /* "prepare time"                    scanRegistration.cpp:254 : filter, ring ids, ring concat, curvature */
  float reg_sort_ms;         /* "sort q time"                     :409 : the sector sorts                                             */
  float reg_separate_ms;     /* "seperate points time"            :410 : picks, less-flat voxel filter, compaction (excl. the sorts)  */
  float odo_association_ms;  /* "data association time"           laserOdometry.cpp:564                                               */
  float odo_solver_ms;       /* "solver time"                     :577                                                                */
  float odo_rest_ms;         /* pose integration, cloud swap, kd-tree (grid) rebuild  :581-641 ("publication time" :664 has no analogue) */
  float map_prepare_ms;      /* "map prepare time"                laserMapping.cpp:552 : cube window, 75-cube gather, stack downsample */
  float map_build_tree_ms;   /* "build tree time"                 :560 : the two search grids                                         */
  float map_association_ms;  /* "mapping data assosiation time"   :710 : 5-NN (= knn_ms) + line / plane fits                          */
  float map_solver_ms;       /* "mapping solver time"             :721                                                                */
  float map_optimization_ms; /* "mapping optimization time"       :728 : association + solver of all outer iterations                 */
  float map_add_points_ms;   /* "add points time"                 :784 : transformUpdate + insertion keys                             */
  float map_filter_ms;       /* "filter time"                     :802 : per-cube re-filter + map rebuild                             */
  float map_pub_ms;          /* "mapping pub time"                :850 : the registered cloud                                         */
} lvo_timings;
int lvo_get_timings(const lvo_ctx* ctx, lvo_timings* out);
/* Enqueue all work of this context on a caller-owned CUDA stream (a cudaStream_t passed as void*; NULL restores the
 * context's own stream).  Lets a harness bracket calls with its own CUDA events on the launching stream. */
int lvo_set_stream(lvo_ctx* ctx, void* cuda_stream);
/* Options.  LVO_OPT_GRAPHS: 1 = replay the per-frame launch sequence of lvo_step_batch* from a CUDA graph (captured once per
 * mapping-on/off state and map generation; all data-dependent sizes live on the device, so the sequence is static),
 * 0 = plain launches (needed for the per-kernel timings of lvo_get_timings), -1 = automatic: graphs when lanes <= 8. */
#define LVO_OPT_GRAPHS 1
/* LVO_OPT_FIXPOINT_SKIP (default 1).  The reference runs a fixed number of outer iterations (laserOdometry.cpp:364,
 * laserMapping.cpp:562), each a function of (pose, clouds) only: a fresh ceres::Problem, correspondences recomputed from the
 * pose.  When an outer iteration returns the pose BIT FOR BIT unchanged (Ceres stopped on a tolerance and discarded its
 * candidate, SURVEY A19), every remaining iteration of that frame has identical inputs and therefore identical outputs; with
 * 1 the kernels of those iterations return immediately for that lane, with 0 they run.  Poses, maps, statuses and lvo_stats
 * are bitwise the same either way (tests/test_gpu_mapping.py::test_fixpoint_skip_is_bitwise_identical); the per-iteration
 * probes of skipped iterations are filled from the last iteration that ran. */
#define LVO_OPT_FIXPOINT_SKIP 2
/* LVO_OPT_STAGE_TIMING (default 1): record the sub-stage CUDA events of lvo_timings in plain-launch lvo_step_batch* calls (~100
 * cudaEventRecord per frame); 0 = only the three whole-stage times.  The three per-stage entry points always record them. */
#define LVO_OPT_STAGE_TIMING 3
/* Option 4 selected a 5-NN map search that has been removed; the value is not reused, and lvo_set_option returns LVO_E_BADARG for it. */
/* LVO_OPT_KNN_REUSE (default 1).  The outer iterations of lvo_scan_to_map
 * (laserMapping.cpp:562) search the same map from a pose that barely moves.  With 1, a full 5-NN search also records a guard radius
 * (a lower bound on the distance to every point outside the neighbour set); a later iteration whose query moved by less than the
 * slack re-ranks the five known neighbours instead of searching, and a query whose row is unchanged keeps its line / plane fit.
 * The certificate is conservative, so index sets, factors and poses are bitwise those of searching every time
 * (tests/test_gpu_mapping.py::test_knn_reuse_is_bitwise_identical); 0 = search and fit every query in every iteration. */
#define LVO_OPT_KNN_REUSE 5
/* LVO_OPT_ODO_REUSE (default 1).  The same idea for lvo_scan_to_scan (laserOdometry.cpp:364):
 * a feature's factor depends only on WHICH points of the previous sweep were chosen (closest point, same-ring and adjacent-ring
 * partners, :386-440 / :470-532).  A full association also records guard radii for its three searches; in a later outer iteration
 * a feature whose three points are certified still to be the strict minima keeps its factor record and is not searched again.
 * Correspondences, factors and poses are bitwise those of searching every time
 * (tests/test_gpu_odometry.py::test_odo_reuse_is_bitwise_identical); 0 = associate every feature in every iteration. */
#define LVO_OPT_ODO_REUSE 6
int lvo_set_option(lvo_ctx* ctx, int option, int value);
/* Bytes copied device->host per lane at the end of every synchronous call (poses, counters, status). */
size_t lvo_state_bytes(void);

#ifdef __cplusplus
}
#endif
#endif /* LVO_H_ */
