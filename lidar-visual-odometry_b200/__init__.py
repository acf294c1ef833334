"""lvo_b200 — thin ctypes binding of liblvo.so (include/lvo.h), used by tests/, bench.py and __graft_entry__.py.

The product is the C-ABI shared library built from csrc/ (hand-written sm_100a CUDA); host code that embeds it is
C++ (host/lvo_handlers.hpp mirrors the reference's three handler bodies).  This module only marshals numpy arrays
across that ABI.  There is no CPU fallback: `Lvo(...)` raises if liblvo.so is missing or no B200 is visible.

The directory name contains a hyphen, so import it with `importlib` (see tests/conftest.py: `load_lvo()`).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LVO_LIB_PATH") or os.path.join(HERE, "liblvo.so")  # LVO_LIB_PATH: another BUILD of the same library (A/B timing)

LVO_OK, LVO_E_BADARG, LVO_E_CAPACITY, LVO_E_CUDA, LVO_E_STATE = 0, -1, -2, -3, -4
LVO_W_FIRST_FRAME, LVO_W_FEW_CORR, LVO_W_MAP_TOO_SMALL = 1, 2, 3
LVO_OPT_GRAPHS = 1
LVO_OPT_FIXPOINT_SKIP = 2
LVO_OPT_STAGE_TIMING = 3
LVO_OPT_KNN_REUSE = 5
LVO_OPT_ODO_REUSE = 6
LVO_MAP_SURROUND, LVO_MAP_WHOLE, LVO_MAP_REGISTERED = 0, 1, 2

# enum lvo_probe
(P_FULL, P_CURVATURE, P_SORT_IND, P_LABEL, P_PICKED, P_SCAN_START, P_SCAN_END, P_SHARP, P_LESS_SHARP, P_FLAT, P_LESS_FLAT,
 P_ODO_CORNER_CORR, P_ODO_PLANE_CORR, P_ODO_LM_TRACE, P_MAP_CORNER_STACK, P_MAP_SURF_STACK, P_MAP_CORNER_FROM_MAP,
 P_MAP_SURF_FROM_MAP, P_MAP_CORNER_KNN, P_MAP_SURF_KNN, P_MAP_CORNER_VALID, P_MAP_SURF_VALID, P_MAP_LM_TRACE, P_REGISTERED) = range(24)


class CloudView(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n", C.c_size_t), ("stride", C.c_size_t), ("off_xyz", C.c_size_t), ("off_intensity", C.c_size_t)]


class CloudOut(C.Structure):
    _fields_ = [("data", C.c_void_p), ("cap", C.c_size_t), ("n", C.c_size_t)]


class Pose(C.Structure):
    _fields_ = [("q", C.c_double * 4), ("t", C.c_double * 3)]


class Config(C.Structure):
    _fields_ = [("n_scans", C.c_int), ("minimum_range", C.c_double), ("line_res", C.c_double), ("plane_res", C.c_double),
                ("skip_frame", C.c_int), ("outer_iters", C.c_int), ("lm_max_iters", C.c_int), ("huber", C.c_double), ("device", C.c_int),
                ("lanes", C.c_int), ("max_points", C.c_int), ("max_map_corner", C.c_int), ("max_map_surf", C.c_int), ("distortion", C.c_int), ("debug_probes", C.c_int)]


class LaneConfig(C.Structure):
    """lvo_lane_config: the per-sensor launch parameters of one lane."""
    _fields_ = [("n_scans", C.c_int), ("minimum_range", C.c_double), ("line_res", C.c_double), ("plane_res", C.c_double), ("skip_frame", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("n_in", C.c_int), ("n_kept", C.c_int), ("n_sharp", C.c_int), ("n_less_sharp", C.c_int), ("n_flat", C.c_int), ("n_less_flat", C.c_int),
                ("odo_corner_corr", C.c_int * 16), ("odo_plane_corr", C.c_int * 16), ("odo_lm_iters", C.c_int * 16), ("odo_final_cost", C.c_double * 16),
                ("map_corner_from_map", C.c_int), ("map_surf_from_map", C.c_int), ("map_corner_stack", C.c_int), ("map_surf_stack", C.c_int),
                ("map_corner_corr", C.c_int * 16), ("map_surf_corr", C.c_int * 16), ("map_lm_iters", C.c_int * 16), ("map_final_cost", C.c_double * 16),
                ("map_corner_total", C.c_int), ("map_surf_total", C.c_int), ("center_cube", C.c_int * 3), ("cen", C.c_int * 3),
                ("odo_outer_executed", C.c_int), ("map_outer_executed", C.c_int), ("map_knn_full", C.c_int * 16), ("odo_slow", C.c_int * 16), ("odo_slow_why", C.c_int * 6), ("odo_certified", C.c_int * 16)]


class Camera(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float), ("width", C.c_int), ("height", C.c_int), ("extrinsic", C.c_float * 12)]


# params/KITTI00.yaml:4-10,27-33 of the reference
KITTI00_CAMERA = dict(fx=718.856, fy=718.856, cx=607.1928, cy=185.2157, width=1241, height=376,
                      extrinsic=[0.0004276802385584, -0.9999672484946, -0.008084491683471, -0.01198459927713,
                                 -0.007210626507497, 0.008081198471645, -0.9999413164504, -0.05403984729748,
                                 0.9999738645903, 0.0004859485810390, -0.007206933692422, -0.2921968648686])


# sub-stage fields of lvo_timings and the reference's TicToc printf they correspond to (scanRegistration.cpp:254,409,410;
# laserOdometry.cpp:564,577; laserMapping.cpp:552,560,710,721,728,784,802,850)
STAGE_FIELDS = ["reg_prepare_ms", "reg_sort_ms", "reg_separate_ms", "odo_association_ms", "odo_solver_ms", "odo_rest_ms", "map_prepare_ms",
                "map_build_tree_ms", "map_association_ms", "map_solver_ms", "map_optimization_ms", "map_add_points_ms", "map_filter_ms", "map_pub_ms"]
STAGE_NAMES = {"reg_prepare_ms": "prepare time", "reg_sort_ms": "sort q time", "reg_separate_ms": "seperate points time",
               "odo_association_ms": "data association time", "odo_solver_ms": "solver time", "odo_rest_ms": "(pose integration + kd-tree rebuild)",
               "map_prepare_ms": "map prepare time", "map_build_tree_ms": "build tree time", "map_association_ms": "mapping data assosiation time",
               "map_solver_ms": "mapping solver time", "map_optimization_ms": "mapping optimization time", "map_add_points_ms": "add points time",
               "map_filter_ms": "filter time", "map_pub_ms": "mapping pub time"}


class Timings(C.Structure):
    _fields_ = [("extract_ms", C.c_float), ("odometry_ms", C.c_float), ("mapping_ms", C.c_float), ("knn_ms", C.c_float), ("knn_launches", C.c_int),
                ("kernel_launches", C.c_int), ("knn_bytes", C.c_double)] + [(n, C.c_float) for n in STAGE_FIELDS]


EXPORTS = ["lvo_default_config", "lvo_create", "lvo_destroy", "lvo_last_error", "lvo_get_stats", "lvo_extract_features", "lvo_scan_to_scan",
           "lvo_scan_to_map", "lvo_step_batch", "lvo_step_batch_dev", "lvo_lane_status", "lvo_map_import", "lvo_map_export",
           "lvo_get_map_correction", "lvo_set_map_correction", "lvo_set_odometry_state", "lvo_probe_fetch", "lvo_voxel_downsample", "lvo_knn",
           "lvo_knn5_throughput", "lvo_get_timings", "lvo_set_stream", "lvo_state_bytes", "lvo_depth_associate", "lvo_step_batch_pipelined", "lvo_set_option", "lvo_voxel_downsample_dev",
           "lvo_map_cloud", "lvo_transform_cloud", "lvo_step_batch_async", "lvo_step_batch_dev_async", "lvo_wait", "lvo_set_lane_active",
           "lvo_lane_reset", "lvo_lane_save", "lvo_lane_load", "lvo_depth_associate_batch", "lvo_depth_associate_batch_dev",
           "lvo_map_cloud_batch", "lvo_map_cloud_batch_dev", "lvo_lane_configure", "lvo_lane_get_config", "lvo_set_lane_map_update"]


def load_library():
    """dlopen liblvo.so and declare the signatures.  Raises OSError when the library has not been built."""
    if not os.path.exists(LIB_PATH):
        raise OSError(f"{LIB_PATH} not built: run `make -C {HERE}` (or __graft_entry__.build())")
    L = C.CDLL(LIB_PATH)
    vp, ip = C.c_void_p, C.c_int
    L.lvo_default_config.argtypes = [C.POINTER(Config)]
    L.lvo_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.lvo_destroy.argtypes = [vp]
    L.lvo_last_error.argtypes = [vp]
    L.lvo_last_error.restype = C.c_char_p
    L.lvo_get_stats.argtypes = [vp, ip, C.POINTER(Stats), C.c_size_t]
    L.lvo_extract_features.argtypes = [vp, CloudView] + [C.POINTER(CloudOut)] * 5
    L.lvo_scan_to_scan.argtypes = [vp] + [CloudView] * 4 + [C.POINTER(Pose)] * 2
    L.lvo_scan_to_map.argtypes = [vp] + [CloudView] * 3 + [C.POINTER(Pose), C.POINTER(Pose), C.POINTER(CloudOut)]
    L.lvo_step_batch.argtypes = [vp, C.POINTER(CloudView), C.POINTER(Pose), C.POINTER(Pose)]
    L.lvo_step_batch_pipelined.argtypes = [vp, C.POINTER(CloudView), C.POINTER(CloudView), C.POINTER(Pose), C.POINTER(Pose)]
    L.lvo_step_batch_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(Pose), C.POINTER(Pose)]
    L.lvo_lane_status.argtypes = [vp, ip]
    L.lvo_step_batch_async.argtypes = [vp, C.POINTER(CloudView)]
    L.lvo_step_batch_dev_async.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.lvo_wait.argtypes = [vp, C.POINTER(Pose), C.POINTER(Pose)]
    L.lvo_set_lane_active.argtypes = [vp, ip, ip]
    L.lvo_set_lane_map_update.argtypes = [vp, ip, ip]
    L.lvo_lane_reset.argtypes = [vp, ip]
    L.lvo_lane_configure.argtypes = [vp, ip, C.POINTER(LaneConfig)]
    L.lvo_lane_get_config.argtypes = [vp, ip, C.POINTER(LaneConfig)]
    L.lvo_lane_save.argtypes = [vp, ip, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.lvo_lane_load.argtypes = [vp, ip, vp, C.c_size_t]
    L.lvo_map_import.argtypes = [vp, ip, vp, vp, C.c_size_t, vp, vp, C.c_size_t]
    L.lvo_map_export.argtypes = [vp, ip, ip, C.POINTER(CloudOut), vp]
    L.lvo_map_cloud.argtypes = [vp, ip, ip, C.POINTER(CloudOut)]
    L.lvo_map_cloud_batch.argtypes = [vp, ip, C.POINTER(CloudOut)]
    L.lvo_map_cloud_batch_dev.argtypes = [vp, ip, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.lvo_transform_cloud.argtypes = [vp, CloudView, C.POINTER(Pose), ip, C.POINTER(CloudOut)]
    L.lvo_get_map_correction.argtypes = [vp, ip, C.POINTER(Pose)]
    L.lvo_set_map_correction.argtypes = [vp, ip, C.POINTER(Pose)]
    L.lvo_set_odometry_state.argtypes = [vp, ip, C.POINTER(Pose), C.POINTER(Pose)]
    L.lvo_probe_fetch.argtypes = [vp, ip, ip, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.lvo_voxel_downsample.argtypes = [vp, CloudView, C.c_float, C.POINTER(CloudOut)]
    L.lvo_voxel_downsample_dev.argtypes = [vp, vp, C.c_size_t, C.c_float, vp, C.POINTER(C.c_size_t), C.POINTER(C.c_float)]
    L.lvo_knn.argtypes = [vp, CloudView, CloudView, ip, C.c_float, vp, vp]
    L.lvo_knn5_throughput.argtypes = [vp, vp, vp, vp, vp, ip, ip, vp, vp, C.POINTER(C.c_float)]
    L.lvo_get_timings.argtypes = [vp, C.POINTER(Timings)]
    L.lvo_set_stream.argtypes = [vp, vp]
    L.lvo_set_option.argtypes = [vp, ip, ip]
    L.lvo_state_bytes.restype = C.c_size_t
    L.lvo_depth_associate.argtypes = [vp, CloudView, C.POINTER(Camera), vp, C.c_size_t, vp, vp, vp, C.POINTER(CloudOut)]
    L.lvo_depth_associate_batch.argtypes = [vp, C.POINTER(Camera), C.POINTER(CloudView), C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(vp),
                                            C.POINTER(vp), C.POINTER(vp)]
    L.lvo_depth_associate_batch_dev.argtypes = [vp, C.POINTER(Camera), C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(vp), C.POINTER(C.c_size_t),
                                                C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    return L


def view_of(a):
    """CloudView over an (n,4) float32 array (packed lvo_point), an (n,8) float32 array (pcl::PointXYZI layout) or, for raw sweeps
    only, an (n,3) float32 array (packed x, y, z)."""
    if a is None:
        return CloudView(None, 0, 16, 0, 12), None
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] in (3, 4, 8)
    if a.shape[1] == 3:
        return CloudView(a.ctypes.data, a.shape[0], 12, 0, 0), a
    if a.shape[1] == 4:
        return CloudView(a.ctypes.data, a.shape[0], 16, 0, 12), a
    return CloudView(a.ctypes.data, a.shape[0], 32, 0, 16), a


def to_pcl_layout(a):
    """packed (n,4) -> pcl::PointXYZI records (n,8): x,y,z,1.0,intensity,pad,pad,pad"""
    a = np.asarray(a, np.float32)
    o = np.zeros((a.shape[0], 8), np.float32)
    o[:, :3] = a[:, :3]
    o[:, 3] = 1.0
    o[:, 4] = a[:, 3]
    return o


def camera_of(d=None):
    """lvo_camera from a dict like KITTI00_CAMERA (None: KITTI00_CAMERA)."""
    cd = dict(KITTI00_CAMERA if d is None else d)
    cam = Camera()
    cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height = cd["fx"], cd["fy"], cd["cx"], cd["cy"], cd["width"], cd["height"]
    for k in range(12):
        cam.extrinsic[k] = cd["extrinsic"][k]
    return cam


def pose_to_np(p):
    return np.array(list(p.q) + list(p.t), np.float64)


def np_to_pose(a):
    p = Pose()
    for k in range(4):
        p.q[k] = float(a[k])
    for k in range(3):
        p.t[k] = float(a[4 + k])
    return p


class LvoError(RuntimeError):
    pass


class Lvo:
    """One lvo_ctx."""

    def __init__(self, n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, skip_frame=1, outer_iters=10, lm_max_iters=4, huber=0.1,
                 device=0, lanes=1, max_points=0, max_map_corner=0, max_map_surf=0, distortion=0, debug_probes=1):
        """debug_probes defaults to 1 HERE (the parity tests read every outer iteration's probes); lvo_default_config and bench.py use 0."""
        self.lib = load_library()
        cfg = Config()
        self.lib.lvo_default_config(C.byref(cfg))
        cfg.n_scans, cfg.minimum_range, cfg.line_res, cfg.plane_res = n_scans, minimum_range, line_res, plane_res
        cfg.skip_frame, cfg.outer_iters, cfg.lm_max_iters, cfg.huber, cfg.device, cfg.lanes = skip_frame, outer_iters, lm_max_iters, huber, device, lanes
        cfg.max_points, cfg.max_map_corner, cfg.max_map_surf = max_points, max_map_corner, max_map_surf
        cfg.distortion = distortion
        cfg.debug_probes = debug_probes
        self.cfg = cfg
        self.h = C.c_void_p()
        r = self.lib.lvo_create(C.byref(cfg), C.byref(self.h))
        if r != LVO_OK:
            msg = self.lib.lvo_last_error(self.h).decode() if self.h else "bad config"
            if self.h:
                self.lib.lvo_destroy(self.h)
                self.h = None
            raise LvoError(f"lvo_create failed ({r}): {msg}")
        self.P = max_points or 262144
        self.lanes = lanes
        self._active = [True] * lanes

    def close(self):
        if getattr(self, "h", None):
            self.lib.lvo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, r):
        if r < 0:
            raise LvoError(f"liblvo error {r}: {self.lib.lvo_last_error(self.h).decode()}")
        return r

    def _out(self, cap):
        buf = np.empty((max(cap, 1), 4), np.float32)
        return CloudOut(buf.ctypes.data, cap, 0), buf

    # ---- the three drop-in entry points
    def extract_features(self, sweep):
        v, keep = view_of(sweep)
        ncap = max(v.n, 1)
        outs = [self._out(ncap) for _ in range(5)]
        r = self._check(self.lib.lvo_extract_features(self.h, v, *[C.byref(o[0]) for o in outs]))
        names = ["full", "sharp", "less_sharp", "flat", "less_flat"]
        return r, {k: o[1][:o[0].n].copy() for k, o in zip(names, outs)}

    def scan_to_scan(self, sharp, less_sharp, flat, less_flat):
        vs = [view_of(a) for a in (sharp, less_sharp, flat, less_flat)]
        p1, p2 = Pose(), Pose()
        r = self._check(self.lib.lvo_scan_to_scan(self.h, *[v[0] for v in vs], C.byref(p1), C.byref(p2)))
        return r, pose_to_np(p1), pose_to_np(p2)

    def scan_to_map(self, corner_last, surf_last, full, odom7, want_registered=False):
        vs = [view_of(a) for a in (corner_last, surf_last, full)]
        pin, pout = np_to_pose(odom7), Pose()
        reg = self._out(vs[2][0].n) if (want_registered and full is not None) else None
        r = self._check(self.lib.lvo_scan_to_map(self.h, *[v[0] for v in vs], C.byref(pin), C.byref(pout), C.byref(reg[0]) if reg else None))
        return r, pose_to_np(pout), (reg[1][:reg[0].n].copy() if reg else None)

    # ---- batched device-resident pipeline.  sweeps[l] may be None for an idle lane (set_lane_active); its pose rows come back NaN.
    def _poses(self):
        """Pose arrays for one step over NaN-filled numpy buffers (the library does not write the entries of idle lanes).  Filled
        and read back as whole arrays: a per-pose Python loop would cost the timing loops of bench.py host time on every step."""
        return tuple((Pose * self.lanes).from_buffer(np.full((self.lanes, 7), np.nan)) for _ in range(2))

    @staticmethod
    def _rows(po, pm):
        return tuple(np.frombuffer(p, np.float64).reshape(-1, 7).copy() for p in (po, pm))

    def step_batch(self, sweeps):
        views = [view_of(s) for s in sweeps]
        arr = (CloudView * self.lanes)(*[v[0] for v in views])
        po, pm = self._poses()
        r = self._check(self.lib.lvo_step_batch(self.h, arr, po, pm))
        return (r,) + self._rows(po, pm)

    def step_batch_async(self, sweeps):
        """Enqueue one frame and return; the arrays must stay alive and unchanged until wait()."""
        self._async_keep = [view_of(s) for s in sweeps]
        arr = (CloudView * self.lanes)(*[v[0] for v in self._async_keep])
        return self._check(self.lib.lvo_step_batch_async(self.h, arr))

    def wait(self):
        po, pm = self._poses()
        r = self._check(self.lib.lvo_wait(self.h, po, pm))
        self._async_keep = None
        return (r,) + self._rows(po, pm)

    def stage_timings(self):
        """{reference TicToc name: milliseconds} of the last plain-launch call, plus the three whole-stage times."""
        t = self.timings()
        d = {STAGE_NAMES[f]: float(getattr(t, f)) for f in STAGE_FIELDS}
        d.update({"scan registration time": float(t.extract_ms), "whole laserOdometry time": float(t.odometry_ms), "whole mapping time": float(t.mapping_ms)})
        return d

    def step_batch_pipelined(self, sweeps, next_sweeps=None):
        """Like step_batch, but uploads next_sweeps on a copy stream while this frame computes.  The arrays of next_sweeps
        must be kept alive and unchanged by the caller until the next call (they are handed over by pointer)."""
        views = [view_of(s) for s in sweeps]
        arr = (CloudView * self.lanes)(*[v[0] for v in views])
        nxt = None
        if next_sweeps is not None:
            nviews = [view_of(s) for s in next_sweeps]
            nxt = (CloudView * self.lanes)(*[v[0] for v in nviews])
        po, pm = self._poses()
        r = self._check(self.lib.lvo_step_batch_pipelined(self.h, arr, nxt, po, pm))
        return (r,) + self._rows(po, pm)

    def step_batch_dev(self, dev_ptrs, counts):
        """dev_ptrs[l] / counts[l] may be None for an idle lane."""
        ptrs = (C.c_void_p * self.lanes)(*[int(p or 0) for p in dev_ptrs])
        ns = (C.c_size_t * self.lanes)(*[int(n or 0) for n in counts])
        po, pm = self._poses()
        r = self._check(self.lib.lvo_step_batch_dev(self.h, ptrs, ns, po, pm))
        return (r,) + self._rows(po, pm)

    def lane_status(self, lane):
        return self.lib.lvo_lane_status(self.h, lane)

    # ---- per-lane lifecycle
    def set_lane_active(self, lane, active):
        """An idle lane is skipped by every step (its sweep may be None) and resumes its sequence bit for bit."""
        self._check(self.lib.lvo_set_lane_active(self.h, lane, int(bool(active))))
        self._active[lane] = bool(active)

    def set_lane_map_update(self, lane, update):
        """update=False: the lane localises in its map (insertion and re-filter skipped, only the cube-window shift changes it);
        True (the default) maps as the reference does.  Takes effect from the next mapping frame."""
        self._check(self.lib.lvo_set_lane_map_update(self.h, lane, int(bool(update))))

    def lane_reset(self, lane):
        """Return `lane` to the first-frame state of a new context (empty map, identity poses, skip_frame phase 0)."""
        self._check(self.lib.lvo_lane_reset(self.h, lane))

    LANE_FIELDS = ("n_scans", "minimum_range", "line_res", "plane_res", "skip_frame")

    def lane_configure(self, lane, n_scans=None, minimum_range=None, line_res=None, plane_res=None, skip_frame=None):
        """Start a new sequence in `lane` with these sensor settings (lvo_lane_configure); None means the context's value."""
        given = dict(n_scans=n_scans, minimum_range=minimum_range, line_res=line_res, plane_res=plane_res, skip_frame=skip_frame)
        if all(v is None for v in given.values()):
            self._check(self.lib.lvo_lane_configure(self.h, lane, None))
            return
        cfg = LaneConfig(**{f: getattr(self.cfg, f) if v is None else v for f, v in given.items()})
        self._check(self.lib.lvo_lane_configure(self.h, lane, C.byref(cfg)))

    def lane_config(self, lane):
        """The sensor settings of `lane` as a dict (lvo_lane_get_config)."""
        cfg = LaneConfig()
        self._check(self.lib.lvo_lane_get_config(self.h, lane, C.byref(cfg)))
        return {f: getattr(cfg, f) for f in self.LANE_FIELDS}

    def lane_save(self, lane):
        """Snapshot of `lane` (lvo_lane_save) as a uint8 array: write it to disk, or lane_load it into any lane of a context with the
        same settings."""
        n = C.c_size_t(0)
        r = self.lib.lvo_lane_save(self.h, lane, None, 0, C.byref(n))
        if r != LVO_E_CAPACITY:
            self._check(r)
        buf = np.empty(n.value, np.uint8)
        self._check(self.lib.lvo_lane_save(self.h, lane, buf.ctypes.data, buf.nbytes, C.byref(n)))
        return buf

    def lane_load(self, lane, data):
        """Continue the sequence of a lane_save snapshot (bytes or a uint8 array) in `lane`."""
        a = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data, np.uint8)
        self._check(self.lib.lvo_lane_load(self.h, lane, a.ctypes.data, a.nbytes))

    def lane_save_dev(self, lane, ptr, cap):
        """lane_save into device memory (any device) at `ptr` with `cap` bytes; returns the snapshot's size."""
        n = C.c_size_t(0)
        self._check(self.lib.lvo_lane_save(self.h, lane, C.c_void_p(ptr), cap, C.byref(n)))
        return n.value

    def lane_load_dev(self, lane, ptr, n):
        """lane_load from device memory (any device): the snapshot's `n` bytes at `ptr`."""
        self._check(self.lib.lvo_lane_load(self.h, lane, C.c_void_p(ptr), n))

    # ---- state
    def map_import(self, lane, corner, corner_cube, surf, surf_cube):
        c = np.ascontiguousarray(corner, np.float32).reshape(-1, 4)
        s = np.ascontiguousarray(surf, np.float32).reshape(-1, 4)
        cc = np.ascontiguousarray(corner_cube, np.int32)
        sc = np.ascontiguousarray(surf_cube, np.int32)
        self._check(self.lib.lvo_map_import(self.h, lane, c.ctypes.data, cc.ctypes.data, len(c), s.ctypes.data, sc.ctypes.data, len(s)))

    def map_export(self, lane, which):
        st = self.stats(lane)
        cap = max(self.cfg.max_map_corner or (1 << 20), self.cfg.max_map_surf or (1 << 21))
        out, buf = self._out(cap)
        cube = np.empty(cap, np.int32)
        self._check(self.lib.lvo_map_export(self.h, lane, which, C.byref(out), cube.ctypes.data))
        return buf[:out.n].copy(), cube[:out.n].copy()

    def map_cloud(self, lane, which):
        """which 0: surround cloud (laserMapping.cpp:806-815), 1: whole map (:823-836)."""
        cap = (self.cfg.max_map_corner or (1 << 20)) + (self.cfg.max_map_surf or (1 << 21))
        out, buf = self._out(cap)
        self._check(self.lib.lvo_map_cloud(self.h, lane, which, C.byref(out)))
        return buf[:out.n].copy()

    def map_cloud_batch(self, which, lanes=None):
        """Map outputs of every lane in one call (lvo_map_cloud_batch).  which: LVO_MAP_SURROUND, LVO_MAP_WHOLE or LVO_MAP_REGISTERED;
        lanes: the lanes to fetch (None: all).  Returns one (n,4) float32 array per lane, None for a lane that was not requested."""
        want = set(range(self.lanes)) if lanes is None else set(lanes)
        outs = (CloudOut * self.lanes)()
        self._check(self.lib.lvo_map_cloud_batch(self.h, which, outs))   # size query: every destination NULL
        bufs = [np.empty((max(outs[l].n, 1), 4), np.float32) if l in want else None for l in range(self.lanes)]
        for l, b in enumerate(bufs):
            outs[l] = CloudOut(b.ctypes.data, len(b), 0) if b is not None else CloudOut(None, 0, 0)
        self._check(self.lib.lvo_map_cloud_batch(self.h, which, outs))
        return [b[:outs[l].n].copy() if b is not None else None for l, b in enumerate(bufs)]

    def map_cloud_batch_dev(self, which, d_out, caps):
        """Device form (lvo_map_cloud_batch_dev): d_out[l] is a device pointer (None: lane not copied) with room for caps[l] points.
        Returns every lane's point count."""
        n = (C.c_size_t * self.lanes)()
        self._check(self.lib.lvo_map_cloud_batch_dev(self.h, which, (C.c_void_p * self.lanes)(*[int(p or 0) for p in d_out]),
                                                     (C.c_size_t * self.lanes)(*[int(c or 0) for c in caps]), n))
        return list(n)

    def transform_cloud(self, pts, T_last_curr=None, to_end=False):
        """TransformToStart / TransformToEnd (laserOdometry.cpp:154-191) with the context's distortion mode."""
        v, keep = view_of(pts)
        out, buf = self._out(max(v.n, 1))
        p = np_to_pose(T_last_curr) if T_last_curr is not None else None
        self._check(self.lib.lvo_transform_cloud(self.h, v, C.byref(p) if p else None, int(to_end), C.byref(out)))
        return buf[:out.n].copy()

    def set_map_correction(self, lane, qt7):
        p = np_to_pose(qt7)
        self._check(self.lib.lvo_set_map_correction(self.h, lane, C.byref(p)))

    def get_map_correction(self, lane):
        p = Pose()
        self._check(self.lib.lvo_get_map_correction(self.h, lane, C.byref(p)))
        return pose_to_np(p)

    def set_odometry_state(self, lane, T_last_curr=None, T_w_curr=None):
        a = np_to_pose(T_last_curr) if T_last_curr is not None else None
        b = np_to_pose(T_w_curr) if T_w_curr is not None else None
        self._check(self.lib.lvo_set_odometry_state(self.h, lane, C.byref(a) if a else None, C.byref(b) if b else None))

    def set_stream(self, cuda_stream_handle):
        self._check(self.lib.lvo_set_stream(self.h, C.c_void_p(cuda_stream_handle) if cuda_stream_handle else None))

    def set_option(self, option, value):
        self._check(self.lib.lvo_set_option(self.h, option, value))

    def stats(self, lane=0):
        s = Stats()
        self._check(self.lib.lvo_get_stats(self.h, lane, C.byref(s), C.sizeof(s)))
        return s

    def timings(self):
        t = Timings()
        self._check(self.lib.lvo_get_timings(self.h, C.byref(t)))
        return t

    # ---- probes
    def probe(self, what, lane=0):
        n = C.c_size_t(0)
        self._check(self.lib.lvo_probe_fetch(self.h, lane, what, None, 0, C.byref(n)))
        buf = np.empty(max(n.value, 1), np.uint8)
        if n.value:
            self._check(self.lib.lvo_probe_fetch(self.h, lane, what, buf.ctypes.data, n.value, C.byref(n)))
        raw = buf[:n.value]
        O = self.cfg.outer_iters
        pt = lambda: raw.view(np.float32).reshape(-1, 4).copy()
        if what in (P_FULL, P_SHARP, P_LESS_SHARP, P_FLAT, P_LESS_FLAT, P_MAP_CORNER_STACK, P_MAP_SURF_STACK, P_MAP_CORNER_FROM_MAP,
                    P_MAP_SURF_FROM_MAP, P_REGISTERED):
            return pt()
        if what == P_CURVATURE:
            return raw.view(np.float32).copy()
        if what in (P_SORT_IND, P_LABEL, P_PICKED, P_SCAN_START, P_SCAN_END):
            return raw.view(np.int32).copy()
        if what == P_ODO_CORNER_CORR:
            return raw.view(np.int32).reshape(O, -1, 2).copy()
        if what == P_ODO_PLANE_CORR:
            return raw.view(np.int32).reshape(O, -1, 3).copy()
        if what in (P_ODO_LM_TRACE, P_MAP_LM_TRACE):
            return raw.view(np.float64).reshape(O, -1, 10).copy()
        if what in (P_MAP_CORNER_KNN, P_MAP_SURF_KNN):
            return raw.view(np.int32).reshape(O, -1, 5).copy()
        if what in (P_MAP_CORNER_VALID, P_MAP_SURF_VALID):
            return raw.view(np.int32).reshape(O, -1).copy()
        raise KeyError(what)

    def knn5_throughput(self, d_maps_ptr, map_counts, d_queries_ptr, query_counts, reps, d_ind_ptr, d_sq_ptr):
        """S problems in one launch (device pointers in, device outputs); returns average kernel milliseconds."""
        S = len(map_counts)
        mc = (C.c_int * S)(*[int(x) for x in map_counts])
        qc = (C.c_int * S)(*[int(x) for x in query_counts])
        ms = C.c_float(0)
        self._check(self.lib.lvo_knn5_throughput(self.h, C.c_void_p(d_maps_ptr), mc, C.c_void_p(d_queries_ptr), qc, S, reps, C.c_void_p(d_ind_ptr),
                                                 C.c_void_p(d_sq_ptr), C.byref(ms)))
        return ms.value

    def depth_associate(self, sweep, keypoints_uv, camera=None):
        """Config 5: returns (depth_cloud, depth[n], valid[n], nn[n,3])."""
        cam = Camera()
        cd = dict(KITTI00_CAMERA if camera is None else camera)
        cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height = cd["fx"], cd["fy"], cd["cx"], cd["cy"], cd["width"], cd["height"]
        for k in range(12):
            cam.extrinsic[k] = cd["extrinsic"][k]
        v, keep = view_of(sweep)
        uv = np.ascontiguousarray(keypoints_uv, np.float32).reshape(-1, 2)
        n = len(uv)
        depth = np.zeros(max(n, 1), np.float32)
        valid = np.zeros(max(n, 1), np.int32)
        nn = np.full((max(n, 1), 3), -1, np.int32)
        out, buf = self._out(max(v.n, 1))
        self._check(self.lib.lvo_depth_associate(self.h, v, C.byref(cam), uv.ctypes.data, n, depth.ctypes.data, valid.ctypes.data, nn.ctypes.data, C.byref(out)))
        return buf[:out.n].copy(), depth[:n], valid[:n], nn[:n]

    def _cameras(self, cameras):
        """cameras: None (KITTI00_CAMERA for every lane), one dict for every lane, or a per-lane list of dicts / None."""
        if cameras is None or isinstance(cameras, dict):
            cameras = [cameras] * self.lanes
        return (Camera * self.lanes)(*[camera_of(c) for c in cameras])

    def depth_associate_batch(self, sweeps, keypoints, cameras=None):
        """Depth association for every active lane in one call (lvo_depth_associate_batch).  sweeps[l]: (n,3), (n,4) or (n,8) float32, one
        layout for all active lanes; keypoints[l]: (k,2) normalised coordinates.  Returns a per-lane list of (depth[k], valid[k], nn[k,3]),
        None for idle lanes (whose entries may be None)."""
        views = [view_of(s if a else None) for s, a in zip(sweeps, self._active)]
        uvs = [np.ascontiguousarray(k, np.float32).reshape(-1, 2) if (a and k is not None) else np.zeros((0, 2), np.float32)
               for k, a in zip(keypoints, self._active)]
        outs = [(np.zeros(len(u), np.float32), np.zeros(len(u), np.int32), np.full((len(u), 3), -1, np.int32)) if a else None
                for u, a in zip(uvs, self._active)]
        ptr = lambda i, o: o[i].ctypes.data if (o is not None and len(o[i])) else None
        VP = C.c_void_p * self.lanes
        r = self.lib.lvo_depth_associate_batch(self.h, self._cameras(cameras), (CloudView * self.lanes)(*[v[0] for v in views]),
                                               VP(*[u.ctypes.data if len(u) else None for u in uvs]), (C.c_size_t * self.lanes)(*[len(u) for u in uvs]),
                                               VP(*[ptr(0, o) for o in outs]), VP(*[ptr(1, o) for o in outs]), VP(*[ptr(2, o) for o in outs]))
        self._check(r)
        return outs

    def depth_associate_batch_dev(self, d_sweeps, counts, d_keypoints, kp_counts, d_depth, d_valid, d_nn=None, cameras=None):
        """Device form (lvo_depth_associate_batch_dev): per-lane device pointers (packed lvo_point sweeps, float2 keypoints, float /
        int / int[3] outputs) and counts, None for idle lanes; d_nn may be None as a whole."""
        VP = C.c_void_p * self.lanes
        NS = C.c_size_t * self.lanes
        p = lambda xs: VP(*[int(x or 0) for x in xs])
        self._check(self.lib.lvo_depth_associate_batch_dev(self.h, self._cameras(cameras), p(d_sweeps), NS(*[int(n or 0) for n in counts]), p(d_keypoints),
                                                           NS(*[int(n or 0) for n in kp_counts]), p(d_depth), p(d_valid),
                                                           p(d_nn) if d_nn is not None else None))

    # ---- stand-alone operators
    def voxel_downsample(self, pts, leaf):
        v, keep = view_of(pts)
        out, buf = self._out(max(v.n, 1))
        self._check(self.lib.lvo_voxel_downsample(self.h, v, leaf, C.byref(out)))
        return buf[:out.n].copy()

    def voxel_downsample_dev(self, d_in_ptr, n, leaf, d_out_ptr):
        """Device pointers in / out; returns (n_out, kernel milliseconds)."""
        n_out, ms = C.c_size_t(0), C.c_float(0)
        self._check(self.lib.lvo_voxel_downsample_dev(self.h, C.c_void_p(d_in_ptr), n, leaf, C.c_void_p(d_out_ptr), C.byref(n_out), C.byref(ms)))
        return n_out.value, ms.value

    def knn(self, cloud, queries, K, max_sq):
        vc, k1 = view_of(cloud)
        vq, k2 = view_of(queries)
        ind = np.empty((max(vq.n, 1), K), np.int32)
        sq = np.empty((max(vq.n, 1), K), np.float32)
        self._check(self.lib.lvo_knn(self.h, vc, vq, K, max_sq, ind.ctypes.data, sq.ctypes.data))
        return ind[:vq.n], sq[:vq.n]
