"""ctypes bindings of the CPU oracle (oracle/liblvo_oracle.so, oracle/_ref/liblvo_oracle_ref.so) and of the synthetic
sweep generator.  TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and bench.py's CPU legs."""
import ctypes as C
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("i", "<f4")])


def _ptr(a, t=C.c_void_p):
    return a.ctypes.data_as(t) if a is not None else None


def as_pts(a):
    """(n,4) float32 view <-> contiguous array."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == 4
    return a


class Synth:
    def __init__(self):
        self.lib = C.CDLL(os.path.join(ROOT, "lidar-visual-odometry_b200", "synth", "liblvo_synth.so"))
        self.lib.lvo_synth_rays.restype = C.c_long
        self.lib.lvo_synth_sweep.restype = C.c_long
        self.lib.lvo_synth_sweep.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_long, C.c_void_p]
        self.lib.lvo_synth_sweep_moving.restype = C.c_long
        self.lib.lvo_synth_sweep_moving.argtypes = self.lib.lvo_synth_sweep.argtypes
        self.lib.lvo_synth_sweep_res.restype = C.c_long
        self.lib.lvo_synth_sweep_res.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_long, C.c_void_p]

    def sweep(self, model, seq, frame, speed=None, moving=False, naz=None):
        """moving=True: the sensor keeps moving while it spins (intra-sweep motion distortion, the DISTORTION 1 input).
        naz: azimuth columns per ring instead of the model's 1800 / 1875 (dense rings; rigid sweeps only)."""
        if speed is None:
            speed = 1.0 if model == 64 else 0.2
        out = np.empty((model * naz if naz else self.lib.lvo_synth_rays(model), 4), np.float32)
        gt = np.empty(7, np.float64)
        if naz:
            assert not moving
            n = self.lib.lvo_synth_sweep_res(model, seq, frame, speed, naz, _ptr(out), len(out), _ptr(gt))
        else:
            n = (self.lib.lvo_synth_sweep_moving if moving else self.lib.lvo_synth_sweep)(model, seq, frame, speed, _ptr(out), len(out), _ptr(gt))
        assert n >= 0
        return out[:n].copy(), gt


class Oracle:
    """One stateful pipeline (scanRegistration + laserOdometry + laserMapping restated)."""

    def __init__(self, n_scans=64, min_range=5.0, line_res=0.4, plane_res=0.8, outer=10, lm_iters=4, huber=0.1, kdtree=True,
                 reference_build=False, distortion=0):
        path = os.path.join(ROOT, "oracle", "_ref", "liblvo_oracle_ref.so") if reference_build else os.path.join(ROOT, "oracle", "liblvo_oracle.so")
        self.lib = L = C.CDLL(path)
        L.lvo_oracle_create.restype = C.c_void_p
        L.lvo_oracle_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.c_int]
        L.lvo_oracle_destroy.argtypes = [C.c_void_p]
        L.lvo_oracle_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_long]
        L.lvo_oracle_extract_get.restype = C.c_long
        L.lvo_oracle_extract_get.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_long]
        L.lvo_oracle_odometry.argtypes = [C.c_void_p] + [C.c_void_p, C.c_long] * 4 + [C.c_void_p, C.c_int]
        L.lvo_oracle_odometry_log.restype = C.c_long
        L.lvo_oracle_odometry_log.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long]
        L.lvo_oracle_mapping.argtypes = [C.c_void_p] + [C.c_void_p, C.c_long] * 3 + [C.c_void_p, C.c_void_p, C.c_int]
        L.lvo_oracle_mapping_log.restype = C.c_long
        L.lvo_oracle_mapping_log.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_long]
        L.lvo_oracle_map_export.restype = C.c_long
        L.lvo_oracle_map_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_long]
        L.lvo_oracle_map_import.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_long]
        L.lvo_oracle_set_map_correction.argtypes = [C.c_void_p, C.c_void_p]
        L.lvo_oracle_step.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p, C.c_int]
        L.lvo_oracle_timings.argtypes = [C.c_void_p, C.c_void_p]
        L.lvo_oracle_set_skip_frame.argtypes = [C.c_void_p, C.c_int]
        L.lvo_oracle_last_frame_mapped.argtypes = [C.c_void_p]
        L.lvo_oracle_voxel_grid.restype = C.c_long
        L.lvo_oracle_voxel_grid.argtypes = [C.c_void_p, C.c_long, C.c_float, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
        L.lvo_oracle_knn.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
        L.lvo_oracle_eval_factor.argtypes = [C.c_void_p] * 4
        L.lvo_oracle_solve.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int]
        L.lvo_oracle_eval_factor_s.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lvo_oracle_transform.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.lvo_oracle_set_distortion.argtypes = [C.c_void_p, C.c_int]
        L.lvo_oracle_odometry_last.restype = C.c_long
        L.lvo_oracle_odometry_last.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_long]
        L.lvo_oracle_map_cloud.restype = C.c_long
        L.lvo_oracle_map_cloud.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_long]
        L.lvo_oracle_atanf.restype = C.c_float
        L.lvo_oracle_atanf.argtypes = [C.c_float]
        L.lvo_oracle_atan2f.restype = C.c_float
        L.lvo_oracle_atan2f.argtypes = [C.c_float, C.c_float]
        L.lvo_oracle_sym_eigen3.argtypes = [C.c_void_p] * 3
        L.lvo_oracle_depth.restype = C.c_long
        L.lvo_oracle_depth.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]
        L.lvo_oracle_plane_fit5.argtypes = [C.c_void_p] * 2
        self.outer = outer
        self.h = L.lvo_oracle_create(n_scans, min_range, line_res, plane_res, outer, lm_iters, huber, 1 if kdtree else 0)
        if distortion:
            L.lvo_oracle_set_distortion(self.h, distortion)

    def __del__(self):
        try:
            self.lib.lvo_oracle_destroy(self.h)
        except Exception:
            pass

    # -- generic "fetch vector" helper
    def _get(self, fn, args, dtype, width=1):
        n = fn(self.h, *args, None, 0)
        if n < 0:
            raise KeyError(args)
        a = np.empty((n, 4), np.float32) if dtype == "pt" else np.empty(n, dtype)
        if n:
            fn(self.h, *args, _ptr(a), n)
        if dtype != "pt" and width > 1:
            a = a.reshape(-1, width)
        return a

    # -- stage 1
    def extract(self, pts):
        pts = as_pts(pts)
        r = self.lib.lvo_oracle_extract(self.h, _ptr(pts), len(pts))
        assert r == 0
        g = lambda w, dt: self._get(self.lib.lvo_oracle_extract_get, (w,), dt)
        return dict(full=g(0, "pt"), sharp=g(1, "pt"), less_sharp=g(2, "pt"), flat=g(3, "pt"), less_flat=g(4, "pt"),
                    curvature=g(10, np.float32), sort_ind=g(11, np.int32), picked=g(12, np.int32), label=g(13, np.int32),
                    scan_start=g(14, np.int32), scan_end=g(15, np.int32))

    # -- stage 2
    def odometry(self, sharp, less_sharp, flat, less_flat, keep_log=True):
        a, b, c, d = map(as_pts, (sharp, less_sharp, flat, less_flat))
        pose = np.zeros(14)
        st = self.lib.lvo_oracle_odometry(self.h, _ptr(a), len(a), _ptr(b), len(b), _ptr(c), len(c), _ptr(d), len(d), _ptr(pose), int(keep_log))
        return st, pose[:7].copy(), pose[7:].copy()

    def odometry_log(self, outer):
        f = self.lib.lvo_oracle_odometry_log
        return dict(corner_corr=self._get(f, (outer, 0), np.int32, 2), plane_corr=self._get(f, (outer, 1), np.int32, 3),
                    lm=self._get(f, (outer, 2), np.float64, 10), counts=self._get(f, (outer, 3), np.int32), cost=self._get(f, (outer, 4), np.float64))

    # -- stage 3
    def mapping(self, corner_last, surf_last, full, odom7, keep_log=True):
        a, b = as_pts(corner_last), as_pts(surf_last)
        f = as_pts(full) if full is not None else None
        odom7 = np.ascontiguousarray(odom7, np.float64)
        pose = np.zeros(14)
        st = self.lib.lvo_oracle_mapping(self.h, _ptr(a), len(a), _ptr(b), len(b), _ptr(f), 0 if f is None else len(f), _ptr(odom7), _ptr(pose), int(keep_log))
        return st, pose[:7].copy(), pose[7:].copy()

    def mapping_info(self):
        f = self.lib.lvo_oracle_mapping_log
        return dict(corner_stack=self._get(f, (0, 0), "pt"), surf_stack=self._get(f, (0, 1), "pt"), corner_from_map=self._get(f, (0, 2), "pt"),
                    surf_from_map=self._get(f, (0, 3), "pt"), registered=self._get(f, (0, 4), "pt"), info=self._get(f, (0, 5), np.int32))

    def mapping_log(self, outer):
        f = self.lib.lvo_oracle_mapping_log
        return dict(corner_knn=self._get(f, (outer, 10), np.int32, 5), surf_knn=self._get(f, (outer, 11), np.int32, 5),
                    corner_valid=self._get(f, (outer, 12), np.int32), surf_valid=self._get(f, (outer, 13), np.int32),
                    lm=self._get(f, (outer, 14), np.float64, 10), counts=self._get(f, (outer, 15), np.int32), cost=self._get(f, (outer, 16), np.float64))

    def map_export(self, which):
        n = self.lib.lvo_oracle_map_export(self.h, which, None, None, 0)
        pts = np.empty((n, 4), np.float32)
        cube = np.empty(n, np.int32)
        if n:
            self.lib.lvo_oracle_map_export(self.h, which, _ptr(pts), _ptr(cube), n)
        return pts, cube

    def map_import(self, which, pts, cube):
        pts = as_pts(pts)
        cube = np.ascontiguousarray(cube, np.int32)
        self.lib.lvo_oracle_map_import(self.h, which, _ptr(pts), _ptr(cube), len(pts))

    def set_map_correction(self, qt7):
        qt7 = np.ascontiguousarray(qt7, np.float64)
        self.lib.lvo_oracle_set_map_correction(self.h, _ptr(qt7))

    # -- all three
    def step(self, pts, keep_log=False):
        pts = as_pts(pts)
        poses = np.zeros(21)
        st = self.lib.lvo_oracle_step(self.h, _ptr(pts), len(pts), _ptr(poses), int(keep_log))
        self.high_freq = poses[14:].copy()   # /aft_mapped_to_init_high_frec of this frame (laserMapping.cpp:197-229)
        return st, poses[:7].copy(), poses[7:14].copy()

    def set_skip_frame(self, skip):
        """mapping_skip_frame (laserOdometry.cpp:274,643): map every skip-th frame; step() then returns the high-frequency pose for the others."""
        self.lib.lvo_oracle_set_skip_frame(self.h, int(skip))

    def last_frame_mapped(self):
        return bool(self.lib.lvo_oracle_last_frame_mapped(self.h))

    def odometry_last(self, which):
        """The "last" clouds after the frame (what laserOdometry.cpp:646-656 publishes): 0 corner, 1 surf, 2 full (distortion 2)."""
        n = self.lib.lvo_oracle_odometry_last(self.h, which, None, 0)
        a = np.empty((n, 4), np.float32)
        if n:
            self.lib.lvo_oracle_odometry_last(self.h, which, _ptr(a), n)
        return a

    def map_cloud(self, which):
        """0: surround cloud (laserMapping.cpp:806-815), 1: whole map (:823-836)."""
        n = self.lib.lvo_oracle_map_cloud(self.h, which, None, 0)
        a = np.empty((n, 4), np.float32)
        if n:
            self.lib.lvo_oracle_map_cloud(self.h, which, _ptr(a), n)
        return a

    def transform(self, pts, qt7, distortion, to_end=False):
        pts = as_pts(pts)
        qt7 = np.ascontiguousarray(qt7, np.float64)
        out = np.empty_like(pts)
        self.lib.lvo_oracle_transform(_ptr(pts), len(pts), _ptr(qt7), distortion, int(to_end), _ptr(out))
        return out

    def eval_factor_s(self, f14, s, x7):
        f14 = np.ascontiguousarray(f14, np.float64)
        x7 = np.ascontiguousarray(x7, np.float64)
        r = np.zeros(3)
        J = np.zeros(18)
        k = self.lib.lvo_oracle_eval_factor_s(_ptr(f14), float(s), _ptr(x7), _ptr(r), _ptr(J))
        return r[:k].copy(), J[:k * 6].reshape(k, 6).copy()

    def timings(self):
        t = np.zeros(3)
        self.lib.lvo_oracle_timings(self.h, _ptr(t))
        return t

    # -- stand-alone operators
    def voxel_grid(self, pts, leaf):
        pts = as_pts(pts)
        n = len(pts)
        out = np.empty((max(n, 1), 4), np.float32)
        idx = np.empty(max(n, 1), np.int32)
        order = np.empty(max(n, 1), np.int32)
        m = self.lib.lvo_oracle_voxel_grid(_ptr(pts), n, leaf, _ptr(out), len(out), _ptr(idx), _ptr(order))
        return out[:m].copy(), idx[:n], order[:n]

    def knn(self, cloud, q, K, max_sq, method=1):
        cloud, q = as_pts(cloud), as_pts(q)
        ind = np.empty((len(q), K), np.int32)
        sq = np.empty((len(q), K), np.float32)
        self.lib.lvo_oracle_knn(_ptr(cloud), len(cloud), _ptr(q), len(q), K, max_sq, method, _ptr(ind), _ptr(sq))
        return ind, sq

    def depth(self, sweep, extr12, uv):
        """Depth cloud + association (config 5).  Returns (depth_cloud, src_index, depth, valid, nn)."""
        sweep = as_pts(sweep)
        extr = np.ascontiguousarray(extr12, np.float32).reshape(12)
        uv = np.ascontiguousarray(uv, np.float32).reshape(-1, 2)
        cap = max(len(sweep), 1)
        dc = np.empty((cap, 4), np.float32)
        src = np.empty(cap, np.int32)
        depth = np.zeros(max(len(uv), 1), np.float32)
        valid = np.zeros(max(len(uv), 1), np.int32)
        nn = np.full((max(len(uv), 1), 3), -1, np.int32)
        n = self.lib.lvo_oracle_depth(_ptr(sweep), len(sweep), _ptr(extr), _ptr(uv), len(uv), _ptr(dc), _ptr(src), cap, _ptr(depth), _ptr(valid), _ptr(nn))
        return dc[:n].copy(), src[:n].copy(), depth[:len(uv)], valid[:len(uv)], nn[:len(uv)]

    def eval_factor(self, f14, x7):
        f14 = np.ascontiguousarray(f14, np.float64)
        x7 = np.ascontiguousarray(x7, np.float64)
        r = np.zeros(3)
        J = np.zeros(18)
        k = self.lib.lvo_oracle_eval_factor(_ptr(f14), _ptr(x7), _ptr(r), _ptr(J))
        return r[:k].copy(), J[:6 * k].reshape(k, 6).copy()

    def solve(self, factors, x7, max_iters=4, huber=0.1):
        factors = np.ascontiguousarray(factors, np.float64)
        x = np.array(x7, np.float64)
        tr = np.zeros((max_iters + 2, 10))
        n = self.lib.lvo_oracle_solve(_ptr(factors), len(factors), _ptr(x), max_iters, huber, _ptr(tr), len(tr))
        return x, tr[:n]
