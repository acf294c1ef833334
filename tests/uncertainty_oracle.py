"""ctypes side of tests/uncertainty_oracle.cpp: the pose-uncertainty record (include/lvo.h lvo_pose_uncertainty) on the CPU oracle, and
the tunnel scene of the synthetic generator.  The library is compiled on first use, with the oracle's flags, into a cache directory
under the system temporary directory (keyed by the hash of its sources).  TEST INFRASTRUCTURE."""
import ctypes as C
import glob
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle_py import ROOT, _ptr, as_pts

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "uncertainty_oracle.cpp")
ORACLE = os.path.join(ROOT, "oracle")
CXXFLAGS = ["-std=c++17", "-O3", "-fPIC", "-ffp-contract=off", "-shared"]   # oracle/Makefile: no FMA contraction
_LIB = None


def _build():
    deps = [SRC] + sorted(glob.glob(os.path.join(ORACLE, "*.hpp"))) + [os.path.join(ROOT, "lidar-visual-odometry_b200", "csrc", "lvo_math.h")]
    h = hashlib.sha256()
    for p in deps:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(CXXFLAGS).encode())
    d = os.path.join(tempfile.gettempdir(), f"lvo_uncertainty_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    lib = os.path.join(d, f"lib_{h.hexdigest()[:16]}.so")
    if not os.path.exists(lib):
        tmp = f"{lib}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-I", ORACLE, "-o", tmp, SRC])
        os.replace(tmp, lib)
    return lib


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(_build())
        L.unc_from_info.argtypes = [C.c_void_p] * 5
        L.unc_from_hu.argtypes = [C.c_void_p] * 6
        L.unc_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p]
        L.unc_pipeline_create.restype = C.c_void_p
        L.unc_pipeline_create.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int]
        L.unc_pipeline_destroy.argtypes = [C.c_void_p]
        L.unc_pipeline_step.argtypes = [C.c_void_p, C.c_void_p, C.c_long]
        L.unc_pipeline_record.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 7
        _LIB = L
    return _LIB


def hu_to_matrix(hu21):
    """21 upper-triangle entries (row-major) -> symmetric 6 x 6."""
    H = np.zeros((6, 6))
    H[np.triu_indices(6)] = hu21
    return H + np.triu(H, 1).T


def uncertainty_from_info(info36):
    """The derived fields (covariance, eigenvalues, eigenvectors, positive_definite) from an information matrix in p = (t, theta),
    computed as the device computes them."""
    info = np.ascontiguousarray(np.asarray(info36, np.float64).reshape(36))
    cov, w, V, pd = np.zeros(36), np.zeros(6), np.zeros(36), np.zeros(1, np.int32)
    lib().unc_from_info(_ptr(info), _ptr(cov), _ptr(w), _ptr(V), _ptr(pd))
    return dict(positive_definite=int(pd[0]), covariance=cov.reshape(6, 6), eigenvalues=w, eigenvectors=V.reshape(6, 6))


def uncertainty_from_hu(hu21):
    """information (p coordinates) and the derived fields from H_u in the solver tangent (delta, dt)."""
    hu = np.ascontiguousarray(np.asarray(hu21, np.float64).reshape(21))
    info, cov, w, V, pd = np.zeros(36), np.zeros(36), np.zeros(6), np.zeros(36), np.zeros(1, np.int32)
    lib().unc_from_hu(_ptr(hu), _ptr(info), _ptr(cov), _ptr(w), _ptr(V), _ptr(pd))
    return dict(positive_definite=int(pd[0]), information=info.reshape(6, 6), covariance=cov.reshape(6, 6), eigenvalues=w, eigenvectors=V.reshape(6, 6))


def solve_info(factors, x7, s=None, max_iters=4, huber=0.1):
    """The oracle's LM solve of factor records (14 doubles each, as Oracle.solve; s: per-factor interpolation ratios or None) and its
    record: (x, dict with hu (H_u, 21 entries), cost and the derived fields)."""
    factors = np.ascontiguousarray(factors, np.float64).reshape(-1, 14)
    sv = None if s is None else np.ascontiguousarray(s, np.float64)
    x = np.array(x7, np.float64)
    hu, cost = np.zeros(21), np.zeros(1)
    lib().unc_solve(_ptr(factors), _ptr(sv), len(factors), _ptr(x), max_iters, huber, _ptr(hu), _ptr(cost))
    return x, dict(uncertainty_from_hu(hu), solved=1, n_factors=len(factors), cost=float(cost[0]), hu=hu)


class UncertaintyPipeline:
    """The oracle's extract -> odometry -> mapping chain (as Oracle.step) that keeps each stage's pose-uncertainty record."""

    def __init__(self, n_scans=64, min_range=5.0, line_res=0.4, plane_res=0.8, outer=10, lm_iters=4, huber=0.1, distortion=0, skip_frame=1):
        self.lib = lib()
        self.h = self.lib.unc_pipeline_create(n_scans, min_range, line_res, plane_res, outer, lm_iters, huber, distortion, skip_frame)

    def __del__(self):
        try:
            self.lib.unc_pipeline_destroy(self.h)
        except Exception:
            pass

    def step(self, pts):
        """One frame; True if it was mapped."""
        pts = as_pts(pts)
        return bool(self.lib.unc_pipeline_step(self.h, _ptr(pts), len(pts)))

    def uncertainty(self, stage):
        """Record of stage "odometry" or "mapping": solved, positive_definite, n_factors, cost, hu, information, covariance, eigenvalues,
        eigenvectors."""
        ints = np.zeros(3, np.int32)
        cost, hu, info, cov, w, V = np.zeros(1), np.zeros(21), np.zeros(36), np.zeros(36), np.zeros(6), np.zeros(36)
        self.lib.unc_pipeline_record(self.h, 1 if stage == "mapping" else 0, _ptr(ints), _ptr(cost), _ptr(hu), _ptr(info), _ptr(cov), _ptr(w), _ptr(V))
        return dict(solved=int(ints[0]), positive_definite=int(ints[1]), n_factors=int(ints[2]), cost=float(cost[0]), hu=hu,
                    information=info.reshape(6, 6), covariance=cov.reshape(6, 6), eigenvalues=w, eigenvectors=V.reshape(6, 6))


def tunnel(synth, model, seq, frame, speed=None):
    """lvo_synth_sweep_tunnel through an oracle_py.Synth: a sweep of the usual trajectory in the street without recesses, poles and
    boxes (ground + two flat facades along world x).  Returns (points, gt_pose7, street axis in the sensor frame of sweep 0)."""
    f = synth.lib.lvo_synth_sweep_tunnel
    f.restype = C.c_long
    f.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
    if speed is None:
        speed = 1.0 if model == 64 else 0.2
    out = np.empty((synth.lib.lvo_synth_rays(model), 4), np.float32)
    gt, axis = np.empty(7, np.float64), np.empty(3, np.float64)
    n = f(model, seq, frame, speed, _ptr(out), len(out), _ptr(gt), _ptr(axis))
    assert n >= 0
    return out[:n].copy(), gt, axis
