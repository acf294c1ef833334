"""Pose uncertainty (include/lvo.h lvo_pose_uncertainty) on the CPU: the oracle's information matrix against numpy, the derived
covariance / eigen-decomposition against numpy.linalg, the degenerate tunnel scene, and the C struct layout against the ctypes mirror."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle_py import ROOT, Oracle, Synth  # noqa: E402
from uncertainty_oracle import (UncertaintyPipeline, hu_to_matrix, solve_info, tunnel, uncertainty_from_hu,  # noqa: E402
                                uncertainty_from_info)

HUBER = 0.1


def _pkg():
    if "lvo_b200" in sys.modules:
        return sys.modules["lvo_b200"]
    spec = importlib.util.spec_from_file_location("lvo_b200", os.path.join(ROOT, "lidar-visual-odometry_b200", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lvo_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def qmul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def plus7(x, d):
    """EigenQuaternionParameterization::Plus on q (q <- [sin|d| d^, cos|d|] q), addition on t."""
    nd = np.linalg.norm(d[:3])
    q = qmul(np.r_[np.sin(nd) / nd * d[:3], np.cos(nd)], x[:4]) if nd > 0 else x[:4]
    return np.r_[q, x[4:] + d[3:]]


def qrot(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def random_factors(rng, n, types):
    """Factor records [type, c, a, b, m, d] (14 doubles) that the identity pose nearly satisfies, with a share of outliers beyond the
    Huber width."""
    F = np.zeros((n, 14))
    for i in range(n):
        t = types[i % len(types)]
        c = rng.uniform(-20, 20, 3)
        off = rng.normal(0, 0.02 if i % 5 else 0.5, 3)
        F[i, 0] = t
        F[i, 1:4] = c
        if t == 0:      # edge through c + off along a random direction
            e = rng.normal(size=3); e /= np.linalg.norm(e)
            F[i, 4:7] = c + off + 0.3 * e
            F[i, 7:10] = c + off - 0.4 * e
        elif t == 1:    # plane through c + off spanned by two random directions
            u, v = rng.normal(size=3), rng.normal(size=3)
            F[i, 4:7] = c + off
            F[i, 7:10] = c + off + 0.5 * u
            F[i, 10:13] = c + off + 0.5 * v
        else:           # unit normal n, offset d: n . p + d = 0 near c
            nrm = rng.normal(size=3); nrm /= np.linalg.norm(nrm)
            F[i, 4:7] = nrm
            F[i, 13] = -(nrm @ (c + off))
    return F


def information_numpy(orc, F, x, s=None):
    """sum rho'(|r|^2) J^T J over the blocks, from the oracle's residuals / local Jacobians (Huber corrector weights)."""
    H = np.zeros((6, 6))
    for i, f in enumerate(F):
        r, J = orc.eval_factor_s(f, 1.0 if s is None else s[i], x)
        sq = r @ r
        w = max(np.finfo(float).tiny, HUBER / np.sqrt(sq)) if sq > HUBER * HUBER else 1.0
        H += w * J.T @ J
    return H


def information_fd(orc, F, x, s=None, h=1e-6):
    """Same with central finite-difference Jacobians taken through plus7."""
    H = np.zeros((6, 6))
    for i, f in enumerate(F):
        si = 1.0 if s is None else s[i]
        r, _ = orc.eval_factor_s(f, si, x)
        J = np.zeros((len(r), 6))
        for c in range(6):
            d = np.zeros(6); d[c] = h
            J[:, c] = (orc.eval_factor_s(f, si, plus7(x, d))[0] - orc.eval_factor_s(f, si, plus7(x, -d))[0]) / (2 * h)
        sq = r @ r
        w = max(np.finfo(float).tiny, HUBER / np.sqrt(sq)) if sq > HUBER * HUBER else 1.0
        H += w * J.T @ J
    return H


@pytest.mark.parametrize("types,distort", [((0,), False), ((1,), False), ((2,), False), ((0, 1, 2), False), ((0, 1), True)])
def test_information_matches_numpy_and_finite_differences(types, distort):
    rng = np.random.default_rng(7 + len(types) + 10 * distort)
    orc = Oracle()
    F = random_factors(rng, 120, types)
    s = rng.uniform(0.05, 1.0, len(F)) if distort else None
    x0 = plus7(np.array([0, 0, 0, 1.0, 0, 0, 0]), rng.normal(0, 0.01, 6))
    x, rec = solve_info(F, x0, s=s, huber=HUBER)
    assert not np.array_equal(x, x0)   # the solve moved: H is taken at the final pose
    H = hu_to_matrix(rec["hu"])
    Hn = information_numpy(orc, F, x, s)
    assert np.abs(H - Hn).max() <= 1e-12 * np.abs(Hn).max()
    Hf = information_fd(orc, F, x, s)
    assert np.abs(H - Hf).max() <= 1e-6 * np.abs(Hn).max()


def _random_spd(rng, cond):
    Q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    lam = np.geomspace(1.0, cond, 6) * rng.uniform(0.5, 2.0)
    return (Q * lam) @ Q.T


@pytest.mark.parametrize("seed", range(6))
def test_derived_values(seed):
    rng = np.random.default_rng(100 + seed)
    hu21 = _random_spd(rng, 10.0 ** (2 + seed))[np.triu_indices(6)]
    Hu = hu_to_matrix(hu21)   # the record keeps the upper triangle
    d = uncertainty_from_hu(hu21)
    info = d["information"]
    # p = (t, theta) = M u, u = (delta, dt): blocks H_tt, H_t,delta / 2, H_delta,delta / 4, exact in binary floating point
    assert np.array_equal(info[:3, :3], Hu[3:, 3:])
    assert np.array_equal(info[:3, 3:], Hu[3:, :3] * 0.5) and np.array_equal(info[3:, :3], Hu[:3, 3:] * 0.5)
    assert np.array_equal(info[3:, 3:], Hu[:3, :3] * 0.25)
    assert d["positive_definite"] == 1
    M = np.zeros((6, 6)); M[:3, 3:] = np.eye(3); M[3:, :3] = 2 * np.eye(3)
    cov_ref = M @ np.linalg.inv(Hu) @ M.T
    assert np.abs(d["covariance"] - cov_ref).max() <= 1e-9 * np.abs(cov_ref).max()
    assert np.array_equal(d["covariance"], d["covariance"].T)
    w_ref, V_ref = np.linalg.eigh(info)
    w, V = d["eigenvalues"], d["eigenvectors"]
    assert np.all(np.diff(w) >= 0)
    assert np.abs(w - w_ref).max() <= 1e-10 * np.abs(w_ref).max()
    for k in range(6):
        m = int(np.argmax(np.abs(V[:, k])))
        assert V[m, k] > 0 and np.all(np.abs(V[:m, k]) < V[m, k])   # documented sign: largest-magnitude entry positive (first on ties)
        v_ref = V_ref[:, k] * np.sign(V_ref[m, k])
        assert np.abs(V[:, k] - v_ref).max() <= 1e-7
    # the same fields from the information matrix directly
    d2 = uncertainty_from_info(info)
    for key in ("covariance", "eigenvalues", "eigenvectors"):
        assert np.array_equal(d2[key], d[key])


@pytest.mark.parametrize("kind", ["zero", "rank5", "cond1e15", "negative"])
def test_near_singular_information_is_not_positive_definite(kind):
    rng = np.random.default_rng(3)
    if kind == "zero":
        info = np.zeros((6, 6))
    elif kind == "rank5":
        A = rng.normal(size=(5, 6))
        info = A.T @ A
    elif kind == "cond1e15":
        info = _random_spd(rng, 1e15)
    else:
        info = _random_spd(rng, 10.0)
        info -= 20.0 * np.outer(info[:, 0], info[:, 0]) / info[0, 0]
    d = uncertainty_from_info(info)
    assert d["positive_definite"] == 0
    assert not np.any(d["covariance"])


# Tunnel: the synthetic street without recesses, poles and boxes (ground + two flat facades along world x).  Measured on the oracle,
# sequence 1, frames 1-5 (frame 0 has no solve):
#   |translation part of the weakest eigenvector . street axis in the parent frame| >= 0.9999 (HDL-64), >= 0.9992 (VLP-16), both stages;
#   median lambda_min / lambda_1 tunnel vs street: HDL-64 odometry 0.103 vs 0.522, mapping 0.077 vs 0.526;
#                                                  VLP-16 odometry 0.222 vs 0.549, mapping 0.022 vs 0.410.
# Bounds with margin: alignment >= cos(5 deg); tunnel median ratio < 0.5 x the street's.
TUNNEL_ALIGN_MIN = np.cos(np.radians(5.0))
TUNNEL_RATIO_FACTOR = 0.5
SENSORS = {64: dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8), 16: dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4)}


def tunnel_axis_in_parent(stage, gt_prev, axis0):
    """The street axis in the parent frame of the stage: the previous sensor frame (odometry) or the map frame = sensor frame 0."""
    return qrot(gt_prev[:4]).T @ axis0 if stage == "odometry" else axis0


def weakest_direction_summary(records, gts, axis0):
    """records[k][stage]: uncertainty dicts of frames 0..n-1.  Returns per stage (alignments, lambda_min / lambda_1 per frame >= 1)."""
    out = {}
    for stage in ("odometry", "mapping"):
        align, ratio = [], []
        for k in range(1, len(records)):
            u = records[k][stage]
            assert u["solved"] == 1
            w, v = u["eigenvalues"], u["eigenvectors"][:, 0]
            ratio.append(w[0] / w[1])
            if axis0 is not None:
                align.append(abs(v[:3] @ tunnel_axis_in_parent(stage, gts[k - 1], axis0)))
        out[stage] = (np.array(align), np.array(ratio))
    return out


def run_oracle(model, in_tunnel, frames=6, seq=1):
    s = SENSORS[model]
    orc = UncertaintyPipeline(s["n_scans"], s["minimum_range"], s["line_res"], s["plane_res"])
    syn = Synth()
    recs, gts, axis0 = [], [], None
    for k in range(frames):
        if in_tunnel:
            pts, gt, axis0 = tunnel(syn, model, seq, k)
        else:
            pts, gt = syn.sweep(model, seq, k)
        orc.step(pts)
        recs.append({st: orc.uncertainty(st) for st in ("odometry", "mapping")})
        gts.append(gt)
    return recs, gts, axis0


@pytest.mark.parametrize("model", [64, 16])
def test_tunnel_weakest_direction_on_oracle(model):
    recs, gts, axis0 = run_oracle(model, True)
    assert recs[0]["odometry"]["solved"] == 0
    street, _, _ = run_oracle(model, False)
    tun = weakest_direction_summary(recs, gts, axis0)
    ref = weakest_direction_summary(street, gts, None)
    for stage in ("odometry", "mapping"):
        align, ratio = tun[stage]
        assert align.min() >= TUNNEL_ALIGN_MIN, (stage, align)
        assert np.median(ratio) < TUNNEL_RATIO_FACTOR * np.median(ref[stage][1]), (stage, ratio, ref[stage][1])


def test_tunnel_generator_leaves_the_street_alone():
    syn = Synth()
    a, gt_a = syn.sweep(64, 1, 3)
    b, gt_b, _ = tunnel(syn, 64, 1, 3)
    assert np.array_equal(gt_a, gt_b)          # same trajectory
    assert len(a) != len(b) or not np.array_equal(a, b)


ABI_PROGRAM = r"""
#include <stddef.h>
#include <stdio.h>
#include "lvo.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(lvo_pose_uncertainty), offsetof(lvo_pose_uncertainty, frame),
         offsetof(lvo_pose_uncertainty, solved), offsetof(lvo_pose_uncertainty, positive_definite), offsetof(lvo_pose_uncertainty, n_factors),
         offsetof(lvo_pose_uncertainty, reserved), offsetof(lvo_pose_uncertainty, cost), offsetof(lvo_pose_uncertainty, information),
         offsetof(lvo_pose_uncertainty, covariance), offsetof(lvo_pose_uncertainty, eigenvalues), offsetof(lvo_pose_uncertainty, eigenvectors));
  printf("%d %d\n", (int)LVO_P_ODO_UNCERTAINTY, (int)LVO_P_MAP_UNCERTAINTY);
  return 0;
}
"""


def test_struct_layout_matches_ctypes_mirror(tmp_path):
    src = tmp_path / "abi.c"
    src.write_text(ABI_PROGRAM)
    exe = tmp_path / "abi"
    cc = os.environ.get("CC", "cc")
    subprocess.check_call([cc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    lines = subprocess.check_output([str(exe)]).decode().split("\n")
    got = [int(v) for v in lines[0].split()]
    mod = _pkg()
    U = mod.PoseUncertainty
    want = [C.sizeof(U)] + [getattr(U, f).offset for f in ("frame", "solved", "positive_definite", "n_factors", "reserved", "cost", "information",
                                                            "covariance", "eigenvalues", "eigenvectors")]
    assert got == want
    assert [int(v) for v in lines[1].split()] == [mod.P_ODO_UNCERTAINTY, mod.P_MAP_UNCERTAINTY]
