"""Pose uncertainty of every lane (LVO_P_ODO_UNCERTAINTY / LVO_P_MAP_UNCERTAINTY, Lvo.pose_uncertainty) on the B200: against the CPU
oracle, bit for bit across lanes, contexts, graphs, the reuse options and the step forms, through the lane lifecycle, in the
degenerate tunnel, in a 128-lane context, and through the C++ adaptor."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, record_metric
from uncertainty_oracle import UncertaintyPipeline, tunnel, uncertainty_from_info
from test_pose_uncertainty_cpu import SENSORS, TUNNEL_ALIGN_MIN, TUNNEL_RATIO_FACTOR, weakest_direction_summary

pytestmark = pytest.mark.gpu
CAPS = dict(max_map_corner=1 << 18, max_map_surf=1 << 19)
STAGES = ("odometry", "mapping")
FIELDS = ("frame", "solved", "positive_definite", "n_factors", "cost", "information", "covariance", "eigenvalues", "eigenvectors")
# Relative Frobenius difference of the information matrix from the oracle's (J^T W J summed in the GPU's fixed tree, in row order on the
# CPU).  Measured on a B200 over the 10 frames of each case: 3.3e-15 (HDL-64 seq 0), 2.3e-15 (VLP-16 seq 1), 3.9e-15 (DISTORTION 1):
# the factors and LM states agree, so only the summation order differs.
INFO_REL_MAX = 1e-11


def records(lvo, lane=0):
    return {st: lvo.pose_uncertainty(lane, st) for st in STAGES}


def same(a, b):
    """Bit-for-bit equality of two records (dicts of Lvo.pose_uncertainty)."""
    return all(np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes() for k in FIELDS)


def same_all(ra, rb):
    return all(same(ra[st], rb[st]) for st in STAGES)


# ---- against the oracle ----------------------------------------------------------------------------------------------------------
ORACLE_CASES = {"hdl64_seq0": (64, 0, 0), "vlp16_seq1": (16, 1, 0), "hdl64_seq0_distortion1": (64, 0, 1)}


@pytest.mark.parametrize("case", list(ORACLE_CASES))
def test_against_oracle(lvo_mod, synth, case):
    L = lvo_mod
    model, seq, distortion = ORACLE_CASES[case]
    s = SENSORS[model]
    lvo = L.Lvo(**s, distortion=distortion, **CAPS)
    orc = UncertaintyPipeline(s["n_scans"], s["minimum_range"], s["line_res"], s["plane_res"], distortion=distortion)
    worst = 0.0
    for k in range(10):
        pts, _ = synth.sweep(model, seq, k, moving=distortion != 0)
        lvo.step_batch([pts])
        orc.step(pts)
        st = lvo.stats(0)
        O = lvo.cfg.outer_iters
        for stage in STAGES:
            g, o = lvo.pose_uncertainty(0, stage), orc.uncertainty(stage)
            assert g["frame"] == k
            assert (g["solved"], g["n_factors"]) == (o["solved"], o["n_factors"]), (k, stage)
            final = (st.odo_final_cost if stage == "odometry" else st.map_final_cost)[O - 1]
            assert np.float64(g["cost"]).tobytes() == np.float64(final).tobytes(), (k, stage)
            if g["solved"]:
                rel = np.linalg.norm(g["information"] - o["information"]) / np.linalg.norm(o["information"])
                worst = max(worst, rel)
            # the derived fields: the oracle's restatement of the conversion, Jacobi and covariance gives the same bits
            d = uncertainty_from_info(g["information"])
            assert d["positive_definite"] == g["positive_definite"]
            for key in ("covariance", "eigenvalues", "eigenvectors"):
                assert d[key].tobytes() == g[key].tobytes(), (k, stage, key)
    record_metric(f"pose_uncertainty_info_rel_frobenius_{case}", worst)
    assert worst <= INFO_REL_MAX
    lvo.close()


# ---- bitwise invariance ------------------------------------------------------------------------------------------------------------
FRAMES = 6


def run(L, synth, lanes=1, graphs=0, options=None, form="plain", frames=FRAMES, seq=0):
    """Records of lane 0 (and of every lane) after each frame of HDL-64 sequence `seq`, every lane running it."""
    lvo = L.Lvo(lanes=lanes, **CAPS)
    lvo.set_option(L.LVO_OPT_GRAPHS, graphs)
    for opt, val in (options or {}).items():
        lvo.set_option(opt, val)
    out = []
    seqs = [[synth.sweep(64, seq, k)[0]] * lanes for k in range(frames)]   # the same arrays every call: the pipelined prefetch hits
    for k in range(frames):
        sw = seqs[k]
        pts = sw[0]
        if form == "plain":
            lvo.step_batch(sw)
        elif form == "async":
            lvo.step_batch_async(sw)
            lvo.wait()
        elif form == "pipelined":
            lvo.step_batch_pipelined(sw, seqs[k + 1] if k + 1 < frames else None)
        elif form == "dev":
            import torch
            d = torch.from_numpy(pts).cuda()
            torch.cuda.synchronize()
            lvo.step_batch_dev([d.data_ptr()] * lanes, [d.shape[0]] * lanes)
        out.append([records(lvo, lane) for lane in range(lanes)])
    lvo.close()
    return out


@pytest.fixture(scope="module")
def baseline(lvo_mod, synth):
    return run(lvo_mod, synth)


def _variant(L, name):
    return {"two_lanes": dict(lanes=2), "second_context": dict(), "graphs": dict(graphs=1),
            "no_fixpoint_skip": dict(options={L.LVO_OPT_FIXPOINT_SKIP: 0}), "no_knn_reuse": dict(options={L.LVO_OPT_KNN_REUSE: 0}),
            "no_odo_reuse": dict(options={L.LVO_OPT_ODO_REUSE: 0}), "async": dict(form="async"), "pipelined": dict(form="pipelined"),
            "dev": dict(form="dev")}[name]


@pytest.mark.parametrize("variant", ["two_lanes", "second_context", "graphs", "no_fixpoint_skip", "no_knn_reuse", "no_odo_reuse", "async",
                                     "pipelined", "dev"])
def test_bitwise_invariance(lvo_mod, synth, baseline, variant):
    got = run(lvo_mod, synth, **_variant(lvo_mod, variant))
    for k in range(FRAMES):
        for lane_recs in got[k]:
            assert same_all(lane_recs, baseline[k][0]), (variant, k)
    assert baseline[-1][0]["odometry"]["solved"] == 1 and baseline[-1][0]["mapping"]["positive_definite"] == 1


def test_map_fixed_lane_equals_its_twin(lvo_mod, synth):
    """Lane 1 stops updating its map at frame 3; on that frame both lanes register against the same map."""
    L = lvo_mod
    lvo = L.Lvo(lanes=2, **CAPS)
    for k in range(4):
        if k == 3:
            lvo.set_lane_map_update(1, False)
        pts = synth.sweep(64, 2, k)[0]
        lvo.step_batch([pts, pts])
        assert same_all(records(lvo, 0), records(lvo, 1)), k
    assert records(lvo, 1)["mapping"]["solved"] == 1
    lvo.close()


# ---- lifecycle ---------------------------------------------------------------------------------------------------------------------
def test_lifecycle(lvo_mod, synth):
    L = lvo_mod
    lvo = L.Lvo(lanes=3, **CAPS)
    lvo.set_option(L.LVO_OPT_GRAPHS, 0)
    lvo.lane_configure(1, skip_frame=2)
    sw = lambda k: [synth.sweep(64, 0, k)[0]] * 3
    fresh = records(lvo, 0)
    assert all(fresh[st]["frame"] == -1 and fresh[st]["solved"] == 0 and not fresh[st]["information"].any() for st in STAGES)
    lvo.step_batch(sw(0))
    r = records(lvo, 0)
    assert r["odometry"]["frame"] == 0 and r["odometry"]["solved"] == 0 and r["odometry"]["n_factors"] == 0
    assert r["mapping"]["frame"] == 0 and r["mapping"]["solved"] == 0   # the map is empty on the first frame
    map_frames = []
    for k in range(1, 5):
        lvo.step_batch(sw(k))
        map_frames.append(records(lvo, 1)["mapping"]["frame"])
        assert records(lvo, 1)["odometry"]["frame"] == k and records(lvo, 0)["mapping"]["frame"] == k
    assert map_frames == [0, 2, 2, 4]   # skip_frame 2: the mapping record advances by 2
    # fetching changes neither the launch count of the step nor the other probes
    launches = lvo.timings().kernel_launches
    before = [lvo.probe(w, 0) for w in (L.P_FULL, L.P_ODO_LM_TRACE, L.P_MAP_LM_TRACE, L.P_REGISTERED)]
    r0 = records(lvo, 0)
    after = [lvo.probe(w, 0) for w in (L.P_FULL, L.P_ODO_LM_TRACE, L.P_MAP_LM_TRACE, L.P_REGISTERED)]
    assert lvo.timings().kernel_launches == launches
    assert all(a.tobytes() == b.tobytes() for a, b in zip(before, after))
    # lvo_knn, the depth calls and the map outputs leave the records alone (a reset of lane 2 makes the next fetch derive them again)
    pts = sw(5)[0]
    lvo.knn(pts[:1000], pts[:100], 5, 1.0)
    lvo.depth_associate(pts, np.zeros((4, 2), np.float32))
    lvo.map_cloud_batch(L.LVO_MAP_SURROUND)
    lvo.map_cloud(0, L.LVO_MAP_WHOLE)
    lvo.lane_reset(2)
    assert same_all(records(lvo, 0), r0)
    assert all(records(lvo, 2)[st]["frame"] == -1 for st in STAGES)
    # an idle lane keeps both records bit for bit
    lvo.set_lane_active(0, False)
    lvo.step_batch([None, pts, pts])
    assert same_all(records(lvo, 0), r0)
    lvo.set_lane_active(0, True)
    # with a step in flight the probes are refused and write nothing
    lvo.step_batch_async(sw(6))
    buf = (C.c_ubyte * C.sizeof(L.PoseUncertainty))(*([0xA5] * C.sizeof(L.PoseUncertainty)))
    for what in (L.P_ODO_UNCERTAINTY, L.P_MAP_UNCERTAINTY):
        assert lvo.lib.lvo_probe_fetch(lvo.h, 0, what, C.addressof(buf), C.sizeof(buf), None) == L.LVO_E_STATE
    assert bytes(buf) == bytes([0xA5]) * C.sizeof(buf)
    lvo.wait()
    # reset and configure clear both records
    lvo.lane_configure(1, skip_frame=1)
    lvo.lane_reset(0)
    for lane in (0, 1):
        assert all(records(lvo, lane)[st]["frame"] == -1 and records(lvo, lane)[st]["solved"] == 0 for st in STAGES)
    # a load gates the probes until the stage runs; the records then follow the loaded sequence
    donor = L.Lvo(lanes=1, **CAPS)
    for k in range(3):
        donor.step_batch([synth.sweep(64, 1, k)[0]])
    snap = donor.lane_save(0)
    lvo.lane_load(2, snap)
    for st in STAGES:
        with pytest.raises(L.LvoError, match="-4"):
            lvo.pose_uncertainty(2, st)
    nxt = synth.sweep(64, 1, 3)[0]
    donor.step_batch([nxt])
    lvo.step_batch([pts, pts, nxt])
    assert same_all(records(lvo, 2), records(donor, 0)) and records(lvo, 2)["odometry"]["frame"] == 3
    donor.close()
    lvo.close()


def test_fetch_leaves_step_launches(lvo_mod, synth):
    L = lvo_mod
    counts = []
    for fetch in (False, True):
        lvo = L.Lvo(**CAPS)
        lvo.set_option(L.LVO_OPT_GRAPHS, 0)
        c = []
        for k in range(3):
            lvo.step_batch([synth.sweep(64, 0, k)[0]])
            t = bytes(lvo.timings())
            c.append(lvo.timings().kernel_launches)
            if fetch:
                records(lvo)
                assert bytes(lvo.timings()) == t   # the fetch's own launch and copy leave lvo_timings as they were
        counts.append(c)
        lvo.close()
    assert counts[0] == counts[1]


def test_empty_fixed_map_is_not_solved(lvo_mod, synth):
    L = lvo_mod
    lvo = L.Lvo(**CAPS)
    lvo.set_lane_map_update(0, False)
    for k in range(3):
        lvo.step_batch([synth.sweep(64, 0, k)[0]])
        r = records(lvo)
        assert r["mapping"]["frame"] == k and r["mapping"]["solved"] == 0 and not r["mapping"]["covariance"].any()
    assert r["odometry"]["solved"] == 1
    lvo.close()


# ---- tunnel --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", [64, 16])
def test_tunnel_weakest_direction(lvo_mod, synth, model):
    L = lvo_mod
    out = {}
    for in_tunnel in (True, False):
        lvo = L.Lvo(**SENSORS[model], **CAPS)
        recs, gts, axis0 = [], [], None
        for k in range(6):
            if in_tunnel:
                pts, gt, axis0 = tunnel(synth, model, 1, k)
            else:
                pts, gt = synth.sweep(model, 1, k)
            lvo.step_batch([pts])
            recs.append(records(lvo))
            gts.append(gt)
        out[in_tunnel] = weakest_direction_summary(recs, gts, axis0)
        lvo.close()
    for st in STAGES:
        align, ratio = out[True][st]
        assert align.min() >= TUNNEL_ALIGN_MIN, (st, align)
        assert np.median(ratio) < TUNNEL_RATIO_FACTOR * np.median(out[False][st][1]), (st, ratio, out[False][st][1])
        record_metric(f"pose_uncertainty_tunnel_{model}_{st}_ratio_vs_street", float(np.median(ratio) / np.median(out[False][st][1])))


# ---- fleet ---------------------------------------------------------------------------------------------------------------------------
def test_128_lanes_equal_one_lane_contexts(lvo_mod, synth):
    from test_gpu_lane_config import HDL64, VLP16
    L = lvo_mod
    lanes, frames = 128, 3
    desc = [(64, l % 4, HDL64) if l % 2 == 0 else (16, l % 4, VLP16) for l in range(lanes)]
    x = L.Lvo(lanes=lanes, max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 20, **HDL64)
    for l, (model, _, cfg) in enumerate(desc):
        if model == 16:
            x.lane_configure(l, **cfg)
    solo = {}
    for key in sorted(set((m, s) for m, s, _ in desc)):
        cfg = HDL64 if key[0] == 64 else VLP16
        solo[key] = L.Lvo(max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 20, **cfg)
    for k in range(frames):
        sweeps = {key: synth.sweep(key[0], key[1], k)[0] for key in solo}
        x.step_batch([sweeps[(m, s)] for m, s, _ in desc])
        ref = {}
        for key, lvo in solo.items():
            lvo.step_batch([sweeps[key]])
            ref[key] = records(lvo)
        for l, (m, s, _) in enumerate(desc):
            assert same_all(records(x, l), ref[(m, s)]), (k, l)
    for lvo in solo.values():
        lvo.close()
    x.close()


# ---- C++ adaptor ---------------------------------------------------------------------------------------------------------------------
ADAPTOR_PROGRAM = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include <vector>
#include "lvo_handlers.hpp"
struct Pt { float x, y, z, intensity; };
struct Cloud { std::vector<Pt> points; };
int main(int argc, char** argv) {
  lvo::Context ctx(lvo::Context::hdl64());
  lvo::ScanRegistration reg(ctx);
  lvo::LaserOdometry odo(ctx);
  lvo::LaserMapping map(ctx);
  int bad = 0;
  for (int k = 1; k < argc; ++k) {
    std::ifstream f(argv[k], std::ios::binary | std::ios::ate);
    Cloud in, full, sharp, lessSharp, flat, lessFlat;
    in.points.resize((size_t)f.tellg() / sizeof(Pt));
    f.seekg(0);
    f.read(reinterpret_cast<char*>(in.points.data()), (std::streamsize)(in.points.size() * sizeof(Pt)));
    reg.laserCloudHandler(in, full, sharp, lessSharp, flat, lessFlat);
    lvo::Pose rel, wodom, wmap;
    odo.process(sharp, lessSharp, flat, lessFlat, rel, wodom);
    map.process(lessSharp, lessFlat, full, wodom, wmap);
    double c_odo[36], c_map[36];
    const bool pd_odo = odo.motionCovariance(c_odo), pd_map = map.poseCovariance(c_map);
    lvo_pose_uncertainty u[2];
    lvo_probe_fetch(ctx.get(), 0, LVO_P_ODO_UNCERTAINTY, &u[0], sizeof(u[0]), nullptr);
    lvo_probe_fetch(ctx.get(), 0, LVO_P_MAP_UNCERTAINTY, &u[1], sizeof(u[1]), nullptr);
    if (std::memcmp(c_odo, u[0].covariance, sizeof(c_odo)) || std::memcmp(c_map, u[1].covariance, sizeof(c_map))) bad = 1;
    if (pd_odo != (u[0].positive_definite != 0) || pd_map != (u[1].positive_definite != 0)) bad = 1;
    std::printf("%d %d %.17g %.17g\n", (int)pd_odo, (int)pd_map, c_odo[0], c_map[35]);
  }
  std::printf(bad ? "MISMATCH\n" : "OK\n");
  return bad;
}
"""


def test_cpp_adaptor_matches_probe(lvo_mod, synth, tmp_path):
    pkg = os.path.join(ROOT, "lidar-visual-odometry_b200")
    src = tmp_path / "adaptor.cpp"
    src.write_text(ADAPTOR_PROGRAM)
    exe = tmp_path / "adaptor"
    subprocess.check_call([os.environ.get("CXX", "g++"), "-std=c++14", "-O1", "-I", os.path.join(pkg, "host"), "-o", str(exe), str(src), "-L", pkg, "-llvo",
                           f"-Wl,-rpath,{pkg}"])
    files = []
    for k in range(3):
        p = tmp_path / f"{k}.bin"
        synth.sweep(64, 0, k)[0].tofile(p)
        files.append(str(p))
    r = subprocess.run([str(exe)] + files, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.split("\n")
    assert lines[3] == "OK"
    assert lines[0].split()[:2] == ["0", "0"] and lines[2].split()[:2] == ["1", "1"]   # first frame: nothing solved; then both constrained
