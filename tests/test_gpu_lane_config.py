"""Per-lane sensor settings: lvo_lane_configure / lvo_lane_get_config.

A lane configured as a VLP-16, HDL-32 or HDL-64 sensor computes bit for bit what lane 0 of a context created with those settings
computes, whatever the context's own n_scans and the other lanes' settings.  "Equal" below is bitwise, as in test_gpu_lanes.py:
poses, statuses, lvo_stats bytes, both map exports with cube ids, both map clouds, the map correction; here also the three
lvo_map_cloud_batch outputs, the ring probes and the lvo_lane_save bytes."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, load_lvo
from test_gpu_golden import rot_err, sha
from test_gpu_lanes import CAPS, lane_state

gpu = pytest.mark.gpu
FIELDS = ("n_scans", "minimum_range", "line_res", "plane_res", "skip_frame")
VLP16 = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4, skip_frame=1)   # launch/aloam_velodyne_VLP_16.launch
HDL64 = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, skip_frame=1)   # launch/aloam_velodyne_HDL_64.launch
CTX = dict(HDL64, minimum_range=4.0, skip_frame=2)   # the mixed context's own values: what its unconfigured lane runs
# lane l of the mixed context: its settings (None: never configured), and the sensor model and sequence of its sweeps
MIXED = [(VLP16, 16, 1), (dict(VLP16, skip_frame=3), 16, 3), (dict(VLP16, n_scans=32, line_res=0.3, plane_res=0.6), 16, 0),
         (HDL64, 64, 0), (dict(HDL64, skip_frame=2), 64, 2), (None, 64, 4)]
FRAMES = 10


class Sweeps:
    """Synthetic sweeps of each sensor model, generated once per (model, sequence, frame)."""

    def __init__(self, synth):
        self.synth, self.cache = synth, {}

    def __call__(self, model, seq, frame):
        key = (model, seq, frame)
        if key not in self.cache:
            self.cache[key] = self.synth.sweep(model, seq, frame)[0]
        return self.cache[key]


@pytest.fixture(scope="module")
def sweeps(synth):
    return Sweeps(synth)


def make(L, graphs, lanes, **kw):
    lvo = L.Lvo(lanes=lanes, **CAPS, **kw)
    lvo.set_option(L.LVO_OPT_GRAPHS, graphs)
    return lvo


def observed(L, lvo, lane):
    """What a caller sees of one lane right after a step: lane_state, the ring probes and the three batched map outputs."""
    d = lane_state(lvo, lane)
    for what in (L.P_SCAN_START, L.P_SCAN_END, L.P_LESS_FLAT):
        d[f"probe{what}"] = lvo.probe(what, lane).tobytes()
    for which in (L.LVO_MAP_SURROUND, L.LVO_MAP_WHOLE, L.LVO_MAP_REGISTERED):
        d[f"batch{which}"] = lvo.map_cloud_batch(which, [lane])[lane].tobytes()
    return d


def dedicated_run(L, graphs, distortion, cfg, model, seq, sweeps):
    """Lane 0 of a context created with `cfg`: per step (status, odometry row, mapping row, observed), then the lane_save bytes."""
    x = make(L, graphs, 1, distortion=distortion, **cfg)
    steps = []
    for k in range(FRAMES):
        _, o, m = x.step_batch([sweeps(model, seq, k)])
        steps.append((x.lane_status(0), o[0], m[0], observed(L, x, 0)))
    snap = x.lane_save(0)
    x.close()
    return steps, snap


class Runner:
    """Steps the mixed context through one of the batched entry points."""

    def __init__(self, lvo, mode):
        self.lvo, self.mode = lvo, mode

    def step(self, sw, nxt):
        lvo = self.lvo
        if self.mode == "async":
            lvo.step_batch_async(sw)
            return lvo.wait()
        if self.mode == "pipelined":
            self.keep = nxt          # handed over by pointer until the next call
            return lvo.step_batch_pipelined(sw, nxt)
        import torch
        dev = [torch.from_numpy(s).cuda() for s in sw]
        torch.cuda.synchronize()
        return lvo.step_batch_dev([d.data_ptr() for d in dev], [d.shape[0] for d in dev])


@gpu
@pytest.mark.parametrize("distortion", [0, 2])
@pytest.mark.parametrize("graphs", [0, 1])
def test_mixed_lanes_equal_dedicated_contexts(lvo_mod, sweeps, graphs, distortion):
    """VLP-16 (skip_frame 1 and 3), 32 beams on VLP-16 sweeps, HDL-64 (skip_frame 1 and 2) and an unconfigured lane in one 64-beam
    context, through lvo_step_batch_dev, lvo_step_batch_pipelined with packed 12-byte records and lvo_step_batch_async + lvo_wait."""
    L = lvo_mod
    refs = [dedicated_run(L, graphs, distortion, cfg or CTX, model, seq, sweeps) for cfg, model, seq in MIXED]
    for mode in ("dev", "pipelined", "async"):
        x = make(L, graphs, len(MIXED), distortion=distortion, **CTX)
        for lane, (cfg, _, _) in enumerate(MIXED):
            if cfg is not None:
                x.lane_configure(lane, **cfg)
            assert x.lane_config(lane) == (cfg or CTX), (mode, lane)
        frames = [[sweeps(model, seq, k) for _, model, seq in MIXED] for k in range(FRAMES)]
        if mode == "pipelined":
            frames = [[np.ascontiguousarray(s[:, :3]) for s in f] for f in frames]
        run = Runner(x, mode)
        for k in range(FRAMES):
            r, o, m = run.step(frames[k], frames[k + 1] if k + 1 < FRAMES else None)
            for lane in range(len(MIXED)):
                st, ro, rm, rs = refs[lane][0][k]
                assert x.lane_status(lane) == st and np.array_equal(o[lane], ro) and np.array_equal(m[lane], rm), (mode, k, lane)
                got = observed(L, x, lane)
                assert got == rs, (mode, k, lane, [key for key in rs if got[key] != rs[key]])
        for lane in range(len(MIXED)):
            assert len(x.probe(L.P_SCAN_START, lane)) == len(x.probe(L.P_SCAN_END, lane)) == (MIXED[lane][0] or CTX)["n_scans"]
            assert np.array_equal(x.lane_save(lane), refs[lane][1]), (mode, lane)
        x.close()


@gpu
def test_reference_node_goldens_side_by_side(lvo_mod, synth):
    """The three reference-node fixtures of test_gpu_golden.py, one per lane of one 64-beam context, stepped in lock-step; a lane goes
    idle when its fixture runs out of frames.  Every lane passes the assertions that test applies to a dedicated context."""
    L = lvo_mod
    fixtures = [("refnode_hdl64_seq0.npz", 64, 0), ("refnode_vlp16_seq1.npz", 16, 1), ("refnode_hdl64_seq2_skip2.npz", 64, 2)]
    gs = [np.load(os.path.join(ROOT, "tests", "golden", f)) for f, _, _ in fixtures]
    lvo = L.Lvo(lanes=len(gs), n_scans=64, max_map_corner=1 << 18, max_map_surf=1 << 19)
    for lane, g in enumerate(gs):
        cfg = g["config"]
        lvo.lane_configure(lane, n_scans=int(cfg[0]), minimum_range=float(cfg[1]), line_res=float(cfg[2]), plane_res=float(cfg[3]),
                           skip_frame=int(g["skip_frame"]))
    assert [lvo.lane_config(l)["n_scans"] for l in range(3)] == [64, 16, 64] and lvo.lane_config(2)["skip_frame"] == 2
    clouds = dict(full=L.P_FULL, sharp=L.P_SHARP, less_sharp=L.P_LESS_SHARP, flat=L.P_FLAT, less_flat=L.P_LESS_FLAT)
    arrays = dict(curvature=L.P_CURVATURE, sort_ind=L.P_SORT_IND, picked=L.P_PICKED, label=L.P_LABEL)
    frames = [int(g["frames"]) for g in gs]
    assert len(set(frames)) > 1, "the fixtures should end at different frames, so that a lane goes idle"
    for k in range(max(frames)):
        sw = []
        for lane, (g, (_, model, seq)) in enumerate(zip(gs, fixtures)):
            if k == frames[lane]:
                lvo.set_lane_active(lane, False)
            sw.append(synth.sweep(model, seq, k)[0] if k < frames[lane] else None)
        _, odo, mp = lvo.step_batch(sw)
        for lane, g in enumerate(gs):
            if k >= frames[lane]:
                assert np.isnan(odo[lane]).all() and np.isnan(mp[lane]).all()
                continue
            assert np.array_equal(sha(sw[lane]), g[f"sweep{k}_sha"]), "synthetic generator drifted"
            n = int(g[f"f{k}_full_n"])
            for name, what in clouds.items():
                a = lvo.probe(what, lane)
                assert len(a) == int(g[f"f{k}_{name}_n"]) and np.array_equal(sha(a), g[f"f{k}_{name}_sha"]), (lane, k, name)
            for name, what in arrays.items():
                assert np.array_equal(sha(lvo.probe(what, lane)[5:n - 5]), g[f"f{k}_{name}_sha"]), (lane, k, name)
            s = lvo.stats(lane)
            w = g[f"odo{k}_world"]
            assert np.linalg.norm(odo[lane][4:] - w[4:]) < 1e-4 and rot_err(odo[lane][:4], w[:4]) < 1e-5, (lane, k)
            if f"odo{k}_counts" in g:
                got = np.stack([np.array(list(s.odo_corner_corr)[:10]) + np.array(list(s.odo_plane_corr)[:10]), list(s.odo_lm_iters)[:10]], 1)
                assert np.array_equal(got, g[f"odo{k}_counts"]), (lane, k, got.tolist(), g[f"odo{k}_counts"].tolist())
                assert np.allclose(list(s.odo_final_cost)[:10], g[f"odo{k}_cost"], rtol=1e-8, atol=1e-300)
            if not bool(g[f"mapped{k}"]):
                hf = g[f"hf{k}"]
                assert np.linalg.norm(mp[lane][4:] - hf[4:]) < 1e-4 and rot_err(mp[lane][:4], hf[:4]) < 1e-5, (lane, k)
                continue
            pose = g[f"map{k}_pose"]
            assert np.linalg.norm(mp[lane][4:] - pose[4:]) < 1e-4 and rot_err(mp[lane][:4], pose[:4]) < 1e-5, (lane, k)
            assert (s.map_corner_from_map, s.map_surf_from_map) == tuple(int(x) for x in g[f"map{k}_from_map_n"]), (lane, k)
            assert list(s.cen) == [int(x) for x in g[f"map{k}_cen"]]
            if f"map{k}_counts" in g:
                got = np.stack([np.array(list(s.map_corner_corr)[:10]) + np.array(list(s.map_surf_corr)[:10]), list(s.map_lm_iters)[:10]], 1)
                assert np.array_equal(got, g[f"map{k}_counts"]), (lane, k, got.tolist(), g[f"map{k}_counts"].tolist())
                assert np.allclose(list(s.map_final_cost)[:10], g[f"map{k}_cost"], rtol=1e-8, atol=1e-300)
            assert (s.map_corner_total, s.map_surf_total) == tuple(int(x) for x in g[f"map{k}_totals"]), (lane, k)
            assert len(lvo.probe(L.P_REGISTERED, lane)) == n
    lvo.close()


@gpu
def test_standalone_entry_points_use_lane_0_settings(lvo_mod):
    """Lane 0 of a 64-beam context configured as a VLP-16: the assertions of test_three_vlp16_frames_against_golden."""
    L = lvo_mod
    g = np.load(os.path.join(ROOT, "tests", "golden", "vlp16_seq1.npz"))
    lvo = L.Lvo(lanes=2, n_scans=64, max_map_corner=1 << 17, max_map_surf=1 << 18)
    lvo.lane_configure(0, **VLP16)
    for k in range(3):
        pts = np.concatenate([g[f"sweep{k}"], np.zeros((len(g[f"sweep{k}"]), 1), np.float32)], 1)
        st, f = lvo.extract_features(pts)
        assert st == 0
        for name in ("full", "sharp", "less_sharp", "flat", "less_flat"):
            assert len(f[name]) == int(g[f"f{k}_{name}_n"]) and np.array_equal(sha(f[name]), g[f"f{k}_{name}_sha"]), (k, name)
        assert np.array_equal(sha(lvo.probe(L.P_LABEL)), g[f"f{k}_label_sha"])
        assert np.array_equal(sha(lvo.probe(L.P_SORT_IND)), g[f"f{k}_sort_ind_sha"])
        assert np.array_equal(sha(lvo.probe(L.P_CURVATURE)), g[f"f{k}_curvature_sha"])
        st, rel, w = lvo.scan_to_scan(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
        assert st == int(g[f"odo{k}_status"])
        assert np.linalg.norm(rel[4:] - g[f"odo{k}_rel"][4:]) < 1e-4 and rot_err(rel[:4], g[f"odo{k}_rel"][:4]) < 1e-5
        assert np.linalg.norm(w[4:] - g[f"odo{k}_world"][4:]) < 1e-4 and rot_err(w[:4], g[f"odo{k}_world"][:4]) < 1e-5
        if k == 1:
            assert np.array_equal(lvo.probe(L.P_ODO_CORNER_CORR)[0], g["odo1_corner_corr0"])
            assert np.array_equal(lvo.probe(L.P_ODO_PLANE_CORR)[0], g["odo1_plane_corr0"])
        st, pose, _ = lvo.scan_to_map(f["less_sharp"], f["less_flat"], f["full"], g[f"odo{k}_world"])
        assert st == int(g[f"map{k}_status"])
        assert np.linalg.norm(pose[4:] - g[f"map{k}_pose"][4:]) < 1e-4 and rot_err(pose[:4], g[f"map{k}_pose"][:4]) < 1e-5
        assert np.array_equal(sha(lvo.probe(L.P_MAP_CORNER_STACK)), g[f"map{k}_corner_stack_sha"])
        assert np.array_equal(sha(lvo.probe(L.P_MAP_SURF_STACK)), g[f"map{k}_surf_stack_sha"])
        if k == 1 and st == 0:
            assert np.array_equal(lvo.probe(L.P_MAP_CORNER_KNN)[0], g["map1_corner_knn0"])
        s = lvo.stats()
        assert abs(s.map_corner_total - int(g[f"map{k}_totals"][0])) <= 2 and abs(s.map_surf_total - int(g[f"map{k}_totals"][1])) <= 2
    # the feature capacities of lane 0's n_scans bound the stand-alone inputs, as in a 16-beam context
    too_many = np.zeros((16 * 6 * 2 + 1, 4), np.float32)
    with pytest.raises(L.LvoError):
        lvo.scan_to_scan(too_many, f["less_sharp"], f["flat"], f["less_flat"])
    lvo.close()


@gpu
@pytest.mark.parametrize("graphs", [0, 1])
def test_configure_touches_only_its_lane(lvo_mod, sweeps, graphs):
    """Lane 1 of an HDL-64 context becomes a VLP-16 after three frames.  Lanes 0 and 2 keep their snapshot bytes and step as in a twin
    context that never made the call; lane 1 runs as a new VLP-16 context; every step launches as many kernels as the twin's."""
    L = lvo_mod
    seqs, K = (0, 1, 4), 3
    x, twin = make(L, graphs, 3), make(L, graphs, 3)
    ref16 = make(L, graphs, 1, **VLP16)
    for k in range(K):
        for y in (x, twin):
            y.step_batch([sweeps(64, s, k) for s in seqs])
    before = [x.lane_save(l) for l in (0, 2)]
    x.lane_configure(1, **VLP16)
    assert x.lane_config(1) == VLP16 and x.lane_config(0) == HDL64
    assert all(np.array_equal(x.lane_save(l), b) for l, b in zip((0, 2), before))
    for j in range(5):
        _, o, m = x.step_batch([sweeps(64, seqs[0], K + j), sweeps(16, 1, j), sweeps(64, seqs[2], K + j)])
        n = x.timings().kernel_launches
        _, to, tm = twin.step_batch([sweeps(64, s, K + j) for s in seqs])
        assert n == twin.timings().kernel_launches, j
        _, ro, rm = ref16.step_batch([sweeps(16, 1, j)])
        assert np.array_equal(o[1], ro[0]) and np.array_equal(m[1], rm[0]) and lane_state(x, 1) == lane_state(ref16, 0), j
        for lane in (0, 2):
            assert np.array_equal(o[lane], to[lane]) and np.array_equal(m[lane], tm[lane]), (j, lane)
            assert lane_state(x, lane) == lane_state(twin, lane), (j, lane)
    # lvo_lane_reset keeps the settings; a configure keeps the lane's activity; NULL restores the context's values
    x.lane_reset(1)
    assert x.lane_config(1) == VLP16
    x.set_lane_active(1, False)
    x.lane_configure(1, **dict(VLP16, n_scans=32))
    held = lane_state(x, 1)
    _, o, m = x.step_batch([sweeps(64, seqs[0], K + 5), None, sweeps(64, seqs[2], K + 5)])
    assert np.isnan(o[1]).all() and np.isnan(m[1]).all() and lane_state(x, 1) == held
    assert x.lane_config(1)["n_scans"] == 32
    x.lane_configure(1)
    assert x.lane_config(1) == HDL64
    for y in (x, twin, ref16):
        y.close()


@gpu
@pytest.mark.parametrize("graphs", [0, 1])
def test_snapshots_between_dedicated_and_configured_lanes(lvo_mod, sweeps, graphs):
    """A VLP-16 lane moves from a 16-beam context into a VLP-16-configured lane of a 64-beam context and back, continuing bit for bit."""
    L = lvo_mod
    K, N = 5, 4
    ded = make(L, graphs, 2, **VLP16)
    mix = make(L, graphs, 3)
    mix.lane_configure(2, **VLP16)
    for k in range(K):
        ded.step_batch([sweeps(16, 1, k), sweeps(16, 3, k)])
        mix.step_batch([sweeps(64, 0, k), sweeps(64, 4, k), sweeps(16, 5, k)])
    snap = ded.lane_save(0)
    mix.lane_load(2, snap)                                                # dedicated -> configured lane
    assert np.array_equal(mix.lane_save(2), snap) and mix.lane_config(2) == VLP16
    assert lane_state(mix, 2) == lane_state(ded, 0)
    for j in range(N):
        _, do, dm = ded.step_batch([sweeps(16, 1, K + j), sweeps(16, 3, K + j)])
        _, o, m = mix.step_batch([sweeps(64, 0, K + j), sweeps(64, 4, K + j), sweeps(16, 1, K + j)])
        assert np.array_equal(o[2], do[0]) and np.array_equal(m[2], dm[0]) and lane_state(mix, 2) == lane_state(ded, 0), j
    back = mix.lane_save(2)
    assert np.array_equal(back, ded.lane_save(0))                        # same sequence, same frame: same bytes
    ded.lane_load(1, back)                                                # configured lane -> dedicated
    assert np.array_equal(ded.lane_save(1), back)
    for j in range(N, 2 * N):
        _, do, dm = ded.step_batch([sweeps(16, 1, K + j), sweeps(16, 1, K + j)])
        _, o, m = mix.step_batch([sweeps(64, 0, K + j), sweeps(64, 4, K + j), sweeps(16, 1, K + j)])
        for lane in (0, 1):
            assert np.array_equal(do[lane], o[2]) and np.array_equal(dm[lane], m[2]) and lane_state(ded, lane) == lane_state(mix, 2), (j, lane)
    # a lane whose settings differ in one field refuses the snapshot and keeps its state and settings
    for field, value in (("n_scans", 32), ("minimum_range", 0.4), ("line_res", 0.3), ("plane_res", 0.5), ("skip_frame", 2)):
        mix.lane_configure(1, **dict(VLP16, **{field: value}))
        cfg, held = mix.lane_config(1), mix.lane_save(1)
        r = mix.lib.lvo_lane_load(mix.h, 1, back.ctypes.data, back.nbytes)
        assert r == L.LVO_E_BADARG and field in mix.lib.lvo_last_error(mix.h).decode(), field
        assert mix.lane_config(1) == cfg and np.array_equal(mix.lane_save(1), held), field
    for y in (ded, mix):
        y.close()


@gpu
def test_invalid_settings_leave_the_lane_unchanged(lvo_mod, sweeps):
    L = lvo_mod
    x = make(L, 0, 2)
    x.lane_configure(1, **dict(HDL64, skip_frame=2))
    for k in range(2):
        x.step_batch([sweeps(64, 0, k), sweeps(64, 1, k)])
    lib, h = x.lib, x.h

    def attempt(lane, **change):
        cfg = L.LaneConfig(**dict(HDL64, **change))
        return lib.lvo_lane_configure(h, lane, C.byref(cfg))

    held, cfg = x.lane_save(1), x.lane_config(1)
    cases = [("n_scans", v, L.LVO_E_BADARG) for v in (0, 8, 48, 128)]
    cases += [("minimum_range", v, L.LVO_E_BADARG) for v in (float("nan"), float("inf"), -0.1)]
    cases += [(f, v, L.LVO_E_BADARG) for f in ("line_res", "plane_res") for v in (0.0, -0.1, float("nan"))]
    cases += [("skip_frame", v, L.LVO_E_BADARG) for v in (0, -1)]
    for field, value, code in cases:
        assert attempt(1, **{field: value}) == code, (field, value)
        assert field in lib.lvo_last_error(h).decode(), (field, value)
        assert x.lane_config(1) == cfg and np.array_equal(x.lane_save(1), held), (field, value)
    for lane in (-1, 2):
        assert attempt(lane) == L.LVO_E_BADARG and lib.lvo_lane_configure(h, lane, None) == L.LVO_E_BADARG
        assert lib.lvo_lane_get_config(h, lane, C.byref(L.LaneConfig())) == L.LVO_E_BADARG
    x.step_batch_async([sweeps(64, 0, 2), sweeps(64, 1, 2)])
    assert attempt(1) == L.LVO_E_STATE
    x.wait()
    # n_scans above the context's: the buffers are sized for the context's n_scans
    y = make(L, 0, 2, **VLP16)
    y.step_batch([sweeps(16, 1, 0), sweeps(16, 3, 0)])
    yheld, ycfg = y.lane_save(1), y.lane_config(1)
    for n in (32, 64):
        r = y.lib.lvo_lane_configure(y.h, 1, C.byref(L.LaneConfig(**dict(VLP16, n_scans=n))))
        assert r == L.LVO_E_CAPACITY and "n_scans" in y.lib.lvo_last_error(y.h).decode(), n
        assert y.lane_config(1) == ycfg and np.array_equal(y.lane_save(1), yheld), n
    x.close(); y.close()


def test_lane_config_struct_matches_the_header(tmp_path):
    L = load_lvo()
    prog = tmp_path / "size.c"
    prog.write_text('#include "lvo.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(void){printf("%zu %zu %zu %zu %zu %zu\\n", '
                    'sizeof(lvo_lane_config), offsetof(lvo_lane_config, n_scans), offsetof(lvo_lane_config, minimum_range), '
                    'offsetof(lvo_lane_config, line_res), offsetof(lvo_lane_config, plane_res), offsetof(lvo_lane_config, skip_frame));return 0;}\n')
    exe = tmp_path / "size"
    assert os.system(f"gcc -std=c99 -Wall -Werror -I{ROOT}/include {prog} -o {exe}") == 0
    got = [int(v) for v in os.popen(str(exe)).read().split()]
    assert got == [C.sizeof(L.LaneConfig)] + [getattr(L.LaneConfig, f).offset for f in FIELDS]
