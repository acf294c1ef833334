"""Per-lane sequence lifecycle of the batched pipeline: lvo_set_lane_active (idle lanes) and lvo_lane_reset.

An idle lane is skipped by every lvo_step_batch* call and resumes its sequence bit for bit; a reset lane starts a new sequence
exactly like lane l of a new context, on its own skip_frame phase; the other lanes of the context never notice.  "Equal" below is
bitwise: poses, statuses, lvo_stats bytes, both map exports (points and cube ids), both map clouds and the map correction."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
CAPS = dict(max_map_corner=1 << 18, max_map_surf=1 << 19)
SEQ = (0, 1, 4)      # sequence of lanes 0, 1, 2
SEQ_B = 5            # the sequence a reset lane starts


class Sweeps:
    """Synthetic HDL-64 sweeps, generated once per (sequence, frame)."""

    def __init__(self, synth):
        self.synth, self.cache = synth, {}

    def __call__(self, seq, frame):
        if (seq, frame) not in self.cache:
            self.cache[(seq, frame)] = self.synth.sweep(64, seq, frame)[0]
        return self.cache[(seq, frame)]


@pytest.fixture(scope="module")
def sweeps(synth):
    return Sweeps(synth)


def make(L, graphs, lanes=3, **kw):
    lvo = L.Lvo(lanes=lanes, **CAPS, **kw)
    lvo.set_option(L.LVO_OPT_GRAPHS, graphs)
    return lvo


def lane_state(lvo, lane):
    """Everything a caller can observe of one lane, as bytes."""
    st = lvo.stats(lane)
    d = {"stats": bytes(st), "status": lvo.lane_status(lane), "corr": lvo.get_map_correction(lane).tobytes()}
    for which in (0, 1):
        pts, cube = lvo.map_export(lane, which)
        d[f"export{which}"] = pts.tobytes() + cube.tobytes()
        d[f"cloud{which}"] = lvo.map_cloud(lane, which).tobytes()
    return d


def probes(L, lvo, lane):
    return {w: lvo.probe(w, lane).tobytes() for w in (L.P_LESS_FLAT, L.P_REGISTERED, L.P_MAP_SURF_STACK, L.P_ODO_LM_TRACE)}


def worst(statuses):
    w = 0
    for s in statuses:
        if s < 0:
            w = s
        elif w >= 0:
            w = max(w, s)
    return w


def hf_pose(corr, odo):
    """High-frequency pose q_wmap_wodom * odometry (laserMapping.cpp:214-215), in the operation order of the library's host code."""
    a, b = corr[:4], odo[:4]
    q = [a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1], a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2],
         a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0], a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2]]
    v = odo[4:]
    uv = [2 * (a[1] * v[2] - a[2] * v[1]), 2 * (a[2] * v[0] - a[0] * v[2]), 2 * (a[0] * v[1] - a[1] * v[0])]
    t = [v[0] + a[3] * uv[0] + (a[1] * uv[2] - a[2] * uv[1]) + corr[4], v[1] + a[3] * uv[1] + (a[2] * uv[0] - a[0] * uv[2]) + corr[5],
         v[2] + a[3] * uv[2] + (a[0] * uv[1] - a[1] * uv[0]) + corr[6]]
    return np.array(q + t, np.float64)


def run_reference(L, graphs, seqs, frames, sweeps, **kw):
    """Every lane l runs seqs[l] from frame 0 without interruption: per step (status per lane, odometry rows, mapping rows, lane_state)."""
    ref = make(L, graphs, lanes=len(seqs), **kw)
    out = []
    for k in range(frames):
        _, o, m = ref.step_batch([sweeps(s, k) for s in seqs])
        out.append(([ref.lane_status(l) for l in range(len(seqs))], o, m, [lane_state(ref, l) for l in range(len(seqs))]))
    ref.close()
    return out


def same_step(ref_step, lane, lvo, o, m):
    st, ro, rm, rs = ref_step
    assert np.array_equal(o[lane], ro[lane]) and np.array_equal(m[lane], rm[lane])
    assert lane_state(lvo, lane) == rs[lane]


@pytest.mark.parametrize("skip_frame", [1, 2])
@pytest.mark.parametrize("graphs", [0, 1])
def test_pause_and_resume(lvo_mod, sweeps, graphs, skip_frame):
    """With skip_frame = 2 the pause has odd length: lane 1 resumes with its own frame 3, which does not map, on an even context
    frame, on which lanes 0 and 2 map.  Had its phase advanced while idle, the comparison with the reference would fail."""
    L = lvo_mod
    idle = range(3, 6)
    n = 12
    ref = run_reference(L, graphs, SEQ, n, sweeps, skip_frame=skip_frame)
    x = make(L, graphs, skip_frame=skip_frame)
    f1 = 0               # lane 1's own frame counter
    before = None
    for k in range(n):
        if k == idle.start:
            x.set_lane_active(1, False)
            before = (lane_state(x, 1), probes(L, x, 1))
        if k == idle.stop:
            x.set_lane_active(1, True)
        active1 = k not in idle
        r, o, m = x.step_batch([sweeps(SEQ[0], k), sweeps(SEQ[1], f1) if active1 else None, sweeps(SEQ[2], k)])
        for lane in (0, 2):
            same_step(ref[k], lane, x, o, m)
        if active1:
            same_step(ref[f1], 1, x, o, m)
            assert r == worst([ref[k][0][0], ref[f1][0][1], ref[k][0][2]]), k
            if skip_frame == 2 and f1 % 2:                              # its own odd frames: high-frequency pose, no mapping
                assert np.array_equal(m[1], hf_pose(x.get_map_correction(1), o[1])), k
            f1 += 1
        else:
            assert np.isnan(o[1]).all() and np.isnan(m[1]).all()      # not written
            assert (lane_state(x, 1), probes(L, x, 1)) == before, k
            assert r == worst([ref[k][0][0], ref[k][0][2]]), k        # the active lanes only
    assert f1 == n - len(idle)
    x.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_reset_starts_a_new_sequence(lvo_mod, sweeps, graphs):
    L = lvo_mod
    n_a, n_b = 4, 6
    ref_b = run_reference(L, graphs, (SEQ_B,) * 3, n_b, sweeps)          # B from frame 0 in a new context
    ref = run_reference(L, graphs, SEQ, n_a + n_b, sweeps)               # lanes 0 and 2 without any reset beside them
    fresh = make(L, graphs)
    fresh_state = lane_state(fresh, 1)
    fresh.close()
    x = make(L, graphs)
    for k in range(n_a + n_b):
        if k == n_a:
            x.lane_reset(1)
            assert lane_state(x, 1) == fresh_state                       # stats, status, map and correction of a new context
        s1 = sweeps(SEQ[1], k) if k < n_a else sweeps(SEQ_B, k - n_a)
        r, o, m = x.step_batch([sweeps(SEQ[0], k), s1, sweeps(SEQ[2], k)])
        for lane in (0, 2):
            same_step(ref[k], lane, x, o, m)
        if k >= n_a:
            same_step(ref_b[k - n_a], 1, x, o, m)
            if k == n_a:
                assert x.stats(1).odo_outer_executed == 0                # the odometry only initialised: its first frame
    x.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_reset_lane_follows_its_own_skip_frame_phase(lvo_mod, sweeps, graphs):
    L = lvo_mod
    n_a, n_b = 3, 6                                                      # reset at context frame 3: odd
    ref_b = run_reference(L, graphs, (SEQ_B,) * 3, n_b, sweeps, skip_frame=2)
    ref = run_reference(L, graphs, SEQ, n_a + n_b, sweeps, skip_frame=2)
    x = make(L, graphs, skip_frame=2)
    for k in range(n_a + n_b):
        if k == n_a:
            x.lane_reset(1)
        s1 = sweeps(SEQ[1], k) if k < n_a else sweeps(SEQ_B, k - n_a)
        _, o, m = x.step_batch([sweeps(SEQ[0], k), s1, sweeps(SEQ[2], k)])
        for lane in (0, 2):                                              # context phase: they map on even context frames
            same_step(ref[k], lane, x, o, m)
        if k >= n_a:
            j = k - n_a
            same_step(ref_b[j], 1, x, o, m)
            if j % 2:                                                    # own odd frame: no mapping, high-frequency pose
                assert np.array_equal(m[1], hf_pose(x.get_map_correction(1), o[1])), j
            else:                                                        # own frames 0, 2, 4 map (odd context frames)
                assert x.stats(1).map_corner_stack > 0, j
    x.close()


class Runner:
    """Steps one context through a schedule with one of the batched entry points."""

    def __init__(self, L, graphs, mode, distortion):
        self.L, self.mode = L, mode
        self.lvo = make(L, graphs, distortion=distortion)

    def step(self, sw, nxt):
        lvo = self.lvo
        if self.mode == "plain":
            return lvo.step_batch(sw)
        if self.mode == "async":
            lvo.step_batch_async(sw)
            return lvo.wait()
        if self.mode == "pipelined":
            self.keep = nxt          # handed over by pointer until the next call
            return lvo.step_batch_pipelined(sw, nxt)
        import torch
        dev = [torch.from_numpy(s).cuda() if s is not None else None for s in sw]
        torch.cuda.synchronize()
        return lvo.step_batch_dev([d.data_ptr() if d is not None else None for d in dev], [d.shape[0] if d is not None else None for d in dev])


@pytest.mark.parametrize("distortion", [0, 2])
@pytest.mark.parametrize("graphs", [0, 1])
def test_entry_points_agree(lvo_mod, sweeps, graphs, distortion):
    """Pause of lane 1 for steps 3-5 and reset of lane 2 into sequence B before step 7, through every batched entry point.  The
    pipelined prefetches include one staged while lane 1 was active and consumed while it is idle (step 2 -> 3) and the reverse (5 -> 6)."""
    L = lvo_mod
    n, idle, reset_at = 10, range(3, 6), 7
    frames = []
    f1 = 0
    for k in range(n):
        a1 = k not in idle
        s2 = sweeps(SEQ[2], k) if k < reset_at else sweeps(SEQ_B, k - reset_at)
        frames.append([sweeps(SEQ[0], k), sweeps(SEQ[1], f1) if a1 else None, s2])
        f1 += a1
    # what the caller hands over as "next" before it knows about the pause / resume: lane 1's next frame of its sequence
    nexts = [list(frames[k + 1]) if k + 1 < n else None for k in range(n)]
    nexts[idle.start - 1][1] = sweeps(SEQ[1], idle.start)               # prefetched while active, consumed while idle
    nexts[idle.stop - 1][1] = frames[idle.stop][1]                      # prefetched while idle (not read), consumed after resume
    runs = {mode: Runner(L, graphs, mode, distortion) for mode in ("plain", "async", "pipelined", "dev")}
    results = {mode: [] for mode in runs}
    for k in range(n):
        for mode, run in runs.items():
            if k == idle.start:
                run.lvo.set_lane_active(1, False)
            if k == idle.stop:
                run.lvo.set_lane_active(1, True)
            if k == reset_at:
                run.lvo.lane_reset(2)
            r, o, m = run.step(frames[k], nexts[k])
            results[mode].append((r, o.tobytes(), m.tobytes(), [run.lvo.lane_status(l) for l in range(3)]))
    for mode, run in runs.items():
        assert results[mode] == results["plain"], mode
        if mode != "plain":
            for lane in range(3):
                assert lane_state(run.lvo, lane) == lane_state(runs["plain"].lvo, lane), (mode, lane)
                assert probes(L, run.lvo, lane) == probes(L, runs["plain"].lvo, lane), (mode, lane)
    for run in runs.values():
        run.lvo.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_errors_and_standalone_calls_after_an_idle_lane(lvo_mod, sweeps, graphs):
    L = lvo_mod
    x = make(L, graphs)
    lib, h = x.lib, x.h
    for lane in (-1, 3):
        assert lib.lvo_set_lane_active(h, lane, 0) == L.LVO_E_BADARG
        assert lib.lvo_lane_reset(h, lane) == L.LVO_E_BADARG
    x.step_batch_async([sweeps(s, 0) for s in SEQ])
    assert lib.lvo_set_lane_active(h, 1, 0) == L.LVO_E_STATE          # a step in flight
    assert lib.lvo_lane_reset(h, 1) == L.LVO_E_STATE
    x.wait()
    # an idle lane's view is not read: NULL data with points and a stride no active lane has
    x.set_lane_active(0, False)
    views = (L.CloudView * 3)(L.CloudView(None, 123, 48, 4, 0), L.view_of(sweeps(SEQ[1], 1))[0], L.view_of(sweeps(SEQ[2], 1))[0])
    keep = [sweeps(SEQ[1], 1), sweeps(SEQ[2], 1)]
    po, pm = (L.Pose * 3)(), (L.Pose * 3)()
    assert lib.lvo_step_batch(h, views, po, pm) >= 0, lib.lvo_last_error(h)
    del keep
    # no lane active: nothing to do, LVO_OK
    for lane in (1, 2):
        x.set_lane_active(lane, False)
    assert x.step_batch([None, None, None])[0] == L.LVO_OK
    # the stand-alone stage calls on lane 0 behave as on a context that never had an idle lane.  Before each of them a batched step
    # in which lane 0 is idle (every lane is) leaves "lane 0 idle, not mapping" in the device's lane flags; the reset only gives lane 0
    # the odometry state and the empty map of a new context.
    x.lane_reset(0)
    y = make(L, graphs)
    idle_step = lambda: x.step_batch([None, None, None])
    for k in range(3):
        idle_step()
        rx, fx = x.extract_features(sweeps(SEQ[0], k))
        ry, fy = y.extract_features(sweeps(SEQ[0], k))
        assert rx == ry and all(np.array_equal(fx[n].view(np.uint32), fy[n].view(np.uint32)) for n in fx), k
        feats = [fx[n] for n in ("sharp", "less_sharp", "flat", "less_flat")]
        idle_step()
        ox, ox1, ox2 = x.scan_to_scan(*feats)
        oy, oy1, oy2 = y.scan_to_scan(*feats)
        assert ox == oy and np.array_equal(ox1, oy1) and np.array_equal(ox2, oy2), k
        idle_step()
        mx, px, gx = x.scan_to_map(fx["less_sharp"], fx["less_flat"], fx["full"], ox2, want_registered=True)
        my, py, gy = y.scan_to_map(fx["less_sharp"], fx["less_flat"], fx["full"], oy2, want_registered=True)
        assert mx == my and np.array_equal(px, py) and np.array_equal(gx.view(np.uint32), gy.view(np.uint32)), k
    assert x.stats(0).map_outer_executed > 0                           # the last scan_to_map solved against a map
    for which in (0, 1):
        assert x.map_export(0, which)[0].tobytes() == y.map_export(0, which)[0].tobytes()
    x.close(); y.close()
