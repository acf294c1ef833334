"""Per-lane localisation mode (lvo_set_lane_map_update): a lane with map updates off runs process() (laserMapping.cpp:307-848) with
the insertion (:737-783) and the per-cube re-filter (:788-801) skipped, against the CPU oracle under the same switch
(tests/oracle_map_fixed.py), against a twin lane that maps, and next to lanes that keep mapping."""
import numpy as np
import pytest

from dense_map import cube_index
from oracle_map_fixed import MapFixedOracle
from oracle_py import Oracle
from test_gpu_lanes import lane_state
from test_gpu_mapping import POS_TOL, ROT_TOL, rot_err

pytestmark = pytest.mark.gpu
CAPS = dict(max_map_corner=1 << 18, max_map_surf=1 << 19)
# Prior-map recipe: largest distance between the pose of a lane localising in a map built from the same sweeps and the pose of the
# lane that built it.  The CPU oracle doing the same over frames 0-9 of HDL-64 sequences 0 and 2 stays within 0.039 m (first frame).
PLAUSIBLE_M = 0.1


class Sweeps:
    def __init__(self, synth):
        self.synth, self.cache = synth, {}

    def __call__(self, seq, frame):
        if (seq, frame) not in self.cache:
            self.cache[(seq, frame)] = self.synth.sweep(64, seq, frame)[0]
        return self.cache[(seq, frame)]


@pytest.fixture(scope="module")
def sweeps(synth):
    return Sweeps(synth)


def make(L, graphs, lanes=1, **kw):
    lvo = L.Lvo(lanes=lanes, **CAPS, **kw)
    lvo.set_option(L.LVO_OPT_GRAPHS, graphs)
    return lvo


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def maps_of(lvo, lane):
    return [lvo.map_export(lane, w) for w in (0, 1)]


def oracle_maps(o):
    return [o.map_export(w) for w in (0, 1)]


def same_maps(a, b):
    return all(np.array_equal(ca, cb) and np.array_equal(_bits(pa), _bits(pb)) for (pa, ca), (pb, cb) in zip(a, b))


def import_maps(lvo, lane, maps):
    (pc, cc), (ps, cs) = maps
    lvo.map_import(lane, pc, cc, ps, cs)


def close_pose(a, b):
    return np.linalg.norm(a[4:] - b[4:]) < POS_TOL and rot_err(a[:4], b[:4]) < ROT_TOL


def oracle_status(o, st):
    """The status the library reports for the oracle's frame: the odometry status, raised to LVO_W_MAP_TOO_SMALL (3) on a mapping frame
    whose map is too small (laserMapping.cpp:554)."""
    if o.last_frame_mapped():
        i = o.mapping_info()
        if not (len(i["corner_from_map"]) > 10 and len(i["surf_from_map"]) > 50):
            return max(st, 3)
    return st


def window_cubes(pts, cen):
    """Recipe step: each point's cube id for a lane whose cube window has centre `cen` (lvo_stats::cen), and whether the point is
    inside the 21 x 21 x 11 window at all (laserMapping.cpp:741-750)."""
    v = pts[:, :3].astype(np.float64) + 25.0
    c = np.trunc(v / 50.0).astype(np.int64) - (v < 0) + np.array(cen)
    inside = ((c >= 0) & (c < np.array([21, 21, 11]))).all(axis=1)
    return cube_index(pts, cen), inside


def stats_without_totals(lvo, lane):
    s = lvo.stats(lane)
    s.map_corner_total = s.map_surf_total = 0
    return bytes(s)


def prior_map(sweeps, seq, frames):
    """The oracle maps `frames` sweeps of `seq`; its map (the window has not moved: cube ids valid for a fresh lane)."""
    o = Oracle()
    for k in range(frames):
        o.step(sweeps(seq, k))
    assert list(o.mapping_info()["info"][3:6]) == [10, 10, 5]
    return oracle_maps(o)


@pytest.mark.parametrize("graphs", [0, 1])
def test_localise_in_prior_map_matches_oracle(lvo_mod, sweeps, graphs):
    """A lane seeded with a map built from the same sequence localises with updates off: statuses equal to the oracle's under the same
    switch, poses within the mapping tolerances, map exports and cube ids bit-identical every frame (no insertion, no float noise)."""
    L = lvo_mod
    prior = prior_map(sweeps, 0, 6)
    lvo, o = make(L, graphs), MapFixedOracle()
    import_maps(lvo, 0, prior)
    for w, (p, c) in enumerate(prior):
        o.map_import(w, p, c)
    lvo.set_lane_map_update(0, False)
    o.set_map_update(False)
    for k in range(8):
        st, odo, mp = lvo.step_batch([sweeps(0, k)])
        st_o, odo_o, mp_o = o.step(sweeps(0, k))
        assert lvo.lane_status(0) == oracle_status(o, st_o), (k, lvo.lane_status(0), st_o)
        assert close_pose(odo[0], odo_o) and close_pose(mp[0], mp_o), (k, mp[0], mp_o)
        assert same_maps(maps_of(lvo, 0), prior) and same_maps(oracle_maps(o), prior), k
        s = lvo.stats(0)
        assert (s.map_corner_total, s.map_surf_total) == (len(prior[0][0]), len(prior[1][0]))
        assert s.map_corner_corr[0] > 0 and s.map_surf_corr[0] > 0   # it registered against the map
    lvo.close()


def test_window_shifts_with_fixed_map_match_oracle(lvo_mod, synth):
    """The window-crossing path of test_cube_window_shifts_match_oracle through the stand-alone lvo_scan_to_map (which honours lane 0's
    setting) with updates off after the first frame: shifted cubes move, cubes that leave the window are dropped, the rest of the map
    is untouched; maps, cube ids, cen and totals bit-identical to the oracle's, and nothing is inserted."""
    L = lvo_mod
    O = MapFixedOracle()
    lvo = L.Lvo(**CAPS)
    f = O.extract(synth.sweep(64, 0, 0)[0])
    path = [(0, 0, 0), (120, 0, 0), (260, 0, 0), (390, 0, 0), (520, 30, 0), (390, 0, 0), (0, 0, 0), (-180, 0, 0), (-390, -40, 0), (-520, 0, 0),
            (0, 200, 0), (0, 395, 0), (0, 520, 60), (0, 520, 130), (0, 520, 210), (0, 0, 0), (0, -400, -130), (0, -560, -260), (300, 300, 100),
            (650, 300, 100), (950, 300, 100), (1250, 300, 100)]   # the last three push the map out of the window: partly, then whole
    shifted, dropped, prev_cen, prev_total = 0, 0, [10, 10, 5], None
    for k, t in enumerate(path):
        if k == 1:
            O.set_map_update(False)
            lvo.set_lane_map_update(0, False)
        odom = np.array([0, 0, 0, 1, t[0], t[1], t[2]], float)
        st_o, pose_o, corr_o = O.mapping(f["less_sharp"], f["less_flat"], None, odom)
        st_g, pose_g, _ = lvo.scan_to_map(f["less_sharp"], f["less_flat"], None, odom)
        info = O.mapping_info()["info"]
        s = lvo.stats()
        assert st_g == st_o, (k, st_g, st_o)
        assert list(s.center_cube) == list(info[:3]) and list(s.cen) == list(info[3:6]), k
        assert np.linalg.norm(pose_g[4:] - pose_o[4:]) < 1e-4, (k, pose_g, pose_o)
        lvo.set_map_correction(0, corr_o)
        assert same_maps(maps_of(lvo, 0), oracle_maps(O)), k
        total = (s.map_corner_total, s.map_surf_total)
        assert total == (info[6], info[7])
        if k >= 1:
            assert total[0] <= prev_total[0] and total[1] <= prev_total[1]   # a fixed map never grows
            dropped += total != prev_total
        shifted += list(s.cen) != prev_cen
        prev_cen, prev_total = list(s.cen), total
    assert shifted >= 8 and dropped >= 2 and prev_total == (0, 0)
    lvo.close()


@pytest.mark.parametrize("skip_frame", [1, 2])
@pytest.mark.parametrize("graphs", [0, 1])
def test_twin_lane_is_bitwise_equal(lvo_mod, sweeps, graphs, skip_frame):
    """Lane A localises with updates off; lane B maps the same sweeps and is handed A's map before every step.  The skipped blocks
    come after everything a frame reports, so the lanes agree bit for bit: poses, statuses, map correction, lvo_stats (except the two
    map totals), the registered cloud and, with the same map, the surround cloud.  A's map after each step is its map before it."""
    L = lvo_mod
    lvo = make(L, graphs, lanes=2, skip_frame=skip_frame)
    for k in range(3):
        lvo.step_batch([sweeps(0, k)] * 2)
    lvo.set_lane_map_update(0, False)
    for k in range(3, 11):
        before = maps_of(lvo, 0)
        import_maps(lvo, 1, before)
        st, odo, mp = lvo.step_batch([sweeps(0, k)] * 2)
        assert lvo.lane_status(0) == lvo.lane_status(1), k
        assert np.array_equal(odo[0], odo[1]) and np.array_equal(mp[0], mp[1]), k
        assert np.array_equal(lvo.get_map_correction(0), lvo.get_map_correction(1)), k
        assert stats_without_totals(lvo, 0) == stats_without_totals(lvo, 1), k
        reg = lvo.map_cloud_batch(L.LVO_MAP_REGISTERED)
        assert (len(reg[0]) > 0) == (k % skip_frame == 0), k   # a registered cloud on the lanes' mapping frames only
        assert np.array_equal(_bits(reg[0]), _bits(reg[1])), k
        assert same_maps(maps_of(lvo, 0), before), k
        import_maps(lvo, 1, before)
        sur = lvo.map_cloud_batch(L.LVO_MAP_SURROUND)
        assert np.array_equal(_bits(sur[0]), _bits(sur[1])), k
    lvo.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_other_lanes_are_isolated(lvo_mod, sweeps, graphs):
    """Lanes 1 and 3 of a 4-lane context localise from frame 3 on: lanes 0 and 2 stay bitwise equal to the same context with no lane
    fixed, and each fixed lane equals the same sequence in a 1-lane context."""
    L = lvo_mod
    seqs, fixed, n = (0, 1, 4, 5), (1, 3), 8
    ref, lvo = make(L, graphs, lanes=4), make(L, graphs, lanes=4)
    solo = {l: make(L, graphs) for l in fixed}
    for k in range(n):
        if k == 3:
            for l in fixed:
                lvo.set_lane_map_update(l, False)
                solo[l].set_lane_map_update(0, False)
        sw = [sweeps(s, k) for s in seqs]
        _, ro, rm = ref.step_batch(sw)
        _, o, m = lvo.step_batch(sw)
        for l in (0, 2):
            assert np.array_equal(o[l], ro[l]) and np.array_equal(m[l], rm[l]), (k, l)
            assert lane_state(lvo, l) == lane_state(ref, l), (k, l)
        for l in fixed:
            _, so, sm = solo[l].step_batch([sw[l]])
            assert np.array_equal(o[l], so[0]) and np.array_equal(m[l], sm[0]), (k, l)
            assert lane_state(lvo, l) == lane_state(solo[l], 0), (k, l)
    for c in [ref, lvo] + list(solo.values()):
        c.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_switching_mid_sequence(lvo_mod, sweeps, graphs):
    """On for frames 0-3, off for 4-7, on again from 8: the map is constant through the off phase, the whole schedule agrees with the
    oracle under the same schedule, and the launch count of a step does not change with the switches (no re-capture, no extra launch)."""
    L = lvo_mod
    lvo, o = make(L, graphs), MapFixedOracle()
    launches = []
    for k in range(11):
        on = not (4 <= k < 8)
        lvo.set_lane_map_update(0, on)
        o.set_map_update(on)
        before = maps_of(lvo, 0)
        _, odo, mp = lvo.step_batch([sweeps(2, k)])
        st_o, odo_o, mp_o = o.step(sweeps(2, k))
        assert lvo.lane_status(0) == oracle_status(o, st_o), (k, lvo.lane_status(0), st_o)
        assert close_pose(odo[0], odo_o) and close_pose(mp[0], mp_o), (k, mp[0], mp_o)
        after = maps_of(lvo, 0)
        assert same_maps(after, before) == (not on), k
        s = lvo.stats(0)
        info = o.mapping_info()["info"]
        assert abs(s.map_corner_total - info[6]) <= max(5, 2e-3 * info[6]) and abs(s.map_surf_total - info[7]) <= max(5, 2e-3 * info[7]), k
        if k:
            launches.append(lvo.timings().kernel_launches)
    if graphs:
        assert len(set(launches)) == 1, launches
    lvo.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_prior_map_recipe(lvo_mod, sweeps, graphs):
    """INTEGRATION.md, "Localisation in a prior map": lane A maps a sequence; its map goes through the recipe (cube ids recomputed for
    the destination lane's cen, points outside the window dropped, lvo_map_import, lvo_set_map_correction, updates off) into a fresh
    lane of another context, which localises the same sweeps: within tolerance of the oracle doing the same, and within PLAUSIBLE_M
    of A's poses."""
    L = lvo_mod
    n = 8
    a = make(L, graphs)
    pa = [a.step_batch([sweeps(0, k)])[2][0] for k in range(n)]
    src = maps_of(a, 0)
    a.close()
    lvo = make(L, graphs, lanes=3)
    dst = 2
    cen = [10, 10, 5]   # the window of a fresh lane; lvo_stats::cen reports it from the lane's first mapping frame on
    recipe = []
    for pts, _ in src:
        cube, inside = window_cubes(pts, cen)
        recipe.append((pts[inside], cube[inside]))
    import_maps(lvo, dst, recipe)
    lvo.set_map_correction(dst, np.array([0, 0, 0, 1, 0, 0, 0], float))
    lvo.set_lane_map_update(dst, False)
    for l in range(3):
        if l != dst:
            lvo.set_lane_active(l, False)
    o = MapFixedOracle()
    for w, (p, c) in enumerate(recipe):
        o.map_import(w, p, c)
    o.set_map_update(False)
    for k in range(n):
        _, odo, mp = lvo.step_batch([None, None, sweeps(0, k)])
        st_o, odo_o, mp_o = o.step(sweeps(0, k))
        assert lvo.lane_status(dst) == oracle_status(o, st_o), (k, lvo.lane_status(dst), st_o)
        assert close_pose(mp[dst], mp_o), (k, mp[dst], mp_o)
        assert np.linalg.norm(mp[dst][4:] - pa[k][4:]) < PLAUSIBLE_M, (k, mp[dst], pa[k])
        assert same_maps(maps_of(lvo, dst), recipe), k
    lvo.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_flag_survives_lane_calls_and_not_in_snapshot(lvo_mod, sweeps, graphs):
    """The setting is host state: lvo_lane_reset, lvo_lane_configure, lvo_lane_load and activity changes leave it as it is, and two
    lanes with the same history give the same lvo_lane_save bytes whatever their setting."""
    L = lvo_mod
    lvo = make(L, graphs, lanes=2)
    for k in range(3):
        lvo.step_batch([sweeps(1, k)] * 2)
    lvo.set_lane_map_update(0, False)
    assert np.array_equal(lvo.lane_save(0), lvo.lane_save(1))
    snap = lvo.lane_save(1)
    prior = maps_of(lvo, 1)
    frame = [3]

    def step_keeps_map_of_lane0():
        before = maps_of(lvo, 0)
        lvo.step_batch([sweeps(1, frame[0])] * 2)
        frame[0] += 1
        return same_maps(maps_of(lvo, 0), before)

    assert step_keeps_map_of_lane0()
    lvo.lane_reset(0)
    import_maps(lvo, 0, prior)
    assert step_keeps_map_of_lane0()
    lvo.lane_configure(0)
    import_maps(lvo, 0, prior)
    assert step_keeps_map_of_lane0()
    lvo.lane_load(0, snap)
    assert step_keeps_map_of_lane0()
    lvo.set_lane_active(0, False)
    lvo.step_batch([None, sweeps(1, frame[0])])
    lvo.set_lane_active(0, True)
    assert step_keeps_map_of_lane0()
    lvo.set_lane_map_update(0, True)
    assert not step_keeps_map_of_lane0()
    lvo.close()


def test_errors_change_nothing(lvo_mod, sweeps):
    """A bad lane gives LVO_E_BADARG, a call while an *_async step is in flight LVO_E_STATE; neither changes a lane's setting."""
    L = lvo_mod
    lvo = make(L, 0, lanes=2)
    lib, h = lvo.lib, lvo.h
    for k in range(2):
        lvo.step_batch([sweeps(0, k)] * 2)
    for lane in (-1, 2, 1 << 20):
        assert lib.lvo_set_lane_map_update(h, lane, 0) == L.LVO_E_BADARG
    assert lib.lvo_set_lane_map_update(None, 0, 0) == L.LVO_E_BADARG
    lvo.step_batch_async([sweeps(0, 2)] * 2)
    assert lib.lvo_set_lane_map_update(h, 0, 0) == L.LVO_E_STATE
    lvo.wait()
    before = maps_of(lvo, 0)
    lvo.step_batch([sweeps(0, 3)] * 2)
    assert not same_maps(maps_of(lvo, 0), before)   # lane 0 still maps
    lvo.set_lane_map_update(1, False)
    lvo.step_batch_async([sweeps(0, 4)] * 2)
    assert lib.lvo_set_lane_map_update(h, 1, 1) == L.LVO_E_STATE
    lvo.wait()
    before = maps_of(lvo, 1)
    lvo.step_batch([sweeps(0, 5)] * 2)
    assert same_maps(maps_of(lvo, 1), before)       # lane 1 still localises
    lvo.close()
