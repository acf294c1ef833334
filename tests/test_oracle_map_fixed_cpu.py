"""CPU tests (no GPU) of the oracle's fixed-map mode (tests/oracle_map_fixed.py), the definition behind lvo_set_lane_map_update: a
frame with map updates off runs process() with the insertion (laserMapping.cpp:737-783) and the per-cube re-filter (:788-801) skipped."""
import numpy as np

from oracle_map_fixed import MapFixedOracle, shift_cubes
from oracle_py import Oracle, Synth


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _maps(o):
    return [o.map_export(w) for w in (0, 1)]


def _same_maps(a, b):
    return all(np.array_equal(ca, cb) and np.array_equal(_bits(pa), _bits(pb)) for (pa, ca), (pb, cb) in zip(a, b))


def test_fixed_map_does_not_change_and_insertion_resumes():
    """Map built for 4 frames, then 4 frames with updates off (the window does not move on this sequence): the exports are
    byte-identical from frame to frame while the pose keeps being estimated against the map.  Switched back on, insertion resumes."""
    s, o = Synth(), MapFixedOracle()
    for k in range(4):
        o.step(s.sweep(64, 0, k)[0])
    o.set_map_update(False)
    before = _maps(o)
    cen = o.cen().copy()
    for k in range(4, 8):
        st, _, pose = o.step(s.sweep(64, 0, k)[0])
        assert st == 0 and o.last_frame_mapped()
        assert list(o.cen()) == list(cen)
        assert _same_maps(_maps(o), before), k
        assert o.mapping_log(0)["counts"][:2].sum() > 100   # it registered against the map
    assert np.linalg.norm(pose[4:]) > 3.0                     # and it moved
    o.set_map_update(True)
    o.step(s.sweep(64, 0, 8)[0])
    after = _maps(o)
    assert not _same_maps(after, before)
    assert len(after[1][0]) > len(before[1][0])               # the new sweep's surf points went into the map


def test_twin_oracle_poses_are_identical():
    """The skipped blocks run after everything a frame reports: a fixed-map oracle and an updating oracle that is handed the fixed
    map before every frame give bit-identical poses and map corrections."""
    s = Synth()
    a, b = MapFixedOracle(), Oracle()
    for k in range(3):
        sw = s.sweep(64, 0, k)[0]
        a.step(sw); b.step(sw)
    a.set_map_update(False)
    for k in range(3, 7):
        for w, (p, c) in enumerate(_maps(a)):
            b.map_import(w, p, c)
        sw = s.sweep(64, 0, k)[0]
        ra, rb = a.step(sw), b.step(sw)
        assert ra[0] == rb[0] and np.array_equal(ra[1], rb[1]) and np.array_equal(ra[2], rb[2]), k
        assert np.array_equal(a.high_freq, b.high_freq)
        assert np.array_equal(_bits(a.mapping_info()["registered"]), _bits(b.mapping_info()["registered"]))


def test_shift_cubes_matches_the_oracle_window_shift():
    """shift_cubes restates the cube-window shift (:312-507).  Checked against the oracle itself on frames that insert nothing (empty
    feature clouds) and whose valid cubes are empty (the re-filter has nothing to do): there the updating oracle's map after the frame
    is exactly the shifted map before it."""
    o = Oracle()
    f = o.extract(Synth().sweep(64, 0, 0)[0])
    o.mapping(f["less_sharp"], f["less_flat"], None, np.array([0, 0, 0, 1, 0, 0, 0], float))
    empty = np.zeros((0, 4), np.float32)
    path = [(120, 0, 0), (260, 0, 0), (390, 0, 0), (520, 30, 0), (390, 0, 0), (-180, 0, 0), (-390, -40, 0), (-520, 0, 0),
            (0, 395, 0), (0, 520, 130), (0, 520, 210), (0, -400, -130), (0, -560, -260)]
    checked = 0
    for t in path:
        cen0 = o.mapping_info()["info"][3:6].copy()
        prev = _maps(o)
        o.mapping(empty, empty, None, np.array([0, 0, 0, 1, *t], float))
        info = o.mapping_info()
        if len(info["corner_from_map"]) or len(info["surf_from_map"]):
            continue
        d = info["info"][3:6] - cen0
        want = [shift_cubes(p, c, d) for p, c in prev]
        assert _same_maps(_maps(o), want), t
        checked += bool(d.any())
    assert checked >= 6
