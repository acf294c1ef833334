"""One 128-lane context, the lane count bench.py and fleet users run, against per-lane references.

128 lanes run 32 sequence descriptors from four start frames each: VLP-16, HDL-32 and HDL-64 settings, mapping_skip_frame 1, 2 and 3,
VLP-16 rings of up to 7200 columns (113 k points, within max_points = 131072), lanes that go idle for two frames, lanes that localise
in an imported map with updates off, and lanes that map into an imported dense map (tests/dense_map.py).  Eight frames go through
lvo_step_batch_dev and, as a second case, lvo_step_batch_pipelined (CUDA graphs are off above 8 lanes).

Every lane must equal, bit for bit, a one-lane replay of its own sequence: everything lane_state observes after every frame (held
while the lane is idle), the poses, and at the end the ring probes, the batched map outputs and the lvo_lane_save bytes.  The replays
of five lanes (first, 63, last, a 7200-column lane and a skip_frame-3 lane) are checked against the oracle.

Some code paths only run at this width, so the test also asserts from lvo_stats and its own inputs that a step crossed them:
  - k_vx_seg_offsets walks the re-filter's 77 segments per lane and type in chunks of 1024: the second chunk needs 7 or more lanes
    mapping in one step;
  - k_sort_onesweep takes more than one tile per block only above 592 x 4096 items; the re-filter of a step sorts, for each lane that
    maps with updates on and for each type, the map points of its valid cubes plus its downsampled stack (k_refilter_offsets)."""
import hashlib

import numpy as np
import pytest

from conftest import record_metric
from dense_map import make_dense_map
from oracle_py import Oracle
from test_gpu_golden import rot_err
from test_gpu_lane_config import HDL64, VLP16, observed
from test_gpu_lanes import lane_state

pytestmark = pytest.mark.gpu
LANES, FRAMES, STARTS = 128, 8, 4
CAPS = dict(max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 20)
H32 = dict(VLP16, n_scans=32, line_res=0.3, plane_res=0.6)
V2, V3, H2, H3 = dict(VLP16, skip_frame=2), dict(VLP16, skip_frame=3), dict(HDL64, skip_frame=2), dict(HDL64, skip_frame=3)
# (model, seq, azimuth columns or None for the model's default, settings, kind): kind "fixed" localises in the dense map with updates
# off, "dense" maps into it, "idle" pauses for two frames
DESCRIPTORS = (
    [(64, s, None, cfg, None) for s, cfg in enumerate([HDL64, HDL64, H2, H3, HDL64, H2, HDL64, HDL64, H3, HDL64])]
    + [(16, s, None, cfg, None) for s, cfg in enumerate([VLP16, V2, V3, H32, VLP16, H32, VLP16, VLP16])]
    + [(16, 10, 3600, VLP16, None), (16, 11, 7200, VLP16, None), (16, 12, 2700, V3, None), (16, 13, 7200, V2, None),
       (16, 14, 3600, H32, None), (16, 15, 5000, VLP16, None)]
    + [(64, 20, None, HDL64, "fixed"), (16, 21, None, VLP16, "fixed"), (64, 22, None, HDL64, "dense"), (64, 23, None, HDL64, "dense")]
    + [(64, 24, None, HDL64, "idle"), (16, 25, None, V2, "idle"), (64, 26, None, H3, "idle"), (16, 27, 3600, VLP16, "idle")])
assert len(DESCRIPTORS) * STARTS == LANES
ORACLE_LANES = (0, 63, LANES - 1, 19, 3)   # lane 19: VLP-16 at 7200 columns; lane 3: HDL-64 with skip_frame 3


def lane_desc(lane):
    """(model, seq, naz, settings, kind, start frame) of a lane."""
    return DESCRIPTORS[lane % len(DESCRIPTORS)] + (lane // len(DESCRIPTORS),)


def idle_frames(lane):
    _, _, _, _, kind, start = lane_desc(lane)
    return {1 + start, 2 + start} if kind == "idle" else set()


def schedule(lane):
    """Per frame of the context: the index of the sweep the lane consumes, or None while it is idle."""
    out, j = [], 0
    for k in range(FRAMES):
        if k in idle_frames(lane):
            out.append(None)
        else:
            out.append(j)
            j += 1
    return out


def digest(d):
    return {k: hashlib.sha256(v if isinstance(v, bytes) else repr(v).encode()).hexdigest() for k, v in d.items()}


class Fleet:
    def __init__(self, synth):
        self.synth, self.cache = synth, {}
        self.dense = make_dense_map()

    def sweep(self, lane, j):
        model, seq, naz, _, _, start = lane_desc(lane)
        key = (model, seq, naz, start + j)
        if key not in self.cache:
            self.cache[key] = self.synth.sweep(model, seq, start + j, naz=naz)[0]
        return self.cache[key]

    def prepare(self, lvo, slot, lane):
        """Lane `slot` of `lvo` starts `lane`'s sequence: settings, imported map, map updates."""
        _, _, _, cfg, kind, _ = lane_desc(lane)
        lvo.lane_configure(slot, **cfg)
        if kind in ("fixed", "dense"):
            lvo.map_import(slot, *self.dense)
        lvo.set_lane_map_update(slot, kind != "fixed")


@pytest.fixture(scope="module")
def fleet(synth, lvo_mod):
    """The fleet's inputs and the one-lane replay of every lane: per consumed sweep (odometry row, mapping row, lane_state digest), and
    at the end the observed() digest and the lane_save bytes.  One context per settings, reused through lane_configure."""
    L = lvo_mod
    f = Fleet(synth)
    solo = {}
    f.replay = []
    for lane in range(LANES):
        model, seq, naz, cfg, kind, start = lane_desc(lane)
        key = tuple(sorted(cfg.items()))
        if key not in solo:
            solo[key] = L.Lvo(lanes=1, **CAPS, **cfg)
        x = solo[key]
        f.prepare(x, 0, lane)
        orc = None
        if lane in ORACLE_LANES:
            assert kind in (None, "idle")
            orc = Oracle(cfg["n_scans"], cfg["minimum_range"], cfg["line_res"], cfg["plane_res"])
            orc.set_skip_frame(cfg["skip_frame"])
        steps = []
        for j in range(sum(s is not None for s in schedule(lane))):
            pts = f.sweep(lane, j)
            _, o, m = x.step_batch([pts])
            steps.append((o[0], m[0], digest(lane_state(x, 0))))
            if orc is not None:
                _, oo, om = orc.step(pts)
                if not orc.last_frame_mapped():
                    om = orc.high_freq
                assert np.linalg.norm(o[0][4:] - oo[4:]) < 1e-4 and rot_err(o[0][:4], oo[:4]) < 1e-5, (lane, j, o[0], oo)
                assert np.linalg.norm(m[0][4:] - om[4:]) < 1e-4 and rot_err(m[0][:4], om[:4]) < 1e-5, (lane, j, m[0], om)
        f.replay.append((steps, digest(observed(L, x, 0)), x.lane_save(0)))
    for x in solo.values():
        x.close()
    return f


@pytest.mark.parametrize("mode", ["dev", "pipelined"])
def test_128_lanes_equal_one_lane_replays(lvo_mod, fleet, mode):
    import torch
    L = lvo_mod
    x = L.Lvo(lanes=LANES, **CAPS, **HDL64)
    for lane in range(LANES):
        fleet.prepare(x, lane, lane)
    sched = [schedule(lane) for lane in range(LANES)]
    frames = [[None if sched[l][k] is None else fleet.sweep(l, sched[l][k]) for l in range(LANES)] for k in range(FRAMES)]
    max_mapping, max_items = 0, 0
    for k in range(FRAMES):
        for lane in range(LANES):
            x.set_lane_active(lane, frames[k][lane] is not None)
        if mode == "dev":
            dev = [None if s is None else torch.from_numpy(s).cuda() for s in frames[k]]
            torch.cuda.synchronize()
            _, o, m = x.step_batch_dev([None if d is None else d.data_ptr() for d in dev], [None if d is None else d.shape[0] for d in dev])
        else:
            _, o, m = x.step_batch_pipelined(frames[k], frames[k + 1] if k + 1 < FRAMES else None)
        # lanes that mapped in this step: by the inputs (the lane's own step count and skip_frame) and as the library reports them
        registered = x.map_cloud_batch_dev(L.LVO_MAP_REGISTERED, [None] * LANES, [0] * LANES)
        mapping, items = 0, 0
        for lane in range(LANES):
            j = sched[lane][k]
            steps = fleet.replay[lane][0]
            if j is None:
                assert np.isnan(o[lane]).all() and np.isnan(m[lane]).all() and registered[lane] == 0, (mode, k, lane)
                prev = [i for i in sched[lane][:k] if i is not None][-1]
                assert digest(lane_state(x, lane)) == steps[prev][2], (mode, k, lane)
                continue
            ro, rm, rs = steps[j]
            assert np.array_equal(o[lane], ro) and np.array_equal(m[lane], rm), (mode, k, lane)
            got = digest(lane_state(x, lane))
            assert got == rs, (mode, k, lane, [key for key in rs if got[key] != rs[key]])
            maps = j % lane_desc(lane)[3]["skip_frame"] == 0
            assert (registered[lane] > 0) == maps, (mode, k, lane, registered[lane])
            if maps:
                mapping += 1
                if lane_desc(lane)[4] != "fixed":
                    s = x.stats(lane)
                    items += s.map_corner_from_map + s.map_corner_stack + s.map_surf_from_map + s.map_surf_stack
        max_mapping, max_items = max(max_mapping, mapping), max(max_items, items)
    for lane in range(LANES):
        _, obs, snap = fleet.replay[lane]
        got = digest(observed(L, x, lane))
        assert got == obs, (mode, lane, [key for key in obs if got[key] != obs[key]])
        assert np.array_equal(x.lane_save(lane), snap), (mode, lane)
    x.close()
    record_metric(f"fleet_scale/{mode}", {"lanes": LANES, "max_lanes_mapping_in_one_step": max_mapping,
                                          "max_refilter_items_in_one_step": int(max_items), "onesweep_one_tile_per_block_limit": 592 * 4096})
    print(f"{mode}: up to {max_mapping} lanes mapped in one step, up to {max_items} re-filter items (one tile per block up to {592 * 4096})")
    assert max_mapping >= 7, "k_vx_seg_offsets' second chunk of 1024 segments needs 7 or more lanes mapping in one step"
    assert max_items > 592 * 4096, "k_sort_onesweep takes several tiles per block only above 592 x 4096 items"


def test_idle_lane_snapshot_ignores_the_other_lanes(lvo_mod, synth):
    """An idle lane's snapshot bytes stay what they were while the other lanes step and map: the odometry and mapping stages skip it
    by its lane flags and write none of its state (they once stored a per-frame skip flag into it)."""
    L = lvo_mod
    x = L.Lvo(lanes=2, **CAPS, **HDL64)
    x.lane_configure(1, **H3)
    for k in range(4):
        x.step_batch([synth.sweep(64, 0, k)[0], synth.sweep(64, 1, k)[0]])
    held = x.lane_save(1)
    x.set_lane_active(1, False)
    for k in range(4, 6):
        x.step_batch([synth.sweep(64, 0, k)[0], None])
        assert np.array_equal(x.lane_save(1), held), k
    x.close()
