"""Feature extraction and the fused pipeline on dense rings (tests/dense_rings.py): rings of 2049..4096 less-flat candidates
(k_lessflat_voxel<256>) and rings too large for the fast path (the generic k_sector_pick with its picked flags in shared or global
memory and its sector sorts in shared memory or in the lane's sort_scratch), bit for bit against the oracle.

Two branches of k_sector_pick cannot be reached by any ring, so no fixture aims at them:
  - the joint sort of all six sectors needs 6 * next_pow2(mmax) <= 3072, i.e. mmax <= 512, but a ring with mmax <= 512 (and so
    RL <= 3079 <= 4096) takes the fast path;
  - the shared-memory less-flat sort needs at most 2048 candidates, but a generic ring has E - S >= 3067 and at most 120 of its
    points (20 per sector) are labelled sharp or less sharp, so it has at least 3067 - 120 candidates.
test_dense_rings_cpu.py checks that no fixture reaches them."""
import numpy as np
import pytest

from conftest import record_metric
from dense_rings import FIXTURES, HDL64, VLP16, make, ring_paths
from oracle_py import Oracle
from test_gpu_extract import _compare_extract
from test_gpu_golden import rot_err
from test_gpu_lane_config import observed
from test_gpu_lanes import CAPS

pytestmark = pytest.mark.gpu
MAX_POINTS = 1 << 19


def _oracle(cfg):
    return Oracle(cfg["n_scans"], cfg["minimum_range"], cfg["line_res"], cfg["plane_res"])


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_dense_ring_extraction_bit_exact(lvo_mod, synth, name):
    L = lvo_mod
    pts, _, cfg = make(synth, name)
    O = _oracle(cfg)
    record_metric(f"dense_rings/paths/{name}", sorted(set().union(*(t for _, _, t in ring_paths(O.extract(pts))))))
    lvo = L.Lvo(max_points=MAX_POINTS, **cfg)
    _compare_extract(L, lvo, O, pts, name)
    lvo.close()


def test_dense_and_sparse_sweeps_on_one_context(lvo_mod, synth):
    """Dense, standard and dense sweeps in turn on one context: nothing of a ring's path (ring_done, counters, scratch keys, picked
    flags) leaks into the next call."""
    L = lvo_mod
    lvo = L.Lvo(max_points=MAX_POINTS, **VLP16)
    O = _oracle(VLP16)
    seq = [make(synth, "boundaries")[0], synth.sweep(16, 0, 0)[0], make(synth, "vlp16_naz20000")[0], synth.sweep(16, 2, 4)[0],
           make(synth, "mixed")[0], make(synth, "vlp16_naz2700")[0], make(synth, "vlp16_naz3600")[0]]
    for k, pts in enumerate(seq):
        _compare_extract(L, lvo, O, pts, f"call {k}")
    lvo.close()


# lane -> (settings, model, seq, naz)
LANES = [(VLP16, 16, 1, 3600), (VLP16, 16, 2, 7200), (HDL64, 64, 0, 3000), (HDL64, 64, 3, None)]
FRAMES = 8


def test_dense_rings_through_the_pipeline(lvo_mod, synth):
    """Four lanes (VLP-16 at 3600 and 7200 columns, HDL-64 at 3000 and 1875) through lvo_step_batch: each lane against its own oracle
    pipeline (poses within 1e-4 m / 1e-5 rad, voxel stacks bit-exact, map sizes within 5 points as in test_gpu_mapping.py) and bit for
    bit against a dedicated one-lane context."""
    L = lvo_mod
    caps = dict(CAPS, max_points=1 << 18)
    sweeps = [[synth.sweep(model, seq, k, naz=naz)[0] for _, model, seq, naz in LANES] for k in range(FRAMES)]
    x = L.Lvo(lanes=len(LANES), **caps, **HDL64)
    for lane, (cfg, _, _, _) in enumerate(LANES):
        x.lane_configure(lane, **cfg, skip_frame=1)
    ded = [L.Lvo(**caps, **cfg) for cfg, _, _, _ in LANES]
    orcs = [_oracle(cfg) for cfg, _, _, _ in LANES]
    for k in range(FRAMES):
        _, odo, mp = x.step_batch(sweeps[k])
        for lane in range(len(LANES)):
            _, do, dm = ded[lane].step_batch([sweeps[k][lane]])
            assert np.array_equal(odo[lane], do[0]) and np.array_equal(mp[lane], dm[0]), (k, lane)
            assert observed(L, x, lane) == observed(L, ded[lane], 0), (k, lane)
            _, oo, om = orcs[lane].step(sweeps[k][lane], keep_log=True)
            assert np.linalg.norm(odo[lane][4:] - oo[4:]) < 1e-4 and rot_err(odo[lane][:4], oo[:4]) < 1e-5, (k, lane, odo[lane], oo)
            assert np.linalg.norm(mp[lane][4:] - om[4:]) < 1e-4 and rot_err(mp[lane][:4], om[:4]) < 1e-5, (k, lane, mp[lane], om)
            info = orcs[lane].mapping_info()
            for what, ref in ((L.P_MAP_CORNER_STACK, info["corner_stack"]), (L.P_MAP_SURF_STACK, info["surf_stack"])):
                got = x.probe(what, lane)
                assert got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (k, lane, what)
            s = x.stats(lane)
            assert abs(s.map_corner_total - info["info"][6]) <= 5 and abs(s.map_surf_total - info["info"][7]) <= 5, (k, lane)
    for lane in range(len(LANES)):
        assert np.array_equal(x.lane_save(lane), ded[lane].lane_save(0)), lane
    for y in [x] + ded:
        y.close()
