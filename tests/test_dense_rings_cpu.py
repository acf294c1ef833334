"""Dense-ring fixtures (tests/dense_rings.py) on the CPU: the generator's default resolution is the standard sweep byte for byte, and
every fixture still reaches the extraction paths it was built for, so that the GPU tests that run them cannot lose coverage silently
when the generator or the oracle drifts."""
import numpy as np
import pytest

from dense_rings import EXPECT, FIXTURES, make, ring_paths
from oracle_py import Oracle


@pytest.mark.parametrize("model,seq,frame", [(16, 0, 0), (16, 3, 5), (64, 0, 0), (64, 2, 7)])
def test_default_resolution_is_the_standard_sweep(synth, model, seq, frame):
    a, ga = synth.sweep(model, seq, frame)
    b, gb = synth.sweep(model, seq, frame, naz=1800 if model == 16 else 1875)
    assert a.tobytes() == b.tobytes() and ga.tobytes() == gb.tobytes()
    c, _ = synth.sweep(model, seq, frame, naz=0)   # 0: the model's default
    assert a.tobytes() == c.tobytes()


def test_dense_sweep_is_the_same_scene(synth):
    """Every 4th column of a 4x denser sweep is not the standard sweep (the start azimuth moves by half a step), but both see the
    same street: ground returns at the same height and nearly the same number of points per column."""
    a, ga = synth.sweep(16, 0, 3)
    b, gb = synth.sweep(16, 0, 3, naz=7200)
    assert np.array_equal(ga, gb)
    assert 3.9 < len(b) / len(a) < 4.1
    assert abs(np.median(a[a[:, 2] < -1.5, 2]) - np.median(b[b[:, 2] < -1.5, 2])) < 0.02


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_fixture_reaches_its_extraction_paths(synth, name):
    pts, model, cfg = make(synth, name)
    assert len(pts) < 400_000   # the reference's scanRegistration arrays hold 400 000 points
    ref = Oracle(cfg["n_scans"], cfg["minimum_range"], cfg["line_res"], cfg["plane_res"]).extract(pts)
    rings = ring_paths(ref)
    reached = set().union(*(t for _, _, t in rings))
    want_all, want_ring = EXPECT[name]
    assert want_all <= reached, (name, want_all - reached, [(d, c) for d, c, _ in rings])
    for r, tags in want_ring.items():
        assert tags <= rings[r][2], (name, r, rings[r])
    # the two branches of k_sector_pick that no ring can reach (see test_gpu_dense_rings.py)
    assert "joint" not in reached and "lf_smem" not in reached


def test_boundary_rings_sit_on_the_limits(synth):
    pts, _, cfg = make(synth, "boundaries")
    rings = ring_paths(Oracle(cfg["n_scans"], cfg["minimum_range"], cfg["line_res"], cfg["plane_res"]).extract(pts))
    d = [r[0] for r in rings]
    assert d[0] == 12288 and d[1] == 12289            # six sectors of 2048 / one of 2049
    assert d[2] + 12 == 4096 and d[3] + 12 == 4097    # RL
    assert (d[4] + 5) // 6 + 1 == 512 and (d[5] + 5) // 6 + 1 == 513   # mmax
    assert rings[6][1] == 2048 and rings[7][1] == 2049                  # less-flat candidates


def test_rejects_bad_resolution(synth):
    out = np.empty((16, 4), np.float32)
    f = synth.lib.lvo_synth_sweep_res
    assert f(16, 0, 0, 0.2, -1, out.ctypes.data, 16 * 100, None) == -1
    assert f(16, 0, 0, 0.2, 100, out.ctypes.data, 16 * 100 - 1, None) == -1   # capacity below model * naz
