"""C-ABI behaviour added in round 2: lvo_step_batch_async + lvo_wait, packed x,y,z sweep records, merged uploads of lanes that are
adjacent in host memory, the sub-stage timings under the reference's TicToc names, lvo_config::debug_probes, two-GPU determinism."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
CAPS = dict(max_map_corner=1 << 18, max_map_surf=1 << 19)


def test_async_wait_xyz_records_and_slab_uploads_are_bitwise_identical(lvo_mod, synth):
    L = lvo_mod
    a = L.Lvo(lanes=3, **CAPS)                      # plain lvo_step_batch, float4 records, separate arrays
    b = L.Lvo(lanes=3, **CAPS)                      # async + wait, packed xyz records, one host slab for all lanes
    c = L.Lvo(lanes=3, debug_probes=0, **CAPS)      # pipelined entry, xyz slab, product configuration (no parity probes)
    frames = []
    for k in range(5):
        sw = [synth.sweep(64, s, k)[0] for s in (0, 1, 4)]
        n = [len(x) for x in sw]
        slab = np.zeros((sum(n) + 64, 3), np.float32)   # lanes back to back (+ a small gap before the last one)
        offs = [0, n[0], n[0] + n[1] + 17]
        for x, o in zip(sw, offs):
            slab[o:o + len(x)] = x[:, :3]
        frames.append((sw, [slab[o:o + m] for o, m in zip(offs, n)], slab))
    for k, (sw, xyz, slab) in enumerate(frames):
        sa, oa, ma = a.step_batch(sw)
        b.step_batch_async(xyz)
        with pytest.raises(L.LvoError):             # one step in flight: every other entry point refuses
            b.extract_features(sw[0])
        sb, ob, mb = b.wait()
        nxt = frames[k + 1][1] if k + 1 < len(frames) else None
        sc, oc, mc = c.step_batch_pipelined(xyz, nxt)
        assert sa == sb == sc and np.array_equal(oa, ob) and np.array_equal(ma, mb) and np.array_equal(oa, oc) and np.array_equal(ma, mc), k
    assert np.array_equal(a.probe(L.P_LESS_FLAT, 2).view(np.uint32), b.probe(L.P_LESS_FLAT, 2).view(np.uint32))
    with pytest.raises(L.LvoError):                 # LVO_E_STATE: per-outer-iteration probes need debug_probes
        c.probe(L.P_MAP_SURF_KNN)
    for x in (a, b, c):
        x.close()


def test_stage_timings_under_reference_names(lvo_mod, synth):
    L = lvo_mod
    lvo = L.Lvo(lanes=1, **CAPS)
    lvo.set_option(L.LVO_OPT_GRAPHS, 0)
    for k in range(3):
        lvo.step_batch([synth.sweep(64, 0, k)[0]])
    t = lvo.stage_timings()
    for name in ("prepare time", "sort q time", "seperate points time", "data association time", "solver time", "map prepare time", "build tree time",
                 "mapping data assosiation time", "mapping solver time", "add points time", "filter time", "scan registration time", "whole laserOdometry time",
                 "whole mapping time"):
        assert t[name] > 0.0, (name, t)
    assert abs(t["prepare time"] + t["sort q time"] + t["seperate points time"] - t["scan registration time"]) < 0.2 * t["scan registration time"] + 0.05
    assert t["mapping optimization time"] <= t["whole mapping time"] * 1.05
    tm = lvo.timings()
    assert tm.knn_launches >= 1 and tm.knn_ms > 0 and tm.knn_bytes > 0
    lvo.close()


def test_two_gpus_give_bitwise_identical_poses(lvo_mod, synth):
    """SURVEY §4: the same sequence must produce bitwise identical poses on any GPU (CUDA path, not the oracle)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = lvo_mod
    a = L.Lvo(device=0, lanes=2, **CAPS)
    b = L.Lvo(device=1, lanes=2, **CAPS)
    for k in range(6):
        sw = [synth.sweep(64, 2, k)[0], synth.sweep(64, 6, k)[0]]
        _, oa, ma = a.step_batch(sw)
        _, ob, mb = b.step_batch(sw)
        assert np.array_equal(oa, ob) and np.array_equal(ma, mb), k
    for which in (0, 1):
        pa, ca = a.map_export(1, which)
        pb, cb = b.map_export(1, which)
        assert np.array_equal(ca, cb) and np.array_equal(pa.view(np.uint32), pb.view(np.uint32))
    a.close(); b.close()


def test_retired_option_value_is_rejected(lvo_mod):
    """Option 4 selected a removed 5-NN search: it is not reused and is refused like any unknown option."""
    L = lvo_mod
    lvo = L.Lvo(lanes=1, **CAPS)
    assert lvo.lib.lvo_set_option(lvo.h, 4, 1) == L.LVO_E_BADARG
    for opt in (L.LVO_OPT_GRAPHS, L.LVO_OPT_FIXPOINT_SKIP, L.LVO_OPT_STAGE_TIMING, L.LVO_OPT_KNN_REUSE, L.LVO_OPT_ODO_REUSE):
        assert lvo.lib.lvo_set_option(lvo.h, opt, 1) == L.LVO_OK, opt
    lvo.close()
