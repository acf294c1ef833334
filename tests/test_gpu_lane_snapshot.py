"""Lane snapshots: lvo_lane_save / lvo_lane_load.

A snapshot taken after frame k and loaded into any lane of any context with the same settings continues the sequence exactly as the
source lane does: "equal" below is bitwise, as in test_gpu_lanes.py (poses, statuses, lvo_stats bytes, both map exports, both map
clouds, the map correction).  Snapshots are saved after an odd number of frames (K = 5; 7 in the move test with skip_frame = 2): with
skip_frame = 2 the lane's next frame is then one of its odd frames, which does not map, so a lost skip_frame phase would show."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_lanes import CAPS, SEQ, Sweeps, lane_state, make, run_reference, same_step

pytestmark = pytest.mark.gpu
K, N = 5, 8                  # frames before the save, frames after the load
DSEQ = (2, 3, 6, 7)          # what the destination contexts run
P2 = 131072                  # destination max_points (the source contexts use the default 262144)
GRID_BUILD_LAUNCHES = 9      # k_grid_reset, _bbox, _setup, _zero, _count, the three scan kernels, _fill
PARAMS = [pytest.mark.parametrize("distortion", [0, 2]), pytest.mark.parametrize("skip_frame", [1, 2]),
          pytest.mark.parametrize("graphs", [0, 1])]


def all_params(f):
    for p in PARAMS:
        f = p(f)
    return f


@pytest.fixture(scope="module")
def sweeps(synth):
    return Sweeps(synth)


def run(lvo, sweeps, seqs, k0, n):
    """n steps of lane l running seqs[l] from its frame k0."""
    for k in range(k0, k0 + n):
        lvo.step_batch([sweeps(s, k) for s in seqs])


def load_raw(lvo, lane, data):
    a = np.ascontiguousarray(data, np.uint8)
    return lvo.lib.lvo_lane_load(lvo.h, lane, a.ctypes.data, a.nbytes)


@all_params
def test_move_to_another_context(lvo_mod, sweeps, graphs, skip_frame, distortion):
    """Lane 1 of a 3-lane context moves to lane 2 of a 4-lane context with another max_points and the other map generation parity:
    the source has run an even number of mapping steps, the destination an odd one.  The source lane keeps running as the
    uninterrupted reference."""
    L = lvo_mod
    kw = dict(skip_frame=skip_frame, distortion=distortion)
    K = 6 if skip_frame == 1 else 7          # with skip_frame 2 the lane's next frame, 7, is one of its odd frames
    D = 3 if skip_frame == 1 else 5
    mapping_steps = lambda frames: sum(1 for k in range(frames) if k % skip_frame == 0)   # every lane of a context shares its phase
    assert mapping_steps(K) % 2 == 0 and mapping_steps(D) % 2 == 1
    ref_dst = run_reference(L, graphs, DSEQ, D + N, sweeps, max_points=P2, **kw)
    src = make(L, graphs, **kw)
    run(src, sweeps, SEQ, 0, K)
    snap = src.lane_save(1)
    dst = make(L, graphs, lanes=4, max_points=P2, **kw)
    run(dst, sweeps, DSEQ, 0, D)
    dst.lane_load(2, snap)
    assert lane_state(dst, 2) == lane_state(src, 1)
    assert np.array_equal(dst.lane_save(2), snap)                       # save(load(x)) == x
    for j in range(N):
        _, so, sm = src.step_batch([sweeps(s, K + j) for s in SEQ])
        r, o, m = dst.step_batch([sweeps(DSEQ[0], D + j), sweeps(DSEQ[1], D + j), sweeps(SEQ[1], K + j), sweeps(DSEQ[3], D + j)])
        assert np.array_equal(o[2], so[1]) and np.array_equal(m[2], sm[1]), j
        assert dst.lane_status(2) == src.lane_status(1) and lane_state(dst, 2) == lane_state(src, 1), j
        for lane in (0, 1, 3):
            same_step(ref_dst[D + j], lane, dst, o, m)
    assert np.array_equal(dst.lane_save(2), src.lane_save(1))           # same sequence, same frame: same bytes
    src.close(); dst.close()


@all_params
def test_restart(lvo_mod, sweeps, graphs, skip_frame, distortion):
    """Checkpoint every lane to host bytes, destroy the context, restore into a new one.  The first step after the restore rebuilds
    the odometry grids once for all lanes; the steps after it launch what an uninterrupted context launches."""
    L = lvo_mod
    kw = dict(skip_frame=skip_frame, distortion=distortion)
    ref = make(L, graphs, **kw)
    a = make(L, graphs, **kw)
    run(ref, sweeps, SEQ, 0, K)
    run(a, sweeps, SEQ, 0, K)
    snaps = [bytes(a.lane_save(lane)) for lane in range(3)]
    assert snaps == [bytes(ref.lane_save(lane)) for lane in range(3)]   # two contexts that ran the same sequences
    a.close()
    b = make(L, graphs, **kw)
    for lane in range(3):
        b.lane_load(lane, snaps[lane])
    for j in range(N):
        rr, ro, rm = ref.step_batch([sweeps(s, K + j) for s in SEQ])
        nr = ref.timings().kernel_launches
        r, o, m = b.step_batch([sweeps(s, K + j) for s in SEQ])
        assert r == rr and np.array_equal(o, ro) and np.array_equal(m, rm), j
        for lane in range(3):
            assert lane_state(b, lane) == lane_state(ref, lane), (j, lane)
        assert b.timings().kernel_launches == nr + (GRID_BUILD_LAUNCHES if j == 0 else 0), j
    ref.close(); b.close()


@all_params
def test_rewind(lvo_mod, sweeps, graphs, skip_frame, distortion):
    """Save lane 0 after frame K, run on, load the snapshot back and replay from frame K; lanes 1 and 2 run on undisturbed."""
    L = lvo_mod
    kw = dict(skip_frame=skip_frame, distortion=distortion)
    R = 3
    ref = run_reference(L, graphs, SEQ, K + R + N, sweeps, **kw)
    x = make(L, graphs, **kw)
    run(x, sweeps, SEQ, 0, K)
    snap = x.lane_save(0)
    for k in range(K, K + R):                                             # the save changed nothing
        _, o, m = x.step_batch([sweeps(s, k) for s in SEQ])
        for lane in range(3):
            same_step(ref[k], lane, x, o, m)
    x.lane_load(0, snap)
    assert lane_state(x, 0) == ref[K - 1][3][0]
    for j in range(N):
        _, o, m = x.step_batch([sweeps(SEQ[0], K + j), sweeps(SEQ[1], K + R + j), sweeps(SEQ[2], K + R + j)])
        same_step(ref[K + j], 0, x, o, m)
        for lane in (1, 2):
            same_step(ref[K + R + j], lane, x, o, m)
    x.close()


def test_device_buffer_matches_host_bytes(lvo_mod, sweeps):
    import torch
    L = lvo_mod
    src = make(L, 0)
    run(src, sweeps, SEQ, 0, K)
    host = src.lane_save(1)
    buf = torch.full((len(host) + 64,), 0xAB, dtype=torch.uint8, device="cuda")
    n = src.lane_save_dev(1, buf.data_ptr(), buf.numel())
    assert n == len(host) and np.array_equal(buf[:n].cpu().numpy(), host)
    a, b = make(L, 0), make(L, 0)
    for x in (a, b):
        run(x, sweeps, DSEQ[:3], 0, 3)
    a.lane_load_dev(0, buf.data_ptr(), n)
    b.lane_load(0, host)
    for j in range(4):
        _, so, sm = src.step_batch([sweeps(s, K + j) for s in SEQ])
        sw = [sweeps(SEQ[1], K + j), sweeps(DSEQ[1], 3 + j), sweeps(DSEQ[2], 3 + j)]
        _, ao, am = a.step_batch(sw)
        _, bo, bm = b.step_batch(sw)
        assert np.array_equal(ao, bo) and np.array_equal(am, bm), j
        assert np.array_equal(ao[0], so[1]) and np.array_equal(am[0], sm[1]), j
        for lane in range(3):
            assert lane_state(a, lane) == lane_state(b, lane), (j, lane)
    assert np.array_equal(a.lane_save(0), src.lane_save(1))
    src.close(); a.close(); b.close()


@pytest.mark.parametrize("graphs", [0, 1])
def test_idle_lanes(lvo_mod, sweeps, graphs):
    """A lane idle at the save is saved; loaded into an idle lane it stays idle, and resumes bit for bit once activated."""
    L = lvo_mod
    ref = run_reference(L, graphs, SEQ, K - 2 + N, sweeps)
    src = make(L, graphs)
    for k in range(K):
        if k == K - 2:
            src.set_lane_active(1, False)
        src.step_batch([sweeps(SEQ[0], k), sweeps(SEQ[1], k) if k < K - 2 else None, sweeps(SEQ[2], k)])
    snap = src.lane_save(1)
    assert lane_state(src, 1) == ref[K - 3][3][1]
    dst = make(L, graphs)
    run(dst, sweeps, DSEQ[:3], 0, 3)
    dst.set_lane_active(2, False)
    dst.lane_load(2, snap)
    held = lane_state(dst, 2)
    assert held == ref[K - 3][3][1]
    for k in (3, 4):
        _, o, m = dst.step_batch([sweeps(DSEQ[0], k), sweeps(DSEQ[1], k), None])
        assert np.isnan(o[2]).all() and np.isnan(m[2]).all() and lane_state(dst, 2) == held, k
    dst.set_lane_active(2, True)
    for j in range(N):
        _, o, m = dst.step_batch([sweeps(DSEQ[0], 5 + j), sweeps(DSEQ[1], 5 + j), sweeps(SEQ[1], K - 2 + j)])
        _, ro, rm, rs = ref[K - 2 + j]                                   # reference lane 1 = lane 2 here
        assert np.array_equal(o[2], ro[1]) and np.array_equal(m[2], rm[1]) and lane_state(dst, 2) == rs[1], j
    src.close(); dst.close()


# byte offsets of the snapshot format (DESIGN.md §3); LaneState offsets as laid out by lvo_internal.h, checked against the
# values they must hold before a test edits them
H_N_SURF_LAST = 104
LS = 128
LS_N_KEPT, LS_N_SHARP, LS_N_LESS_FLAT = 16, 1056, 1068
LS_N_SURF_LAST, LS_CORNER_RING_FIRST, LS_MAP_X, LS_CEN, LS_N_VALID, LS_VALID_CUBE, LS_N_STACK = 1460, 1464, 2000, 2168, 2204, 2208, 3116
CUBE_START = LS + 4096
CAP_SHARP = 64 * 6 * 2      # sharp features per sweep for n_scans 64


def i32(a, off):
    return int(a[off:off + 4].view(np.int32)[0])


def f64(a, off):
    return float(a[off:off + 8].view(np.float64)[0])


def edited(a, off, value, dtype=np.int32):
    b = a.copy()
    v = np.array([value], dtype).view(np.uint8)
    b[off:off + len(v)] = v
    return b


def test_errors_leave_the_lane_unchanged(lvo_mod, sweeps):
    L = lvo_mod
    src = make(L, 0)
    run(src, sweeps, SEQ, 0, K)
    snap = src.lane_save(1)
    dst = make(L, 0)
    lib, h = dst.lib, dst.h
    run(dst, sweeps, DSEQ[:3], 0, 2)
    # a step in flight
    dst.step_batch_async([sweeps(s, 2) for s in DSEQ[:3]])
    n = C.c_size_t(0)
    assert lib.lvo_lane_save(h, 1, None, 0, C.byref(n)) == L.LVO_E_STATE
    assert load_raw(dst, 1, snap) == L.LVO_E_STATE
    dst.wait()
    before = lane_state(dst, 1)
    # bad lanes
    for lane in (-1, 3):
        assert lib.lvo_lane_save(h, lane, None, 0, C.byref(n)) == L.LVO_E_BADARG
        assert load_raw(dst, lane, snap) == L.LVO_E_BADARG
    # a buffer too small: the size needed
    small = np.zeros(100, np.uint8)
    for ptr, cap in ((None, 0), (small.ctypes.data, small.nbytes), (small.ctypes.data, len(snap) - 1)):
        n.value = 0
        assert src.lib.lvo_lane_save(src.h, 1, ptr, cap, C.byref(n)) == L.LVO_E_CAPACITY and n.value == len(snap)
    assert not small.any()
    # malformed snapshots
    n_surf = i32(snap, H_N_SURF_LAST)
    assert i32(snap, LS + LS_N_SURF_LAST) == n_surf > 1000
    assert 1 <= i32(snap, LS + LS_N_VALID) <= 75 and i32(snap, CUBE_START) == 0
    assert all(i32(snap, LS + LS_CORNER_RING_FIRST + 4 * r) >= 0 for r in range(66))
    st = src.stats(1)
    assert (i32(snap, LS + LS_N_KEPT), i32(snap, LS + LS_N_SHARP), i32(snap, LS + LS_N_LESS_FLAT), i32(snap, LS + LS_N_STACK + 4)) == (
        st.n_kept, st.n_sharp, st.n_less_flat, st.map_surf_stack)
    assert abs(sum(f64(snap, LS + LS_MAP_X + 8 * k) ** 2 for k in range(4)) - 1) < 1e-9     # map_x: a unit quaternion, then t
    bad_magic = snap.copy()
    bad_magic[0] ^= 0xFF
    cases = {"truncated": snap[:-16], "short": snap[:100], "trailing": np.concatenate([snap, np.zeros(16, np.uint8)]), "magic": bad_magic,
             "n_surf_last": edited(snap, LS + LS_N_SURF_LAST, n_surf + 1),
             "n_surf_last both": edited(edited(snap, LS + LS_N_SURF_LAST, 1 << 30), H_N_SURF_LAST, 1 << 30),
             "n_valid": edited(snap, LS + LS_N_VALID, 76), "valid_cube": edited(snap, LS + LS_VALID_CUBE, 4851),
             "ring_first": edited(snap, LS + LS_CORNER_RING_FIRST + 8, -1), "cen": edited(snap, LS + LS_CEN, 1 << 30),
             "cube_start": edited(snap, CUBE_START + 4 * 100, 0x7FFFFFFF), "cube_start first": edited(snap, CUBE_START, 5),
             # the counts of the last frame, which the stand-alone stage calls read for every lane
             "n_kept < 0": edited(snap, LS + LS_N_KEPT, -1), "n_sharp < 0": edited(snap, LS + LS_N_SHARP, -5),
             "n_sharp > cap": edited(snap, LS + LS_N_SHARP, CAP_SHARP + 1), "n_less_flat < 0": edited(snap, LS + LS_N_LESS_FLAT, -1),
             "n_stack < 0": edited(snap, LS + LS_N_STACK + 4, -1),
             # poses
             "map_x t huge": edited(snap, LS + LS_MAP_X + 32, 1e300, np.float64), "map_x t nan": edited(snap, LS + LS_MAP_X + 40, np.nan, np.float64),
             "map_x q huge": edited(snap, LS + LS_MAP_X, 3.0, np.float64)}
    for name, data in cases.items():
        assert load_raw(dst, 1, data) == L.LVO_E_BADARG, name
        assert lane_state(dst, 1) == before, name
    # counts of the last frame above what this context's max_points holds
    for name, off in (("n_kept", LS_N_KEPT), ("n_less_flat", LS_N_LESS_FLAT), ("n_stack[1]", LS_N_STACK + 4)):
        for value in (dst.P + 1, 1 << 30):
            assert load_raw(dst, 1, edited(snap, LS + off, value)) == L.LVO_E_CAPACITY, (name, value)
            assert name in lib.lvo_last_error(h).decode() and lane_state(dst, 1) == before, (name, value)
    # settings that change results: one mismatch at a time
    small_caps = dict(lanes=2, max_points=1 << 15, max_map_corner=1 << 12, max_map_surf=1 << 12, debug_probes=0)
    for field, value in (("n_scans", 32), ("minimum_range", 4.0), ("line_res", 0.3), ("plane_res", 0.6), ("skip_frame", 2),
                         ("outer_iters", 8), ("lm_max_iters", 3), ("huber", 0.2), ("distortion", 1)):
        y = L.Lvo(**{**small_caps, field: value})
        yb = lane_state(y, 1)
        assert load_raw(y, 1, snap) == L.LVO_E_BADARG, field
        assert field in y.lib.lvo_last_error(y.h).decode(), field
        assert lane_state(y, 1) == yb, field
        y.close()
    # capacities too small for what was saved
    assert len(src.map_export(1, 1)[0]) > 1024
    for caps in (dict(CAPS, max_map_surf=1024), dict(CAPS, max_points=1000)):
        y = L.Lvo(lanes=2, **caps)
        yb = lane_state(y, 1)
        assert load_raw(y, 1, snap) == L.LVO_E_CAPACITY, caps
        assert lane_state(y, 1) == yb, caps
        y.close()
    # probes of a freshly loaded lane: none until it has run a frame, then those of the source lane
    dst.lane_load(1, snap)
    for what in (L.P_LESS_FLAT, L.P_MAP_SURF_STACK, L.P_MAP_SURF_KNN):
        assert lib.lvo_probe_fetch(h, 1, what, None, 0, C.byref(n)) == L.LVO_E_STATE, what
    src.step_batch([sweeps(s, K) for s in SEQ])
    dst.step_batch([sweeps(DSEQ[0], 3), sweeps(SEQ[1], K), sweeps(DSEQ[2], 3)])
    # the clouds a frame writes in full.  Not the per-iteration records: e.g. the LM trace rows of LM iterations an outer iteration
    # did not reach keep what earlier frames of the lane wrote there, and a snapshot does not carry probes.
    for what in (L.P_LESS_FLAT, L.P_REGISTERED, L.P_MAP_SURF_STACK, L.P_MAP_SURF_FROM_MAP):
        assert dst.probe(what, 1).tobytes() == src.probe(what, 1).tobytes(), what
    src.close(); dst.close()


@pytest.mark.parametrize("distortion", [0, 2])
def test_standalone_entry_points_after_a_load(lvo_mod, sweeps, distortion):
    """A loaded lane 0 driven by lvo_extract_features / lvo_scan_to_scan / lvo_scan_to_map computes what the source lane computes.
    Its probes come back one stage at a time, as each stage runs."""
    L = lvo_mod
    src = make(L, 0, distortion=distortion)
    run(src, sweeps, SEQ, 0, K)
    y = make(L, 0, distortion=distortion)
    run(y, sweeps, DSEQ[:3], 0, 3)
    y.lane_load(0, src.lane_save(0))
    n = C.c_size_t(0)
    state = lambda what: y.lib.lvo_probe_fetch(y.h, 0, what, None, 0, C.byref(n))
    gated = lambda: [state(w) == L.LVO_E_STATE for w in (L.P_LESS_FLAT, L.P_ODO_LM_TRACE, L.P_MAP_SURF_STACK, L.P_REGISTERED)]
    assert gated() == [True] * 4
    for k in range(K, K + 3):
        rs, fs = src.extract_features(sweeps(SEQ[0], k))
        ry, fy = y.extract_features(sweeps(SEQ[0], k))
        assert rs == ry and all(fs[x].tobytes() == fy[x].tobytes() for x in fs), k
        if k == K:
            assert gated() == [False, True, True, True]
        feats = [fs[x] for x in ("sharp", "less_sharp", "flat", "less_flat")]
        os_, os1, os2 = src.scan_to_scan(*feats)
        oy, oy1, oy2 = y.scan_to_scan(*feats)
        assert os_ == oy and os1.tobytes() == oy1.tobytes() and os2.tobytes() == oy2.tobytes(), k
        if k == K:
            assert gated() == [False, False, True, True]
        ms, ps, gs = src.scan_to_map(fs["less_sharp"], fs["less_flat"], fs["full"], os2, want_registered=True)
        my, py, gy = y.scan_to_map(fs["less_sharp"], fs["less_flat"], fs["full"], oy2, want_registered=True)
        assert ms == my and ps.tobytes() == py.tobytes() and gs.tobytes() == gy.tobytes(), k
        assert gated() == [False] * 4
        assert lane_state(y, 0) == lane_state(src, 0), k
        assert y.probe(L.P_MAP_SURF_STACK, 0).tobytes() == src.probe(L.P_MAP_SURF_STACK, 0).tobytes(), k
    src.close(); y.close()


def test_move_to_another_gpu(lvo_mod, sweeps):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = lvo_mod
    src = make(L, 0)
    run(src, sweeps, SEQ, 0, K)
    buf = torch.empty(len(src.lane_save(1)), dtype=torch.uint8, device="cuda:0")
    n = src.lane_save_dev(1, buf.data_ptr(), buf.numel())
    dst = L.Lvo(device=1, lanes=3, **CAPS)
    dst.set_option(L.LVO_OPT_GRAPHS, 0)
    run(dst, sweeps, DSEQ[:3], 0, 3)
    dst.lane_load_dev(1, buf.data_ptr(), n)                              # a device-0 buffer
    assert lane_state(dst, 1) == lane_state(src, 1)
    for j in range(N):
        _, so, sm = src.step_batch([sweeps(s, K + j) for s in SEQ])
        _, o, m = dst.step_batch([sweeps(DSEQ[0], 3 + j), sweeps(SEQ[1], K + j), sweeps(DSEQ[2], 3 + j)])
        assert np.array_equal(o[1], so[1]) and np.array_equal(m[1], sm[1]), j
        assert lane_state(dst, 1) == lane_state(src, 1), j
    src.close(); dst.close()
