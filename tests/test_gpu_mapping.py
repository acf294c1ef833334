"""GPU parity: lvo_scan_to_map vs the oracle's laserMapping restatement (reference src/laserMapping.cpp:307-848)."""
import numpy as np
import pytest

from oracle_py import Oracle

pytestmark = pytest.mark.gpu
POS_TOL, ROT_TOL = 1e-4, 1e-5


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def rot_err(qa, qb):
    return 2 * np.arccos(min(1.0, abs(float(np.dot(qa, qb)))))


def _frames(synth, O, model, seq, n):
    """Run the oracle pipeline; yield per-frame inputs of the mapping stage."""
    out = []
    for k in range(n):
        pts, _ = synth.sweep(model, seq, k)
        f = O.extract(pts)
        _, _, w = O.odometry(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"], keep_log=False)
        out.append((f, w))
    return out


@pytest.mark.parametrize("model,cfg,seq", [(64, (64, 5.0, 0.4, 0.8), 0), (16, (16, 0.3, 0.2, 0.4), 1)])
def test_scan_to_map_from_imported_state(lvo_mod, synth, model, cfg, seq):
    L = lvo_mod
    O = Oracle(*cfg)
    lvo = L.Lvo(n_scans=cfg[0], minimum_range=cfg[1], line_res=cfg[2], plane_res=cfg[3], max_map_corner=1 << 18, max_map_surf=1 << 19)
    frames = _frames(synth, O, model, seq, 7)
    flips = rows = 0
    corr_prev = np.array([0, 0, 0, 1, 0, 0, 0], float)
    for k, (f, w) in enumerate(frames):
        # identical starting state on both sides: the oracle's map and map correction
        pc, cc = O.map_export(0)
        ps, cs = O.map_export(1)
        lvo.map_import(0, pc, cc, ps, cs)
        lvo.set_map_correction(0, corr_prev)
        st_o, pose_o, corr_o = O.mapping(f["less_sharp"], f["less_flat"], f["full"], w)
        st_g, pose_g, reg_g = lvo.scan_to_map(f["less_sharp"], f["less_flat"], f["full"], w, want_registered=True)
        assert st_g == st_o, (k, st_g, st_o)
        info = O.mapping_info()
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_CORNER_STACK)), _bits(info["corner_stack"])), f"frame {k}: corner stack (VoxelGrid lineRes)"
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_SURF_STACK)), _bits(info["surf_stack"])), f"frame {k}: surf stack (VoxelGrid planeRes)"
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_CORNER_FROM_MAP)), _bits(info["corner_from_map"])), f"frame {k}: corner FromMap order"
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_SURF_FROM_MAP)), _bits(info["surf_from_map"])), f"frame {k}: surf FromMap order"
        s = lvo.stats()
        assert list(s.center_cube) == list(info["info"][:3]) and list(s.cen) == list(info["info"][3:6])
        if st_o == 0:
            kc, ks = lvo.probe(L.P_MAP_CORNER_KNN), lvo.probe(L.P_MAP_SURF_KNN)
            vc, vs = lvo.probe(L.P_MAP_CORNER_VALID), lvo.probe(L.P_MAP_SURF_VALID)
            tr = lvo.probe(L.P_MAP_LM_TRACE)
            for o in range(O.outer):
                lg = O.mapping_log(o)
                f1 = (kc[o] != lg["corner_knn"]).any(axis=1).sum() + (ks[o] != lg["surf_knn"]).any(axis=1).sum()
                f2 = (vc[o] != lg["corner_valid"]).sum() + (vs[o] != lg["surf_valid"]).sum()
                if o == 0:  # identical pose -> identical queries: kNN index sets and accept flags must be bit-exact
                    assert f1 == 0, f"frame {k} outer 0: {f1} kNN rows differ"
                    assert f2 == 0, f"frame {k} outer 0: {f2} factor accept flags differ"
                flips += f1 + f2
                rows += 2 * (len(kc[o]) + len(ks[o]))
                if f1 == 0 and f2 == 0:
                    n = len(lg["lm"])
                    assert np.array_equal(tr[o][:n, 9], lg["lm"][:, 9]), f"frame {k} outer {o}: LM control flow {tr[o][:n, 9]} vs {lg['lm'][:, 9]}"
                    assert np.allclose(tr[o][:n, :7], lg["lm"][:, :7], atol=1e-7, rtol=0)
                    assert np.allclose(tr[o][:n, 7], lg["lm"][:, 7], rtol=1e-7, atol=1e-12)
        assert np.linalg.norm(pose_g[4:] - pose_o[4:]) < POS_TOL and rot_err(pose_g[:4], pose_o[:4]) < ROT_TOL, (k, pose_g, pose_o)
        corr_g = lvo.get_map_correction(0)
        corr_prev = corr_o
        assert np.linalg.norm(corr_g[4:] - corr_o[4:]) < POS_TOL and rot_err(corr_g[:4], corr_o[:4]) < ROT_TOL
        # map after insertion + per-cube re-filter: same cube occupancy; coordinates equal up to the pose difference
        for which in (0, 1):
            pg, cg = lvo.map_export(0, which)
            po, co = O.map_export(which)
            assert len(pg) == len(po) or abs(len(pg) - len(po)) <= 3, (k, which, len(pg), len(po))
            if len(pg) == len(po):
                assert np.array_equal(cg, co)
                assert np.abs(pg[:, :3] - po[:, :3]).max() < 1e-3
        assert (s.map_corner_total, s.map_surf_total) == (len(lvo.map_export(0, 0)[0]), len(lvo.map_export(0, 1)[0]))
        reg_o = info["registered"]
        assert reg_g.shape == reg_o.shape and np.abs(reg_g - reg_o).max() < 1e-3
    from conftest import record_metric
    record_metric(f"mapping_knn_and_accept_rows_differing_from_oracle/model{model}_seq{seq}", {"differ": int(flips), "rows": int(rows), "frames": len(frames)})
    # both sides are deterministic on fixed inputs: a B200 run records 0 differing rows on both sequences of this test
    print(f"mapping model {model} seq {seq}: {flips} of {rows} kNN / accept rows differ")
    assert flips == 0, f"{flips} of {rows} kNN / accept rows differ"
    lvo.close()


def test_full_pipeline_batch_two_lanes(lvo_mod, synth):
    """lvo_step_batch (extract -> scan-to-scan -> scan-to-map on device, 2 lanes) vs two oracle pipelines."""
    L = lvo_mod
    lvo = L.Lvo(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    Os = [Oracle(), Oracle()]
    seqs = [0, 3]
    for k in range(8):
        sweeps = [synth.sweep(64, s, k)[0] for s in seqs]
        st, odo_g, map_g = lvo.step_batch(sweeps)
        for l in range(2):
            st_o, odo_o, map_o = Os[l].step(sweeps[l])
            assert np.linalg.norm(odo_g[l][4:] - odo_o[4:]) < POS_TOL and rot_err(odo_g[l][:4], odo_o[:4]) < ROT_TOL, (k, l, odo_g[l], odo_o)
            assert np.linalg.norm(map_g[l][4:] - map_o[4:]) < POS_TOL and rot_err(map_g[l][:4], map_o[:4]) < ROT_TOL, (k, l, map_g[l], map_o)
            s = lvo.stats(l)
            info = Os[l].mapping_info()["info"]
            assert abs(s.map_corner_total - info[6]) <= 5 and abs(s.map_surf_total - info[7]) <= 5
    lvo.close()


def test_lanes_are_bitwise_reproducible(lvo_mod, synth):
    """The same sequence in two lanes (and in a 1-lane context) gives bitwise identical poses: deterministic reductions."""
    L = lvo_mod
    a = L.Lvo(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    b = L.Lvo(lanes=1, max_map_corner=1 << 18, max_map_surf=1 << 19)
    for k in range(5):
        sw = synth.sweep(64, 2, k)[0]
        _, oa, ma = a.step_batch([sw, sw])
        _, ob, mb = b.step_batch([sw])
        assert np.array_equal(oa[0], oa[1]) and np.array_equal(ma[0], ma[1])
        assert np.array_equal(oa[0], ob[0]) and np.array_equal(ma[0], mb[0])
    a.close(); b.close()


def test_map_too_small_warning(lvo_mod, synth):
    L = lvo_mod
    lvo = L.Lvo(max_map_corner=1 << 18, max_map_surf=1 << 19)
    O = Oracle()
    f = O.extract(synth.sweep(64, 0, 0)[0])
    ident = np.array([0, 0, 0, 1, 0, 0, 0], float)
    st_o, pose_o, _ = O.mapping(f["less_sharp"], f["less_flat"], None, ident)
    st_g, pose_g, _ = lvo.scan_to_map(f["less_sharp"], f["less_flat"], None, ident)
    assert st_o == 3 and st_g == L.LVO_W_MAP_TOO_SMALL and np.array_equal(pose_g, pose_o)
    for which in (0, 1):  # the map is still updated (laserMapping.cpp:737-801)
        pg, cg = lvo.map_export(0, which)
        po, co = O.map_export(which)
        assert np.array_equal(cg, co) and np.array_equal(_bits(pg), _bits(po))
    lvo.close()


def test_pipelined_host_entry_matches_plain(lvo_mod, synth):
    """lvo_step_batch_pipelined (next frame uploaded on a copy stream during compute) gives bit-identical poses."""
    L = lvo_mod
    a = L.Lvo(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    b = L.Lvo(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    frames = [[np.ascontiguousarray(synth.sweep(64, s, k)[0]) for s in (0, 1)] for k in range(5)]
    for k in range(5):
        _, oa, ma = a.step_batch(frames[k])
        nxt = frames[k + 1] if (k + 1 < 5 and k != 2) else None   # k == 2: no prefetch -> next call takes the fallback copy path
        _, ob, mb = b.step_batch_pipelined(frames[k], nxt)
        assert np.array_equal(oa, ob) and np.array_equal(ma, mb), k
    a.close(); b.close()


def test_cube_window_shifts_match_oracle(lvo_mod, synth):
    """Drive the 21x21x11 cube window across its edges on every axis (laserMapping.cpp:312-507): centre-cube indices,
    laserCloudCen*, which cubes are recycled, and the surviving map must match the oracle exactly.  The poses jump by tens of
    metres, so most frames see an (almost) empty neighbourhood and skip the optimisation — the map bookkeeping is what is tested."""
    L = lvo_mod
    O = Oracle()
    lvo = L.Lvo(max_map_corner=1 << 18, max_map_surf=1 << 19)
    f = O.extract(synth.sweep(64, 0, 0)[0])
    path = [(0, 0, 0), (120, 0, 0), (260, 0, 0), (390, 0, 0), (520, 30, 0), (390, 0, 0), (0, 0, 0), (-180, 0, 0), (-390, -40, 0), (-520, 0, 0),
            (0, 200, 0), (0, 395, 0), (0, 520, 60), (0, 520, 130), (0, 520, 210), (0, 0, 0), (0, -400, -130), (0, -560, -260), (300, 300, 100)]
    shifted = 0
    prev_cen = [10, 10, 5]
    exact = True   # until an optimised frame inserts points with a pose that agrees to ~1e-13 m rather than to the last bit
    for k, t in enumerate(path):
        odom = np.array([0, 0, 0, 1, t[0], t[1], t[2]], float)
        st_o, pose_o, corr_o = O.mapping(f["less_sharp"], f["less_flat"], None, odom)
        st_g, pose_g, _ = lvo.scan_to_map(f["less_sharp"], f["less_flat"], None, odom)
        info = O.mapping_info()["info"]
        s = lvo.stats()
        assert st_g == st_o, (k, st_g, st_o)
        assert list(s.center_cube) == list(info[:3]) and list(s.cen) == list(info[3:6]), (k, list(s.center_cube), list(s.cen), list(info[:6]))
        if list(s.cen) != prev_cen:
            shifted += 1
        prev_cen = list(s.cen)
        assert np.linalg.norm(pose_g[4:] - pose_o[4:]) < 1e-4, (k, pose_g, pose_o)
        lvo.set_map_correction(0, corr_o)   # keep both sides on the same correction so that inserted points stay bit-identical
        for which in (0, 1):
            pg, cg = lvo.map_export(0, which)
            po, co = O.map_export(which)
            assert len(pg) == len(po) and np.array_equal(cg, co), (k, which, len(pg), len(po))
            if st_o != 3:
                exact = False
            if exact:       # no optimisation ran so far: identical poses -> identical floats
                assert np.array_equal(_bits(pg), _bits(po)), (k, which)
            else:           # same points in the same cubes and order; float noise in at most a handful of coordinates
                assert np.abs(pg[:, :3] - po[:, :3]).max() < 1e-3
                assert (_bits(pg) != _bits(po)).mean() < 1e-3, (k, which)
        assert (s.map_corner_total, s.map_surf_total) == (info[6], info[7])
    assert shifted >= 8   # the window really moved, in both directions on all three axes
    lvo.close()


def test_graph_replay_matches_plain_launches(lvo_mod, synth):
    """The CUDA-graph replay of the fused frame (default for few lanes) and plain launches give bit-identical poses, also with
    mapping_skip_frame = 2 (two graph variants) and when the point layout changes (graphs are re-captured)."""
    L = lvo_mod
    for skip in (1, 2):
        a = L.Lvo(lanes=1, skip_frame=skip, max_map_corner=1 << 18, max_map_surf=1 << 19)
        b = L.Lvo(lanes=1, skip_frame=skip, max_map_corner=1 << 18, max_map_surf=1 << 19)
        a.set_option(L.LVO_OPT_GRAPHS, 1)
        b.set_option(L.LVO_OPT_GRAPHS, 0)
        for k in range(7):
            sw = synth.sweep(64, 1, k)[0]
            arg = L.to_pcl_layout(sw) if k >= 5 else sw    # stride 32 from frame 5 on
            _, oa, ma = a.step_batch([arg])
            _, ob, mb = b.step_batch([arg])
            assert np.array_equal(oa, ob) and np.array_equal(ma, mb), (skip, k)
        assert a.timings().kernel_launches == b.timings().kernel_launches
        a.close(); b.close()


def test_fixpoint_skip_is_bitwise_identical(lvo_mod, synth):
    """LVO_OPT_FIXPOINT_SKIP (default on): once an outer iteration returns the pose bit for bit unchanged, the remaining outer
    iterations (laserOdometry.cpp:364, laserMapping.cpp:562) are exact repeats and are not run.  Poses, statuses, every
    per-iteration counter, the correspondence / kNN probes of ALL ten iterations and the maps must equal the full schedule's."""
    L = lvo_mod
    mk = dict(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    a, b = L.Lvo(**mk), L.Lvo(**mk)
    for c, v in ((a, 1), (b, 0)):
        c.set_option(L.LVO_OPT_GRAPHS, 0)
        c.set_option(L.LVO_OPT_FIXPOINT_SKIP, v)
    arrays = ("odo_corner_corr", "odo_plane_corr", "odo_lm_iters", "odo_final_cost", "map_corner_corr", "map_surf_corr", "map_lm_iters", "map_final_cost")
    probes = (L.P_ODO_CORNER_CORR, L.P_ODO_PLANE_CORR, L.P_MAP_CORNER_KNN, L.P_MAP_SURF_KNN, L.P_MAP_CORNER_VALID, L.P_MAP_SURF_VALID)
    cut = 0
    for k in range(8):
        sws = [synth.sweep(64, 0, k)[0], synth.sweep(64, 3, k)[0]]
        sa, oa, ma = a.step_batch(sws)
        sb, ob, mb = b.step_batch(sws)
        assert sa == sb and np.array_equal(oa, ob) and np.array_equal(ma, mb), k
        for lane in range(2):
            x, y = a.stats(lane), b.stats(lane)
            assert a.lane_status(lane) == b.lane_status(lane)
            assert y.odo_outer_executed == (10 if k else 0)
            assert y.map_outer_executed in (0, 10) and 0 <= x.map_outer_executed <= 10 and (x.odo_outer_executed >= 1) == (k > 0)
            for name in arrays:
                assert list(getattr(x, name)) == list(getattr(y, name)), (k, lane, name)
            for what in probes:
                assert np.array_equal(a.probe(what, lane), b.probe(what, lane)), (k, lane, what)
            cut += (y.odo_outer_executed - x.odo_outer_executed) + (y.map_outer_executed - x.map_outer_executed)
    assert cut > 20   # the shortcut really fired (typically after 3-6 of the 10 iterations)
    for lane in range(2):
        for which in (0, 1):
            pa, ca = a.map_export(lane, which)
            pb, cb = b.map_export(lane, which)
            assert np.array_equal(ca, cb) and np.array_equal(_bits(pa), _bits(pb))
    # the option also holds under graph replay (the flag is a kernel argument: graphs are re-captured when it changes)
    a.set_option(L.LVO_OPT_GRAPHS, 1)
    b.set_option(L.LVO_OPT_GRAPHS, 1)
    for k in range(8, 11):
        sws = [synth.sweep(64, 0, k)[0], synth.sweep(64, 3, k)[0]]
        _, oa, ma = a.step_batch(sws)
        _, ob, mb = b.step_batch(sws)
        assert np.array_equal(oa, ob) and np.array_equal(ma, mb), k
    assert a.stats(0).odo_outer_executed < 10 and b.stats(0).odo_outer_executed == 10
    a.close(); b.close()


def test_map_capacity_overflow_keeps_lanes_safe(lvo_mod, synth):
    """A lane whose map outgrows max_map_* reports LVO_E_CAPACITY, loses the tail of its map consistently (offset table, n_map and
    the stored points agree) and keeps stepping; its neighbour lane is untouched (bitwise equal to a context of its own)."""
    import ctypes as C
    L = lvo_mod
    caps = dict(max_map_corner=3000, max_map_surf=6000)
    a = L.Lvo(lanes=2, **caps)
    b = L.Lvo(lanes=1, **caps)
    overflowed = 0
    for k in range(8):
        big = synth.sweep(64, 0, k)[0]
        small = np.ascontiguousarray(synth.sweep(64, 1, 0)[0][::24])     # sparse sweep of a sensor at rest: its map stays far below the caps
        views = [L.view_of(big), L.view_of(small)]
        arr = (L.CloudView * 2)(*[v[0] for v in views])
        po, pm = (L.Pose * 2)(), (L.Pose * 2)()
        r = a.lib.lvo_step_batch(a.h, arr, po, pm)
        assert r in (L.LVO_OK, L.LVO_W_FIRST_FRAME, L.LVO_W_FEW_CORR, L.LVO_W_MAP_TOO_SMALL, L.LVO_E_CAPACITY), (k, r, a.lib.lvo_last_error(a.h))
        overflowed += r == L.LVO_E_CAPACITY
        s0, s1 = a.stats(0), a.stats(1)
        assert 0 <= s0.map_corner_total <= caps["max_map_corner"] and 0 <= s0.map_surf_total <= caps["max_map_surf"]
        assert s0.map_corner_from_map <= caps["max_map_corner"] and s0.map_surf_from_map <= caps["max_map_surf"]
        for which in (0, 1):
            pts, cube = a.map_export(0, which)
            assert len(pts) == (s0.map_corner_total, s0.map_surf_total)[which] and np.isfinite(pts).all()
            assert (np.diff(cube) >= 0).all()
        assert a.lane_status(1) >= 0, (k, a.lane_status(1))
        _, ob, mb = b.step_batch([small])
        assert np.array_equal(L.pose_to_np(po[1]), ob[0]) and np.array_equal(L.pose_to_np(pm[1]), mb[0]), k
        assert (s1.map_corner_total, s1.map_surf_total) == (b.stats(0).map_corner_total, b.stats(0).map_surf_total)
    assert overflowed >= 1
    a.close(); b.close()


def test_knn_reuse_is_bitwise_identical(lvo_mod, synth):
    """LVO_OPT_KNN_REUSE (default on): a query of lvo_scan_to_map keeps its neighbour set across the outer iterations
    (laserMapping.cpp:562, :582 / :648) when a guard radius recorded by its last full search certifies that no other map point
    can enter it, and keeps its fit when the row is unchanged.  Every 5-NN row and factor flag of ALL ten iterations, the counters,
    poses and maps must equal those of searching and fitting every query every time."""
    L = lvo_mod
    mk = dict(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    a, b = L.Lvo(**mk), L.Lvo(**mk)
    for c, v in ((a, 1), (b, 0)):
        c.set_option(L.LVO_OPT_GRAPHS, 0)
        c.set_option(L.LVO_OPT_KNN_REUSE, v)
        c.set_option(L.LVO_OPT_FIXPOINT_SKIP, 0)   # every one of the ten iterations runs, so the certificate is exercised ten times
    arrays = ("map_corner_corr", "map_surf_corr", "map_lm_iters", "map_final_cost")
    probes = (L.P_MAP_CORNER_KNN, L.P_MAP_SURF_KNN, L.P_MAP_CORNER_VALID, L.P_MAP_SURF_VALID, L.P_MAP_LM_TRACE)
    full = reused = 0
    for k in range(12):
        sws = [synth.sweep(64, 0, k)[0], synth.sweep(64, 5, k)[0]]
        sa, oa, ma = a.step_batch(sws)
        sb, ob, mb = b.step_batch(sws)
        assert sa == sb and np.array_equal(oa, ob) and np.array_equal(ma, mb), k
        for lane in range(2):
            x, y = a.stats(lane), b.stats(lane)
            for name in arrays:
                assert list(getattr(x, name)) == list(getattr(y, name)), (k, lane, name)
            for what in probes:
                assert np.array_equal(a.probe(what, lane), b.probe(what, lane)), (k, lane, what)
            if x.map_outer_executed:
                q = x.map_corner_stack + x.map_surf_stack
                assert x.map_knn_full[0] == q and list(y.map_knn_full) == [0] * 16
                full += sum(x.map_knn_full[1:10]); reused += 9 * q - sum(x.map_knn_full[1:10])
    assert reused > 4 * full, (reused, full)   # the certificate carries most rows (typically > 90 %)
    for lane in range(2):
        for which in (0, 1):
            pa, ca = a.map_export(lane, which)
            pb, cb = b.map_export(lane, which)
            assert np.array_equal(ca, cb) and np.array_equal(_bits(pa), _bits(pb))
    a.close(); b.close()
