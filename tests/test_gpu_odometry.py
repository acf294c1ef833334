"""GPU parity: lvo_scan_to_scan vs the oracle's laserOdometry restatement (reference src/laserOdometry.cpp:353-641).
Correspondence triples bit-exact on identical poses; LM trajectory and per-frame poses within 1e-4 m / 1e-5 rad."""
import numpy as np
import pytest

from oracle_py import Oracle

pytestmark = pytest.mark.gpu

POS_TOL = 1e-4   # m   (north_star)
ROT_TOL = 1e-5   # rad (north_star)


def rot_err(qa, qb):
    d = abs(float(np.dot(qa, qb)))
    return 2 * np.arccos(min(1.0, d))


def _run(lvo_mod, synth, model, cfg, nframes, seq, distortion=0):
    L = lvo_mod
    O = Oracle(*cfg, distortion=distortion)
    lvo = L.Lvo(n_scans=cfg[0], minimum_range=cfg[1], line_res=cfg[2], plane_res=cfg[3], distortion=distortion)
    flips_total = rows_total = 0
    for k in range(nframes):
        pts, _ = synth.sweep(model, seq, k, moving=distortion != 0)
        f = O.extract(pts)
        st_o, rel_o, w_o = O.odometry(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
        st_g, rel_g, w_g = lvo.scan_to_scan(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
        assert st_g == st_o, (k, st_g, st_o)
        if k == 0:
            assert st_g == L.LVO_W_FIRST_FRAME
            continue
        cc, pc, tr = lvo.probe(L.P_ODO_CORNER_CORR), lvo.probe(L.P_ODO_PLANE_CORR), lvo.probe(L.P_ODO_LM_TRACE)
        s = lvo.stats()
        for o in range(O.outer):
            lg = O.odometry_log(o)
            fc = (cc[o] != lg["corner_corr"]).any(axis=1).sum()
            fp = (pc[o] != lg["plane_corr"]).any(axis=1).sum()
            if o == 0 and k == 1:
                # identical initial pose (identity): associations must be bit-exact
                assert fc == 0 and fp == 0, f"frame {k} outer 0: {fc} corner / {fp} plane correspondence rows differ"
            flips_total += fc + fp
            rows_total += len(cc[o]) + len(pc[o])
            if fc == 0 and fp == 0:
                assert s.odo_corner_corr[o] == lg["counts"][0] and s.odo_plane_corr[o] == lg["counts"][1]
            # LM trace: same number of rows, same accept / reject / termination flags, state within 1e-7
            rows = len(lg["lm"])
            if fc == 0 and fp == 0:
                assert np.array_equal(tr[o][:rows, 9], lg["lm"][:, 9]), f"frame {k} outer {o}: LM control flow differs {tr[o][:rows, 9]} vs {lg['lm'][:, 9]}"
                assert np.allclose(tr[o][:rows, :7], lg["lm"][:, :7], atol=1e-7, rtol=0)
                assert np.allclose(tr[o][:rows, 7], lg["lm"][:, 7], rtol=1e-7, atol=1e-12)
        assert np.linalg.norm(rel_g[4:] - rel_o[4:]) < POS_TOL and rot_err(rel_g[:4], rel_o[:4]) < ROT_TOL, (k, rel_g, rel_o)
        assert np.linalg.norm(w_g[4:] - w_o[4:]) < POS_TOL and rot_err(w_g[:4], w_o[:4]) < ROT_TOL, (k, w_g, w_o)
    from conftest import record_metric
    record_metric(f"odometry_rows_differing_from_oracle/model{model}_seq{seq}_distortion{distortion}", {"differ": int(flips_total), "rows": int(rows_total), "frames": nframes})
    # both sides are deterministic on fixed inputs: a B200 run records 0 differing rows on every sequence of this test
    print(f"odometry model {model} seq {seq} distortion {distortion}: {flips_total} of {rows_total} correspondence rows differ")
    assert flips_total == 0, f"{flips_total} of {rows_total} correspondence rows differ"
    lvo.close()


def test_hdl64_scan_to_scan(lvo_mod, synth):
    _run(lvo_mod, synth, 64, (64, 5.0, 0.4, 0.8), 6, 0)


def test_vlp16_scan_to_scan(lvo_mod, synth):
    _run(lvo_mod, synth, 16, (16, 0.3, 0.2, 0.4), 6, 1)


@pytest.mark.parametrize("model,cfg,seq", [(64, (64, 5.0, 0.4, 0.8), 3), (16, (16, 0.3, 0.2, 0.4), 2)])
def test_scan_to_scan_distortion_1(lvo_mod, synth, model, cfg, seq):
    """DISTORTION 1 (laserOdometry.cpp:67): per-point interpolation ratio in TransformToStart (:157-163) and in the factors
    (:455-459, :549-553; lidarFactor.hpp:27-30, 79-82), on sweeps cast from a moving sensor."""
    _run(lvo_mod, synth, model, cfg, 6, seq, distortion=1)


def test_few_correspondences_warning(lvo_mod, synth):
    """Second frame far away from the first: no correspondences -> LVO_W_FEW_CORR (laserOdometry.cpp:566-568), pose unchanged."""
    L = lvo_mod
    O = Oracle()
    lvo = L.Lvo()
    pts, _ = synth.sweep(64, 0, 0)
    f = O.extract(pts)
    lvo.scan_to_scan(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
    O.odometry(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
    shift = np.array([500, 500, 0, 0], np.float32)
    args = [f[k] + shift for k in ("sharp", "less_sharp", "flat", "less_flat")]
    st_o, rel_o, _ = O.odometry(*args)
    st_g, rel_g, _ = lvo.scan_to_scan(*args)
    assert st_o == 2 and st_g == L.LVO_W_FEW_CORR
    assert np.array_equal(rel_g, rel_o)
    lvo.close()


def test_odo_reuse_is_bitwise_identical(lvo_mod, synth):
    """LVO_OPT_ODO_REUSE (default on): a scan-to-scan feature whose closest / same-ring / adjacent-ring points (laserOdometry.cpp:386-440,
    :470-532) are certified unchanged by the guard radii of its last full association keeps its factor record in the following outer
    iterations (:364).  Correspondence rows of ALL ten iterations, counters, LM traces, poses and the maps built from them must equal
    those of associating every feature every time."""
    L = lvo_mod
    mk = dict(lanes=2, max_map_corner=1 << 18, max_map_surf=1 << 19)
    a, b = L.Lvo(**mk), L.Lvo(**mk)
    for c, v in ((a, 1), (b, 0)):
        c.set_option(L.LVO_OPT_GRAPHS, 0)
        c.set_option(L.LVO_OPT_ODO_REUSE, v)
        c.set_option(L.LVO_OPT_FIXPOINT_SKIP, 0)   # all ten iterations run: the certificate is exercised nine times per frame
    arrays = ("odo_corner_corr", "odo_plane_corr", "odo_lm_iters", "odo_final_cost", "map_corner_corr", "map_surf_corr", "map_lm_iters", "map_final_cost")
    probes = (L.P_ODO_CORNER_CORR, L.P_ODO_PLANE_CORR, L.P_ODO_LM_TRACE, L.P_MAP_CORNER_KNN, L.P_MAP_SURF_KNN)
    cert = feats = 0
    for k in range(12):
        sws = [synth.sweep(64, 0, k)[0], synth.sweep(64, 6, k)[0]]
        sa, oa, ma = a.step_batch(sws)
        sb, ob, mb = b.step_batch(sws)
        assert sa == sb and np.array_equal(oa, ob) and np.array_equal(ma, mb), k
        for lane in range(2):
            x, y = a.stats(lane), b.stats(lane)
            for name in arrays:
                assert list(getattr(x, name)) == list(getattr(y, name)), (k, lane, name)
            for what in probes:
                assert np.array_equal(a.probe(what, lane), b.probe(what, lane)), (k, lane, what)
            assert list(y.odo_certified) == [0] * 16 and x.odo_certified[0] == 0
            if k > 0:
                cert += sum(x.odo_certified[1:10]); feats += 9 * (x.n_sharp + x.n_flat)
    assert cert > 0.5 * feats, (cert, feats)   # most features are carried over from the second or third iteration on
    for lane in range(2):
        for which in (0, 1):
            pa, ca = a.map_export(lane, which)
            pb, cb = b.map_export(lane, which)
            assert np.array_equal(ca, cb) and np.array_equal(pa.view(np.uint32), pb.view(np.uint32))
    a.close(); b.close()
