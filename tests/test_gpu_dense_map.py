"""BASELINE.json configs[2] at its stated size: lvo_scan_to_map against a map of ~100 k corner + ~400 k surf points in the 75-cube
neighbourhood (after the per-cube re-filter), CUDA vs the oracle: FromMap order, voxel stacks and the 5-NN index sets of outer
iteration 0 bit-exact, LM control flow, pose within 1e-4 m / 1e-5 rad, map sizes after insertion + re-filter equal
(reference src/laserMapping.cpp:509-549, 582-584, 648-652, 737-801)."""
import numpy as np
import pytest

from conftest import record_metric
from dense_map import make_dense_map
from oracle_py import Oracle

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def rot_err(qa, qb):
    return 2 * np.arccos(min(1.0, abs(float(np.dot(qa, qb)))))


def test_scan_to_map_dense_map_parity(lvo_mod, synth):
    L = lvo_mod
    corner, cc, surf, sc = make_dense_map()
    assert len(corner) >= 95000 and len(surf) >= 380000
    O = Oracle()
    lvo = L.Lvo(max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 20)
    O.map_import(0, corner, cc); O.map_import(1, surf, sc)
    lvo.map_import(0, corner, cc, surf, sc)
    ident = np.array([0, 0, 0, 1, 0, 0, 0], float)
    for k in range(2):   # the second call searches the map as the first one's re-filter left it
        f = O.extract(synth.sweep(64, 0, k)[0])
        odom = np.array([0, 0, 0, 1, 0.8 * k, 0.02 * k, 0], float)
        st_o, pose_o, corr_o = O.mapping(f["less_sharp"], f["less_flat"], f["full"], odom)
        st_g, pose_g, _ = lvo.scan_to_map(f["less_sharp"], f["less_flat"], f["full"], odom)
        assert st_o == 0 and st_g == 0
        info = O.mapping_info()
        s = lvo.stats()
        assert s.map_corner_from_map + s.map_surf_from_map >= 400000, (s.map_corner_from_map, s.map_surf_from_map)
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_CORNER_FROM_MAP)), _bits(info["corner_from_map"])), k
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_SURF_FROM_MAP)), _bits(info["surf_from_map"])), k
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_CORNER_STACK)), _bits(info["corner_stack"]))
        assert np.array_equal(_bits(lvo.probe(L.P_MAP_SURF_STACK)), _bits(info["surf_stack"]))
        kc, ks = lvo.probe(L.P_MAP_CORNER_KNN), lvo.probe(L.P_MAP_SURF_KNN)
        vc, vs = lvo.probe(L.P_MAP_CORNER_VALID), lvo.probe(L.P_MAP_SURF_VALID)
        tr = lvo.probe(L.P_MAP_LM_TRACE)
        flips = rows = 0
        for o in range(O.outer):
            lg = O.mapping_log(o)
            f1 = int((kc[o] != lg["corner_knn"]).any(axis=1).sum() + (ks[o] != lg["surf_knn"]).any(axis=1).sum())
            f2 = int((vc[o] != lg["corner_valid"]).sum() + (vs[o] != lg["surf_valid"]).sum())
            if o == 0:   # identical pose -> identical queries
                assert f1 == 0 and f2 == 0, (k, f1, f2)
                assert (kc[0][:, 0] >= 0).mean() > 0.02 and (ks[0][:, 0] >= 0).mean() > 0.25   # the searches really hit the (unrelated, synthetic) map
            flips += f1 + f2
            rows += 2 * (len(kc[o]) + len(ks[o]))
            if f1 == 0 and f2 == 0:
                n = len(lg["lm"])
                assert np.array_equal(tr[o][:n, 9], lg["lm"][:, 9]), (k, o)
        # both sides are deterministic on fixed inputs: a B200 run records 0 differing rows on every frame of this test
        print(f"dense map frame {k}: {flips} of {rows} kNN / accept rows differ")
        record_metric(f"dense_map_rows_differing_from_oracle/frame{k}", {"differ": flips, "rows": rows})
        assert flips == 0, (flips, rows)
        assert np.linalg.norm(pose_g[4:] - pose_o[4:]) < 1e-4 and rot_err(pose_g[:4], pose_o[:4]) < 1e-5, (k, pose_g, pose_o)
        lvo.set_map_correction(0, corr_o)
        for which in (0, 1):
            pg, cg = lvo.map_export(0, which)
            po, co = O.map_export(which)
            assert len(pg) == len(po) and np.array_equal(cg, co), (k, which, len(pg), len(po))
            assert (_bits(pg) != _bits(po)).mean() < 1e-3
        print(f"dense map frame {k}: neighbourhood {s.map_corner_from_map}+{s.map_surf_from_map} pts, queries {s.map_corner_stack}+{s.map_surf_stack}, "
              f"kNN/accept rows that differ from the oracle over 10 outer iterations: {flips} of {rows}")
    lvo.close()
