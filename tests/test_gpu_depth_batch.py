"""GPU tests of the batched camera-lidar depth association (lvo_depth_associate_batch / _dev): per lane bit-exact against the CPU
oracle and the single call, independent of the other lanes, idle lanes skipped, no effect on the batched pipeline, a launch
count that does not depend on lanes or keypoints, errors before anything is enqueued, and arena growth."""
import ctypes as C

import numpy as np
import pytest

from oracle_py import Oracle
from test_gpu_depth import keypoints

pytestmark = pytest.mark.gpu

P = 131072   # max_points of the contexts below: every synthetic HDL-64 sweep (~119.4 k points) fits, keypoints up to P / 2
EDGE_UV = np.array([[5.0, 5.0], [-3.0, 0.1], [0.0, 0.0], [0.0, 0.0], [0.84, -0.24], [-0.84, 0.24]], np.float32)


def small_ctx(L, lanes, **kw):
    return L.Lvo(lanes=lanes, max_points=P, max_map_corner=1 << 16, max_map_surf=1 << 17, **kw)


def camera(L, lane):
    """KITTI00_CAMERA with the extrinsic turned by a small rotation and shifted, different for every lane."""
    cam = dict(L.KITTI00_CAMERA)
    if lane == 0:
        return cam
    a = 0.004 * lane * np.array([1.0, -0.5, 0.7])
    th = np.linalg.norm(a)
    k = a / th
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
    E = np.array(cam["extrinsic"], np.float64).reshape(3, 4)
    E2 = np.concatenate([R @ E[:, :3], (R @ E[:, 3:]) + 0.03 * lane * np.array([[1.0], [-1.0], [0.5]])], 1)
    cam["extrinsic"] = [float(x) for x in E2.astype(np.float32).reshape(12)]
    return cam


def camera_z(pts, cam):
    E = np.array(cam["extrinsic"], np.float64).reshape(3, 4)
    return pts[:, :3].astype(np.float64) @ E[2, :3] + E[2, 3]


def lane_inputs(L, synth):
    """8 lanes on different sequences and frames, with 0, 1120, the edge set and P / 2 keypoints, a sweep entirely behind the
    camera and one with two depth points."""
    cam0 = L.KITTI00_CAMERA
    rng = np.random.default_rng(7)
    sw, kp, cams = [], [], []
    for lane, (seq, frame) in enumerate([(0, 0), (1, 3), (2, 5), (3, 1), (4, 2), (0, 7), (1, 9), (2, 2)]):
        pts, _ = synth.sweep(64, seq, frame)
        cam = camera(L, lane)
        z = camera_z(pts, cam)
        if lane == 4:
            pts = pts[z < -0.5]                                             # entirely behind the camera
        if lane == 5:
            pts = np.concatenate([pts[z < -0.5][:50], pts[z > 5.0][:2]])     # two depth points
        if lane == 1:
            uv = np.zeros((0, 2), np.float32)
        elif lane == 2:
            uv = EDGE_UV
        elif lane == 3:
            uv = np.stack([rng.uniform(-0.9, 0.9, P // 2), rng.uniform(-0.3, 0.3, P // 2)], 1).astype(np.float32)
        elif lane == 7:
            uv = keypoints(cam0, rng)[:5]
        else:
            uv = keypoints(cam0, rng)
        sw.append(np.ascontiguousarray(pts, np.float32))
        kp.append(uv)
        cams.append(cam)
    return sw, kp, cams


def reference(L, sweeps, kps, cams):
    """Per lane: the oracle, and the single call in a 1-lane context; both must agree."""
    O = Oracle()
    one = small_ctx(L, 1)
    refs = []
    for pts, uv, cam in zip(sweeps, kps, cams):
        _, _, d_o, v_o, nn_o = O.depth(pts, cam["extrinsic"], uv)
        _, d_g, v_g, nn_g = one.depth_associate(pts, uv, camera=cam)
        assert_same((d_g, v_g, nn_g), (d_o, v_o, nn_o))
        refs.append((d_o.copy(), v_o.copy(), nn_o.copy()))
    one.close()
    return refs


def assert_same(got, ref, what=""):
    d, v, nn = got
    d_r, v_r, nn_r = ref
    assert d.shape == d_r.shape and np.array_equal(d.view(np.uint32), d_r.view(np.uint32)), f"{what} depth"
    assert np.array_equal(v, v_r), f"{what} valid"
    assert np.array_equal(nn, nn_r), f"{what} nn"


def layout(L, pts, stride):
    return {12: lambda: np.ascontiguousarray(pts[:, :3]), 16: lambda: pts, 32: lambda: L.to_pcl_layout(pts)}[stride]()


def dev_call(lvo, sweeps, kps, cams, want_nn=True):
    """lvo_depth_associate_batch_dev over torch device buffers; returns per-lane numpy results (None for idle lanes)."""
    import torch
    act = lvo._active
    d_sw = [torch.from_numpy(s).cuda() if a else None for s, a in zip(sweeps, act)]
    d_kp = [torch.from_numpy(np.ascontiguousarray(k)).cuda() if a else None for k, a in zip(kps, act)]
    d_d = [torch.full((max(len(k), 1),), -7.0, device="cuda") if a else None for k, a in zip(kps, act)]
    d_v = [torch.full((max(len(k), 1),), -7, dtype=torch.int32, device="cuda") if a else None for k, a in zip(kps, act)]
    d_n = [torch.full((max(len(k), 1), 3), -7, dtype=torch.int32, device="cuda") if a else None for k, a in zip(kps, act)]
    torch.cuda.synchronize()
    ptr = lambda t: t.data_ptr() if t is not None else None
    lvo.depth_associate_batch_dev([ptr(t) for t in d_sw], [len(s) if a else None for s, a in zip(sweeps, act)], [ptr(t) for t in d_kp],
                                  [len(k) if a else None for k, a in zip(kps, act)], [ptr(t) for t in d_d], [ptr(t) for t in d_v],
                                  [ptr(t) for t in d_n] if want_nn else None, cameras=cams)
    out = []
    for k, a, d, v, n in zip(kps, act, d_d, d_v, d_n):
        out.append((d.cpu().numpy()[:len(k)], v.cpu().numpy()[:len(k)], n.cpu().numpy()[:len(k)]) if a else None)
    return out


def test_parity_host_and_device_forms(lvo_mod, synth):
    L = lvo_mod
    sweeps, kps, cams = lane_inputs(L, synth)
    assert len(sweeps[4]) > 1000 and len(kps[3]) == P // 2
    refs = reference(L, sweeps, kps, cams)
    assert not refs[4][1].any() and not refs[5][1].any() and 0.3 < refs[0][1].mean() < 0.95
    lvo = small_ctx(L, 8)
    for stride in (12, 16, 32):
        got = lvo.depth_associate_batch([layout(L, s, stride) for s in sweeps], kps, cameras=cams)
        for lane in range(8):
            assert_same(got[lane], refs[lane], f"host stride {stride} lane {lane}")
    got = dev_call(lvo, sweeps, kps, cams)
    for lane in range(8):
        assert_same(got[lane], refs[lane], f"device lane {lane}")
    # without nn: the other outputs are the same
    got = dev_call(lvo, sweeps, kps, cams, want_nn=False)
    for lane in range(8):
        assert np.array_equal(got[lane][0].view(np.uint32), refs[lane][0].view(np.uint32)) and (got[lane][2] == -7).all()
    lvo.close()


def test_lane_independence(lvo_mod, synth):
    L = lvo_mod
    sweeps, kps, cams = lane_inputs(L, synth)
    lvo = small_ctx(L, 8)
    base = lvo.depth_associate_batch(sweeps, kps, cameras=cams)
    perm = [5, 2, 7, 0, 3, 6, 1, 4]
    got = lvo.depth_associate_batch([sweeps[p] for p in perm], [kps[p] for p in perm], cameras=[cams[p] for p in perm])
    for lane, p in enumerate(perm):
        assert_same(got[lane], base[p], f"permuted lane {lane}")
    # other lanes' sweeps and keypoints replaced: lanes 0 and 3 unchanged
    other_sw = [synth.sweep(64, 5, lane)[0] for lane in range(8)]
    other_kp = [keypoints(L.KITTI00_CAMERA, np.random.default_rng(100 + lane)) for lane in range(8)]
    sw2 = [sweeps[l] if l in (0, 3) else other_sw[l] for l in range(8)]
    kp2 = [kps[l] if l in (0, 3) else other_kp[l] for l in range(8)]
    got = dev_call(lvo, sw2, kp2, cams)
    for lane in (0, 3):
        assert_same(got[lane], base[lane], f"lane {lane} with other neighbours")
    lvo.close()


def raw_batch(lvo, cams, views, kps, nkp, depth, valid, nn):
    """lvo_depth_associate_batch with explicit per-lane pointers (None = NULL entry); an argument that is None is a NULL array."""
    n = lvo.lanes
    VP = C.c_void_p * n
    arr = lambda xs: None if xs is None else VP(*[x for x in xs])
    return lvo.lib.lvo_depth_associate_batch(lvo.h, None if cams is None else lvo._cameras(cams),
                                             None if views is None else (type(views[0]) * n)(*views), arr(kps),
                                             None if nkp is None else (C.c_size_t * n)(*nkp), arr(depth), arr(valid), arr(nn))


def buffers(kps, sentinel=-7):
    d = [np.full(max(len(k), 1), float(sentinel), np.float32) for k in kps]
    v = [np.full(max(len(k), 1), sentinel, np.int32) for k in kps]
    nn = [np.full((max(len(k), 1), 3), sentinel, np.int32) for k in kps]
    return d, v, nn


def untouched(bufs, lanes, sentinel=-7):
    d, v, nn = bufs
    return all((d[l] == sentinel).all() and (v[l] == sentinel).all() and (nn[l] == sentinel).all() for l in lanes)


def test_idle_lanes(lvo_mod, synth):
    L = lvo_mod
    sweeps, kps, cams = lane_inputs(L, synth)
    lvo = small_ctx(L, 8)
    full = lvo.depth_associate_batch(sweeps, kps, cameras=cams)
    idle = (1, 4, 6)
    for l in idle:
        lvo.set_lane_active(l, False)
    # NULL entries for the idle lanes (the binding passes None)
    got = lvo.depth_associate_batch([None if l in idle else s for l, s in enumerate(sweeps)], [None if l in idle else k for l, k in enumerate(kps)], cameras=cams)
    for l in range(8):
        if l in idle:
            assert got[l] is None
        else:
            assert_same(got[l], full[l], f"active lane {l}")
    got = dev_call(lvo, sweeps, kps, cams)
    for l in range(8):
        if l in idle:
            assert got[l] is None
        else:
            assert_same(got[l], full[l], f"device active lane {l}")
    # valid pointers and sentinel-filled buffers for the idle lanes: not written
    views = [L.view_of(s)[0] for s in sweeps]
    bufs = buffers(kps)
    r = raw_batch(lvo, cams, views, [k.ctypes.data if len(k) else None for k in kps], [len(k) for k in kps],
                  [x.ctypes.data for x in bufs[0]], [x.ctypes.data for x in bufs[1]], [x.ctypes.data for x in bufs[2]])
    assert r == L.LVO_OK
    assert untouched(bufs, idle)
    for l in range(8):
        if l not in idle:
            n = len(kps[l])
            assert_same((bufs[0][l][:n], bufs[1][l][:n], bufs[2][l][:n]), full[l], f"raw active lane {l}")
    # all lanes idle: nothing to do
    for l in range(8):
        lvo.set_lane_active(l, False)
    assert lvo.depth_associate_batch([None] * 8, [None] * 8) == [None] * 8
    lvo.close()


PROBES = 24


def probes(lvo, lane):
    out = []
    for what in range(PROBES):
        try:
            out.append(lvo.probe(what, lane).tobytes())
        except Exception as e:   # a probe that is not available must be unavailable in both contexts
            out.append(str(e))
    return out


@pytest.mark.parametrize("skip,graphs", [(1, 0), (1, 1), (2, 0), (2, 1)])
def test_no_effect_on_pipeline(lvo_mod, synth, skip, graphs):
    import torch
    L = lvo_mod
    ctx = [small_ctx(L, 2, skip_frame=skip) for _ in range(2)]   # ctx[0] runs depth calls between its steps, ctx[1] does not
    for c in ctx:
        c.set_option(L.LVO_OPT_GRAPHS, graphs)
    frames = [[synth.sweep(64, lane, f)[0] for lane in range(2)] for f in range(13)]
    rng = np.random.default_rng(3)
    uv = [keypoints(L.KITTI00_CAMERA, rng) for _ in range(2)]
    cams = [camera(L, 1), camera(L, 2)]
    ref = reference(L, frames[0], uv, cams)
    for f in range(12):
        outs = []
        for i, c in enumerate(ctx):
            if i == 0:
                got = c.depth_associate_batch(frames[f], uv, cameras=cams)
                if f == 0:
                    for lane in range(2):
                        assert_same(got[lane], ref[lane])
            if f < 8:
                r = c.step_batch_pipelined(frames[f], frames[f + 1])
            else:
                d = [torch.from_numpy(s).cuda() for s in frames[f]]
                torch.cuda.synchronize()
                r = c.step_batch_dev([t.data_ptr() for t in d], [len(s) for s in frames[f]])
            launches = c.timings().kernel_launches
            if i == 0:
                dev_call(c, frames[(f + 5) % 13], uv, cams)
            outs.append((r, launches, [c.lane_status(l) for l in range(2)], [bytes(c.stats(l)) for l in range(2)]))
        (r0, n0, s0, st0), (r1, n1, s1, st1) = outs
        assert r0[0] == r1[0] and np.array_equal(r0[1], r1[1]) and np.array_equal(r0[2], r1[2]), f"frame {f} poses"
        assert n0 == n1 and s0 == s1 and st0 == st1, f"frame {f} launches / statuses / stats"
    for lane in range(2):
        for which in range(2):
            a, b = ctx[0].map_export(lane, which), ctx[1].map_export(lane, which)
            assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[1], b[1])
        assert np.array_equal(ctx[0].lane_save(lane), ctx[1].lane_save(lane))
        assert probes(ctx[0], lane) == probes(ctx[1], lane)
    for c in ctx:
        c.close()


def test_launch_count_is_independent_of_lanes_and_keypoints(lvo_mod, synth):
    L = lvo_mod
    pts = synth.sweep(64, 0, 0)[0]
    uv = keypoints(L.KITTI00_CAMERA, np.random.default_rng(1))
    counts = set()
    for lanes in (1, 8, 32):
        lvo = small_ctx(L, lanes)
        for k in (1, 1120):
            lvo.depth_associate_batch([pts] * lanes, [uv[:k]] * lanes)
            counts.add(("host", lvo.timings().kernel_launches))
            dev_call(lvo, [pts] * lanes, [uv[:k]] * lanes, None)
            counts.add(("dev", lvo.timings().kernel_launches))
        lvo.close()
    assert counts == {("host", 16), ("dev", 16)}, counts


def test_errors_leave_outputs_untouched(lvo_mod, synth):
    import torch
    L = lvo_mod
    pts = synth.sweep(64, 1, 1)[0]
    small = pts[:4000]
    lvo = L.Lvo(lanes=2, max_points=4096, max_map_corner=1 << 14, max_map_surf=1 << 15)
    uv = keypoints(L.KITTI00_CAMERA, np.random.default_rng(2))[:100]
    kps = [uv, uv]
    cams = [camera(L, 0), camera(L, 1)]
    ref = reference(L, [small, small], kps, cams)
    V = lambda a: L.view_of(a)[0]
    kp_ptr = [k.ctypes.data for k in kps]

    def call(views, kp=kp_ptr, nkp=(100, 100), null=None, cams_=cams, nn=True):
        bufs = buffers(kps)
        ptrs = [[x.ctypes.data for x in b] for b in bufs]
        if null is not None:
            ptrs[null[0]][null[1]] = None
        r = raw_batch(lvo, cams_, views, kp, list(nkp), ptrs[0], ptrs[1], ptrs[2] if nn else None)
        return r, bufs

    r, bufs = call([V(small), V(small)])
    assert r == L.LVO_OK
    for l in range(2):
        assert_same((bufs[0][l][:100], bufs[1][l][:100], bufs[2][l]), ref[l])
    # in flight
    lvo.step_batch_async([small, small])
    r, bufs = call([V(small), V(small)])
    assert r == L.LVO_E_STATE and untouched(bufs, (0, 1))
    lvo.wait()
    # capacity: too many points, too many keypoints (2 n_kp > max_points)
    big = pts[:4097]
    r, bufs = call([V(small), V(big)])
    assert r == L.LVO_E_CAPACITY and untouched(bufs, (0, 1))
    many = np.zeros((2049, 2), np.float32)
    r, bufs = call([V(small), V(small)], kp=[kp_ptr[0], many.ctypes.data], nkp=(100, 2049))
    assert r == L.LVO_E_CAPACITY and untouched(bufs, (0, 1))
    # bad arguments: mixed layouts, stride > 32, NULL arrays, NULL pointers of an active lane
    r, bufs = call([V(small), V(np.ascontiguousarray(small[:, :3]))])
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    wide = np.zeros((len(small), 12), np.float32)
    wide[:, :4] = small
    wv = L.CloudView(wide.ctypes.data, len(small), 48, 0, 12)
    r, bufs = call([wv, wv])
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    r, bufs = call([V(small), V(small)], cams_=None)
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    r, bufs = call(None)
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    r, bufs = call([V(small), V(small)], kp=None)
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    r, bufs = call([V(small), V(small)], kp=[kp_ptr[0], None])
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    for which in range(3):
        r, bufs = call([V(small), V(small)], null=(which, 1))
        assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1)), which
    bad_view = L.CloudView(None, len(small), 16, 0, 12)
    r, bufs = call([V(small), bad_view])
    assert r == L.LVO_E_BADARG and untouched(bufs, (0, 1))
    # device form: NULL arrays, capacity, NULL pointers
    d_sw = torch.from_numpy(small).cuda()
    d_big = torch.from_numpy(np.ascontiguousarray(big)).cuda()
    d_kp = torch.from_numpy(uv).cuda()
    d_out = [torch.full((100,), -7.0, device="cuda"), torch.full((100,), -7, dtype=torch.int32, device="cuda")]
    torch.cuda.synchronize()
    p = [d_sw.data_ptr(), d_sw.data_ptr()]
    kpp = [d_kp.data_ptr()] * 2
    outs = [[d_out[0].data_ptr()] * 2, [d_out[1].data_ptr()] * 2]
    with pytest.raises(L.LvoError, match="-1"):
        lvo.depth_associate_batch_dev(p, [4000, 4000], kpp, [100, 100], outs[0], [None, None])
    with pytest.raises(L.LvoError, match="-2"):
        lvo.depth_associate_batch_dev([p[0], d_big.data_ptr()], [4000, 4097], kpp, [100, 100], *outs)
    with pytest.raises(L.LvoError, match="-2"):
        lvo.depth_associate_batch_dev(p, [4000, 4000], kpp, [100, 2049], *outs)
    with pytest.raises(L.LvoError, match="-1"):
        lvo.depth_associate_batch_dev([p[0], None], [4000, 4000], kpp, [100, 100], *outs)
    n = C.c_size_t * 2
    assert lvo.lib.lvo_depth_associate_batch_dev(lvo.h, lvo._cameras(cams), None, n(4000, 4000), (C.c_void_p * 2)(*kpp), n(100, 100),
                                                 (C.c_void_p * 2)(*outs[0]), (C.c_void_p * 2)(*outs[1]), None) == L.LVO_E_BADARG
    assert (d_out[0] == -7).all() and (d_out[1] == -7).all()
    # the context still works, and so does its pipeline
    got = lvo.depth_associate_batch([small, small], kps, cameras=cams)
    for l in range(2):
        assert_same(got[l], ref[l])
    lvo.step_batch([small, small])
    lvo.close()


def test_arena_growth(lvo_mod, synth):
    L = lvo_mod
    O = Oracle()
    rng = np.random.default_rng(11)
    pts = [synth.sweep(64, l, 4)[0] for l in range(3)]
    uv = [keypoints(L.KITTI00_CAMERA, rng) for _ in range(3)]
    cams = [camera(L, l) for l in range(3)]
    lvo = small_ctx(L, 3)

    def check(sw, kp):
        for got in (lvo.depth_associate_batch(sw, kp, cameras=cams), dev_call(lvo, sw, kp, cams)):
            for l in range(3):
                if not lvo._active[l]:
                    assert got[l] is None
                    continue
                _, _, d, v, nn = O.depth(sw[l], cams[l]["extrinsic"], kp[l])
                assert_same(got[l], (d, v, nn), f"lane {l}")

    lvo.set_lane_active(2, False)
    check([p[:3000] for p in pts], [k[:10] for k in uv])          # small, two lanes
    lvo.set_lane_active(2, True)
    big_uv = [np.concatenate([k] * 20) for k in uv]                 # 22 400 keypoints per lane
    check(pts, big_uv)                                              # larger: points, keypoints and lanes grow
    check([p[:3000] for p in pts], [k[:10] for k in uv])           # small again
    lvo.close()
    lvo = small_ctx(L, 1)                                           # the device is healthy after lvo_destroy of a grown arena
    got = lvo.depth_associate_batch([pts[0]], [uv[0]], cameras=[cams[0]])
    _, _, d, v, nn = O.depth(pts[0], cams[0]["extrinsic"], uv[0])
    assert_same(got[0], (d, v, nn))
    lvo.close()
