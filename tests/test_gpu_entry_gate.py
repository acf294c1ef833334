"""GPU tests of the entry gate every context-taking entry point passes first: while an *_async step is in flight every entry point
but lvo_wait, lvo_destroy and lvo_last_error returns LVO_E_STATE, writes none of its outputs and leaves the step's results exactly
as an undisturbed twin context computes them; every per-lane entry point refuses a bad lane with LVO_E_BADARG and a message.

The calls below get only valid host and device buffers: a call that a context accepted would run stream-ordered after the step."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_depth import keypoints

pytestmark = pytest.mark.gpu

P = 131072   # max_points: every synthetic HDL-64 sweep (~119.4 k points) fits
CAPS = dict(max_points=P, max_map_corner=1 << 16, max_map_surf=1 << 17)
LANES = 2
PROBES = 24
SENT = -7.0
# context-free, or usable while a step is in flight
EXEMPT = {"lvo_default_config", "lvo_create", "lvo_state_bytes", "lvo_destroy", "lvo_last_error", "lvo_wait"}


def sentinel(ctype):
    o = ctype()
    C.memset(C.addressof(o), 0xA5, C.sizeof(o))
    return o


def is_sentinel(o):
    return bytes(o) == b"\xa5" * C.sizeof(o)


class Calls:
    """One valid call of every entry point that takes a context, into sentinel-filled outputs.  calls()[name](lane) returns
    (status, outputs untouched); lane is ignored by the calls that take none."""

    def __init__(self, L, x, sw, feats, snap):
        import torch
        self.L, self.x, self.lib, self.h = L, x, x.lib, x.h
        self.sw, self.feats, self.snap = sw, feats, snap
        self.keep = []   # arrays behind the views, alive until the calls have returned
        self.views = (L.CloudView * LANES)(*[self.view(s) for s in sw])
        self.d_sw = [torch.from_numpy(s).cuda() for s in sw]
        self.small = np.ascontiguousarray(sw[0][:5000])
        self.d_small = torch.from_numpy(self.small).cuda()
        self.uv = np.ascontiguousarray(keypoints(L.KITTI00_CAMERA, np.random.default_rng(5)), np.float32)
        self.d_uv = torch.from_numpy(np.ascontiguousarray(self.uv)).cuda()
        self.cam = L.camera_of()
        self.cams = (L.Camera * LANES)(*[L.camera_of() for _ in range(LANES)])
        torch.cuda.synchronize()

    def view(self, a):
        v, arr = self.L.view_of(a)
        self.keep.append(arr)
        return v

    def cloud_out(self, cap):
        buf = np.full((max(cap, 1), 4), SENT, np.float32)
        return self.L.CloudOut(buf.ctypes.data, cap, 12345), buf

    @staticmethod
    def out_untouched(o):
        return o[0].n == 12345 and (o[1] == SENT).all()

    def dev(self, shape, dtype):
        import torch
        t = torch.full(shape, -7, dtype=dtype, device="cuda")
        torch.cuda.synchronize()
        return t

    @staticmethod
    def dev_untouched(*ts):
        return all(bool((t == -7).all()) for t in ts)

    def poses(self):
        return sentinel(self.L.Pose * LANES), sentinel(self.L.Pose * LANES)

    def calls(self):
        L, lib, h = self.L, self.lib, self.h
        ident = L.np_to_pose([0, 0, 0, 1, 0, 0, 0])
        VP, NS = C.c_void_p * LANES, C.c_size_t * LANES
        ptrs = VP(*[t.data_ptr() for t in self.d_sw])
        ns = NS(*[len(s) for s in self.sw])
        view = self.view

        def get_stats(lane):
            s = sentinel(L.Stats)
            return lib.lvo_get_stats(h, lane, C.byref(s), C.sizeof(s)), is_sentinel(s)

        def extract_features(lane):
            outs = [self.cloud_out(P) for _ in range(5)]
            r = lib.lvo_extract_features(h, view(self.sw[0]), *[C.byref(o[0]) for o in outs])
            return r, all(self.out_untouched(o) for o in outs)

        def scan_to_scan(lane):
            f = self.feats
            a, b = sentinel(L.Pose), sentinel(L.Pose)
            r = lib.lvo_scan_to_scan(h, view(f["sharp"]), view(f["less_sharp"]), view(f["flat"]), view(f["less_flat"]), C.byref(a), C.byref(b))
            return r, is_sentinel(a) and is_sentinel(b)

        def scan_to_map(lane):
            f = self.feats
            p, o = sentinel(L.Pose), self.cloud_out(P)
            r = lib.lvo_scan_to_map(h, view(f["less_sharp"]), view(f["less_flat"]), view(f["full"]), C.byref(ident), C.byref(p), C.byref(o[0]))
            return r, is_sentinel(p) and self.out_untouched(o)

        def step_batch(lane):
            po, pm = self.poses()
            return lib.lvo_step_batch(h, self.views, po, pm), is_sentinel(po) and is_sentinel(pm)

        def step_batch_dev(lane):
            po, pm = self.poses()
            return lib.lvo_step_batch_dev(h, ptrs, ns, po, pm), is_sentinel(po) and is_sentinel(pm)

        def step_batch_pipelined(lane):
            po, pm = self.poses()
            return lib.lvo_step_batch_pipelined(h, self.views, None, po, pm), is_sentinel(po) and is_sentinel(pm)

        def map_import(lane):
            pts = np.ascontiguousarray(self.small[:10])
            cube = np.arange(10, dtype=np.int32)
            r = lib.lvo_map_import(h, lane, pts.ctypes.data, cube.ctypes.data, 10, pts.ctypes.data, cube.ctypes.data, 10)
            return r, True

        def map_export(lane):
            o = self.cloud_out(1 << 17)
            cube = np.full(1 << 17, -7, np.int32)
            r = lib.lvo_map_export(h, lane, 1, C.byref(o[0]), cube.ctypes.data)
            return r, self.out_untouched(o) and (cube == -7).all()

        def get_map_correction(lane):
            p = sentinel(L.Pose)
            return lib.lvo_get_map_correction(h, lane, C.byref(p)), is_sentinel(p)

        def probe_fetch(lane):
            buf = np.full(P * 16, 0xA5, np.uint8)
            n = C.c_size_t(12345)
            r = lib.lvo_probe_fetch(h, lane, L.P_FULL, buf.ctypes.data, buf.nbytes, C.byref(n))
            return r, n.value == 12345 and (buf == 0xA5).all()

        def voxel_downsample(lane):
            o = self.cloud_out(len(self.small))
            return lib.lvo_voxel_downsample(h, view(self.small), 0.4, C.byref(o[0])), self.out_untouched(o)

        def voxel_downsample_dev(lane):
            import torch
            d_out = self.dev((len(self.small), 4), torch.float32)
            n, ms = C.c_size_t(12345), C.c_float(SENT)
            r = lib.lvo_voxel_downsample_dev(h, self.d_small.data_ptr(), len(self.small), 0.4, d_out.data_ptr(), C.byref(n), C.byref(ms))
            return r, n.value == 12345 and ms.value == SENT and self.dev_untouched(d_out)

        def knn(lane):
            ind = np.full((100, 5), -7, np.int32)
            sq = np.full((100, 5), SENT, np.float32)
            r = lib.lvo_knn(h, view(self.small), view(self.small[:100]), 5, 1.0, ind.ctypes.data, sq.ctypes.data)
            return r, (ind == -7).all() and (sq == SENT).all()

        def knn5_throughput(lane):
            import torch
            d_ind, d_sq = self.dev((100, 5), torch.int32), self.dev((100, 5), torch.float32)
            mc, qc, ms = (C.c_int * 1)(len(self.small)), (C.c_int * 1)(100), C.c_float(SENT)
            r = lib.lvo_knn5_throughput(h, self.d_small.data_ptr(), mc, self.d_small.data_ptr(), qc, 1, 1, d_ind.data_ptr(), d_sq.data_ptr(), C.byref(ms))
            return r, ms.value == SENT and self.dev_untouched(d_ind, d_sq)

        def get_timings(lane):
            t = sentinel(L.Timings)
            return lib.lvo_get_timings(h, C.byref(t)), is_sentinel(t)

        def depth_associate(lane):
            k = len(self.uv)
            d, v, nn = np.full(k, SENT, np.float32), np.full(k, -7, np.int32), np.full((k, 3), -7, np.int32)
            o = self.cloud_out(P)
            r = lib.lvo_depth_associate(h, view(self.sw[0]), C.byref(self.cam), self.uv.ctypes.data, k, d.ctypes.data, v.ctypes.data, nn.ctypes.data,
                                        C.byref(o[0]))
            return r, (d == SENT).all() and (v == -7).all() and (nn == -7).all() and self.out_untouched(o)

        def depth_associate_batch(lane):
            k = len(self.uv)
            d = [np.full(k, SENT, np.float32) for _ in range(LANES)]
            v = [np.full(k, -7, np.int32) for _ in range(LANES)]
            nn = [np.full((k, 3), -7, np.int32) for _ in range(LANES)]
            p = lambda xs: VP(*[a.ctypes.data for a in xs])
            r = lib.lvo_depth_associate_batch(h, self.cams, self.views, VP(*[self.uv.ctypes.data] * LANES), NS(*[k] * LANES), p(d), p(v), p(nn))
            return r, all((a == SENT).all() and (b == -7).all() and (c == -7).all() for a, b, c in zip(d, v, nn))

        def depth_associate_batch_dev(lane):
            import torch
            k = len(self.uv)
            d = [self.dev((k,), torch.float32) for _ in range(LANES)]
            v = [self.dev((k,), torch.int32) for _ in range(LANES)]
            nn = [self.dev((k, 3), torch.int32) for _ in range(LANES)]
            p = lambda xs: VP(*[t.data_ptr() for t in xs])
            r = lib.lvo_depth_associate_batch_dev(h, self.cams, ptrs, ns, VP(*[self.d_uv.data_ptr()] * LANES), NS(*[k] * LANES), p(d), p(v), p(nn))
            return r, self.dev_untouched(*d, *v, *nn)

        def map_cloud(lane):
            o = self.cloud_out(3 << 16)
            return lib.lvo_map_cloud(h, lane, 1, C.byref(o[0])), self.out_untouched(o)

        def map_cloud_batch(lane):
            outs = [self.cloud_out(3 << 16) for _ in range(LANES)]
            arr = (L.CloudOut * LANES)(*[o[0] for o in outs])
            r = lib.lvo_map_cloud_batch(h, L.LVO_MAP_WHOLE, arr)
            return r, all(arr[l].n == 12345 and (outs[l][1] == SENT).all() for l in range(LANES))

        def map_cloud_batch_dev(lane):
            import torch
            d = [self.dev((3 << 16, 4), torch.float32) for _ in range(LANES)]
            n = NS(*[12345] * LANES)
            r = lib.lvo_map_cloud_batch_dev(h, L.LVO_MAP_WHOLE, VP(*[t.data_ptr() for t in d]), NS(*[3 << 16] * LANES), n)
            return r, list(n) == [12345] * LANES and self.dev_untouched(*d)

        def transform_cloud(lane):
            o = self.cloud_out(len(self.small))
            return lib.lvo_transform_cloud(h, view(self.small), None, 0, C.byref(o[0])), self.out_untouched(o)

        def lane_save(lane):
            buf = np.full(len(self.snap), 0xA5, np.uint8)
            n = C.c_size_t(12345)
            r = lib.lvo_lane_save(h, lane, buf.ctypes.data, buf.nbytes, C.byref(n))
            return r, n.value == 12345 and (buf == 0xA5).all()

        def lane_get_config(lane):
            cfg = sentinel(L.LaneConfig)
            return lib.lvo_lane_get_config(h, lane, C.byref(cfg)), is_sentinel(cfg)

        nothing = lambda f: (lambda lane: (f(lane), True))
        return {
            "lvo_get_stats": get_stats,
            "lvo_lane_status": nothing(lambda lane: lib.lvo_lane_status(h, lane)),
            "lvo_extract_features": extract_features,
            "lvo_scan_to_scan": scan_to_scan,
            "lvo_scan_to_map": scan_to_map,
            "lvo_step_batch": step_batch,
            "lvo_step_batch_dev": step_batch_dev,
            "lvo_step_batch_pipelined": step_batch_pipelined,
            "lvo_step_batch_async": nothing(lambda lane: lib.lvo_step_batch_async(h, self.views)),
            "lvo_step_batch_dev_async": nothing(lambda lane: lib.lvo_step_batch_dev_async(h, ptrs, ns)),
            "lvo_set_lane_active": nothing(lambda lane: lib.lvo_set_lane_active(h, lane, 1)),
            "lvo_set_lane_map_update": nothing(lambda lane: lib.lvo_set_lane_map_update(h, lane, 1)),
            "lvo_lane_reset": nothing(lambda lane: lib.lvo_lane_reset(h, lane)),
            "lvo_lane_configure": nothing(lambda lane: lib.lvo_lane_configure(h, lane, None)),
            "lvo_lane_get_config": lane_get_config,
            "lvo_lane_save": lane_save,
            "lvo_lane_load": nothing(lambda lane: lib.lvo_lane_load(h, lane, self.snap.ctypes.data, self.snap.nbytes)),
            "lvo_map_import": map_import,
            "lvo_map_export": map_export,
            "lvo_map_cloud": map_cloud,
            "lvo_map_cloud_batch": map_cloud_batch,
            "lvo_map_cloud_batch_dev": map_cloud_batch_dev,
            "lvo_get_map_correction": get_map_correction,
            "lvo_set_map_correction": nothing(lambda lane: lib.lvo_set_map_correction(h, lane, C.byref(ident))),
            "lvo_set_odometry_state": nothing(lambda lane: lib.lvo_set_odometry_state(h, lane, C.byref(ident), C.byref(ident))),
            "lvo_probe_fetch": probe_fetch,
            "lvo_transform_cloud": transform_cloud,
            "lvo_voxel_downsample": voxel_downsample,
            "lvo_voxel_downsample_dev": voxel_downsample_dev,
            "lvo_knn": knn,
            "lvo_knn5_throughput": knn5_throughput,
            "lvo_depth_associate": depth_associate,
            "lvo_depth_associate_batch": depth_associate_batch,
            "lvo_depth_associate_batch_dev": depth_associate_batch_dev,
            "lvo_get_timings": get_timings,
            "lvo_set_stream": nothing(lambda lane: lib.lvo_set_stream(h, None)),
            "lvo_set_option": nothing(lambda lane: lib.lvo_set_option(h, L.LVO_OPT_STAGE_TIMING, 1)),
        }


LANE_CALLS = {"lvo_get_stats", "lvo_lane_status", "lvo_set_lane_active", "lvo_set_lane_map_update", "lvo_lane_reset", "lvo_lane_configure",
              "lvo_lane_get_config", "lvo_lane_save", "lvo_lane_load", "lvo_map_import", "lvo_map_export", "lvo_map_cloud",
              "lvo_get_map_correction", "lvo_set_map_correction", "lvo_set_odometry_state", "lvo_probe_fetch"}


def make(L):
    return L.Lvo(lanes=LANES, **CAPS)


def frames(synth, f):
    return [np.ascontiguousarray(synth.sweep(64, lane, f)[0], np.float32) for lane in range(LANES)]


def features(L, synth):
    one = L.Lvo(lanes=1, **CAPS)
    ex = one.extract_features(synth.sweep(64, 3, 0)[0])[1]
    one.close()
    return ex


def probes(lvo, lane):
    out = []
    for what in range(PROBES):
        try:
            out.append(lvo.probe(what, lane).tobytes())
        except Exception as e:   # a probe that is not available must be unavailable in both contexts
            out.append(str(e))
    return out


def test_every_entry_point_waits_for_an_async_step(lvo_mod, synth):
    L = lvo_mod
    x, twin = make(L), make(L)
    for f in range(3):
        for c in (x, twin):
            c.step_batch(frames(synth, f))
    sw = frames(synth, 3)
    table = Calls(L, x, sw, features(L, synth), x.lane_save(1)).calls()
    assert set(table) == set(L.EXPORTS) - EXEMPT, "an entry point without a row here would not be checked against the gate"
    x.step_batch_async(sw)
    twin.step_batch_async(sw)
    for name, call in table.items():
        r, untouched = call(1)
        assert r == L.LVO_E_STATE, (name, r)
        assert untouched, f"{name} wrote an output while a step was in flight"
        assert b"lvo_wait" in x.lib.lvo_last_error(x.h), name
    got, ref = x.wait(), twin.wait()
    assert got[0] == ref[0] and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2]), "poses"
    assert [x.lane_status(l) for l in range(LANES)] == [twin.lane_status(l) for l in range(LANES)]
    assert [bytes(x.stats(l)) for l in range(LANES)] == [bytes(twin.stats(l)) for l in range(LANES)]
    assert x.timings().kernel_launches == twin.timings().kernel_launches
    for a, b in zip(x.map_cloud_batch(L.LVO_MAP_REGISTERED), twin.map_cloud_batch(L.LVO_MAP_REGISTERED)):
        assert len(a) > 1000 and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    for lane in range(LANES):
        assert probes(x, lane) == probes(twin, lane), lane
    x.close()
    twin.close()


def test_bad_lane(lvo_mod, synth):
    L = lvo_mod
    x = make(L)
    x.step_batch(frames(synth, 0))
    table = Calls(L, x, frames(synth, 1), features(L, synth), x.lane_save(1)).calls()
    assert LANE_CALLS <= set(table)
    outs = (L.CloudOut * LANES)()
    for name in sorted(LANE_CALLS):
        for lane in (-1, LANES):
            assert x.lib.lvo_map_cloud_batch(x.h, 7, outs) == L.LVO_E_BADARG   # an error message without the word "lane"
            assert b"lane" not in x.lib.lvo_last_error(x.h)
            r, untouched = table[name](lane)
            assert r == L.LVO_E_BADARG and untouched, (name, lane, r)
            assert b"lane" in x.lib.lvo_last_error(x.h), (name, lane)
    x.close()
