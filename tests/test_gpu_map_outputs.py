"""GPU tests of the batched map outputs (lvo_map_cloud_batch / _dev): the surround and whole-map clouds of every lane equal
lvo_map_cloud, the registered clouds equal the LVO_P_REGISTERED probe of the lanes that mapped in the last step, lane selection
and size queries, lane lifecycle, errors before anything is written, no effect on the batched pipeline, a launch count that does
not depend on the number of lanes, and arena growth.  Every comparison is bitwise."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 131072   # max_points: every synthetic HDL-64 sweep (~119.4 k points) fits
CAPS = dict(max_points=P, max_map_corner=1 << 16, max_map_surf=1 << 17)
WHICH = (0, 1, 2)
SENTINEL = -7.0


class Sweeps:
    """Synthetic HDL-64 sweeps, generated once per (sequence, frame)."""

    def __init__(self, synth):
        self.synth, self.cache = synth, {}

    def __call__(self, seq, frame):
        if (seq, frame) not in self.cache:
            self.cache[(seq, frame)] = self.synth.sweep(64, seq, frame)[0]
        return self.cache[(seq, frame)]


@pytest.fixture(scope="module")
def sweeps(synth):
    return Sweeps(synth)


def make(L, lanes, graphs=-1, **kw):
    lvo = L.Lvo(lanes=lanes, debug_probes=0, **CAPS, **kw)
    lvo.set_option(L.LVO_OPT_GRAPHS, graphs)
    return lvo


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same(a, b):
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def dev_step(lvo, frame):
    import torch
    d = [torch.from_numpy(s).cuda() if s is not None else None for s in frame]
    torch.cuda.synchronize()
    return lvo.step_batch_dev([t.data_ptr() if t is not None else None for t in d], [len(s) if s is not None else None for s in frame])


def dev_call(lvo, which, lanes=None, slack=3):
    """lvo_map_cloud_batch_dev into sentinel-filled torch buffers with `slack` spare rows; checks that nothing beyond n was written
    and returns per-lane numpy clouds (None for lanes that were not requested)."""
    import torch
    n = lvo.map_cloud_batch_dev(which, [None] * lvo.lanes, [0] * lvo.lanes)
    want = set(range(lvo.lanes)) if lanes is None else set(lanes)
    bufs = [torch.full((n[l] + slack, 4), SENTINEL, device="cuda") if l in want else None for l in range(lvo.lanes)]
    torch.cuda.synchronize()
    got = lvo.map_cloud_batch_dev(which, [b.data_ptr() if b is not None else None for b in bufs], [len(b) if b is not None else 0 for b in bufs])
    assert got == n
    out = []
    for l, b in enumerate(bufs):
        if b is None:
            out.append(None)
            continue
        h = b.cpu().numpy()
        assert (h[n[l]:] == SENTINEL).all(), f"lane {l}: written beyond its {n[l]} points"
        out.append(h[:n[l]].copy())
    return out


def single(L, lvo, lane, which):
    """The single-lane route: lvo_map_cloud for which 0 / 1, the LVO_P_REGISTERED probe for which 2."""
    return lvo.map_cloud(lane, which) if which < 2 else lvo.probe(L.P_REGISTERED, lane)


def check_outputs(L, lvo, mapped):
    """Both forms of all three outputs against the single-lane route; `mapped[l]`: lane l mapped in the last step."""
    outs = {}
    for which in WHICH:
        host = lvo.map_cloud_batch(which)
        dev = dev_call(lvo, which)
        for l in range(lvo.lanes):
            assert same(host[l], dev[l]), f"which {which} lane {l}: host and device forms differ"
            if which < 2 or mapped[l]:
                ref = single(L, lvo, l, which)
                assert same(host[l], ref), f"which {which} lane {l}"
                if which == 2:
                    assert len(ref) > 1000
            else:
                assert len(host[l]) == 0, f"lane {l} did not map: registered n = 0"
        outs[which] = host
    return outs


@pytest.mark.parametrize("skip", [1, 2])
@pytest.mark.parametrize("distortion", [0, 2])
@pytest.mark.parametrize("graphs", [0, 1])
def test_parity_with_single_lane_routes(lvo_mod, sweeps, skip, distortion, graphs):
    L = lvo_mod
    seqs = list(range(8))
    lvo = make(L, 8, graphs, skip_frame=skip, distortion=distortion)
    one = make(L, 1, graphs, skip_frame=skip, distortion=distortion)   # lane 5's sequence alone
    for f in range(6):
        frame = [sweeps(s, f) for s in seqs]
        if f % 2:
            lvo.step_batch(frame)
            one.step_batch([frame[5]])
        else:
            dev_step(lvo, frame)
            dev_step(one, [frame[5]])
        mapped = f % skip == 0
        outs = check_outputs(L, lvo, [mapped] * 8)
        alone = check_outputs(L, one, [mapped])
        for which in WHICH:
            assert same(outs[which][5], alone[which][0]), f"frame {f} which {which}: 8-lane context vs 1-lane context"
        if f >= 2:
            assert all(len(outs[1][l]) >= len(outs[0][l]) > 1000 for l in range(8))
    lvo.close()
    one.close()


def test_lane_lifecycle(lvo_mod, sweeps):
    L = lvo_mod
    lvo = make(L, 4)
    for f in range(3):
        lvo.step_batch([sweeps(l, f) for l in range(4)])
    before = {w: lvo.map_cloud_batch(w) for w in (0, 1)}
    # idle lane 1: its map clouds are still returned (unchanged), its registered cloud is empty
    lvo.set_lane_active(1, False)
    lvo.step_batch([sweeps(l, 3) if l != 1 else None for l in range(4)])
    outs = check_outputs(L, lvo, [True, False, True, True])
    for w in (0, 1):
        assert same(outs[w][1], before[w][1]) and len(outs[w][1]) > 1000
    # reset lane 2: empty outputs at once
    lvo.lane_reset(2)
    for w in WHICH:
        assert [len(x) for x in lvo.map_cloud_batch(w)][2] == 0
        assert lvo.map_cloud_batch_dev(w, [None] * 4, [0] * 4)[2] == 0
    assert len(lvo.map_cloud_batch(2)[0]) > 1000            # the other lanes keep theirs
    # lane 3 loaded from lane 0: its map clouds at once, no registered cloud until its next mapping frame
    lvo.lane_load(3, lvo.lane_save(0))
    outs = {w: lvo.map_cloud_batch(w) for w in WHICH}
    for w in (0, 1):
        assert same(outs[w][3], outs[w][0]) and same(outs[w][3], lvo.map_cloud(3, w))
        assert same(dev_call(lvo, w)[3], outs[w][0])
    assert len(outs[2][3]) == 0 and len(outs[2][0]) > 1000
    lvo.set_lane_active(1, True)
    lvo.step_batch([sweeps(l, 4) for l in range(4)])
    check_outputs(L, lvo, [True] * 4)
    lvo.close()


def test_selection_and_size_query(lvo_mod, sweeps):
    L = lvo_mod
    lvo = make(L, 4)
    for f in range(3):
        lvo.step_batch([sweeps(l, f) for l in range(4)])
    for which in WHICH:
        full = lvo.map_cloud_batch(which)
        # all-NULL call: every n
        outs = (L.CloudOut * 4)(*[L.CloudOut(None, 0, 12345) for _ in range(4)])
        assert lvo.lib.lvo_map_cloud_batch(lvo.h, which, outs) == L.LVO_OK
        assert [o.n for o in outs] == [len(x) for x in full]
        assert lvo.map_cloud_batch_dev(which, [None] * 4, [0] * 4) == [len(x) for x in full]
        # lanes 0 and 2 requested
        got = lvo.map_cloud_batch(which, lanes=[0, 2])
        assert got[1] is None and got[3] is None and same(got[0], full[0]) and same(got[2], full[2])
        got = dev_call(lvo, which, lanes=[1, 3])
        assert got[0] is None and got[2] is None and same(got[1], full[1]) and same(got[3], full[3])
    lvo.close()


def raw_host(L, lvo, which, caps, sentinel_n=12345):
    """lvo_map_cloud_batch with sentinel-filled buffers of caps[l] points (None: NULL destination); returns (r, n, buffers)."""
    bufs = [np.full((max(c, 1), 4), SENTINEL, np.float32) if c is not None else None for c in caps]
    outs = (L.CloudOut * lvo.lanes)(*[L.CloudOut(b.ctypes.data if b is not None else None, c or 0, sentinel_n) for b, c in zip(bufs, caps)])
    r = lvo.lib.lvo_map_cloud_batch(lvo.h, which, outs)
    return r, [o.n for o in outs], bufs


def untouched(bufs):
    return all(b is None or (b == SENTINEL).all() for b in bufs)


def test_errors_leave_buffers_untouched_and_depth_keeps_registered(lvo_mod, sweeps):
    import torch
    L = lvo_mod
    lvo = make(L, 2)
    for f in range(3):
        lvo.step_batch([sweeps(l, f) for l in range(2)])
    n = {w: [len(x) for x in lvo.map_cloud_batch(w)] for w in WHICH}
    big = [[k + 5 for k in n[w]] for w in WHICH]
    d_buf = torch.full((max(max(big[w]) for w in WHICH), 4), SENTINEL, device="cuda")
    torch.cuda.synchronize()
    NS, VP = C.c_size_t * 2, C.c_void_p * 2

    def raw_dev(which, caps, null=None):
        n_out = NS(777, 777)
        args = [VP(d_buf.data_ptr(), d_buf.data_ptr()), NS(*caps), n_out]
        if null is not None:
            args[null] = None
        return lvo.lib.lvo_map_cloud_batch_dev(lvo.h, which, *args), list(n_out)

    def dev_untouched():
        return bool((d_buf == SENTINEL).all())

    # bad which, NULL arrays
    for which in (-1, 3):
        r, got_n, bufs = raw_host(L, lvo, which, big[0])
        assert r == L.LVO_E_BADARG and got_n == [12345, 12345] and untouched(bufs)
        assert raw_dev(which, big[0]) == (L.LVO_E_BADARG, [777, 777]) and dev_untouched()
    assert lvo.lib.lvo_map_cloud_batch(lvo.h, 0, None) == L.LVO_E_BADARG
    for k in range(3):
        r, got_n = raw_dev(0, big[0], null=k)
        assert r == L.LVO_E_BADARG and dev_untouched() and (k == 2 or got_n == [777, 777])
    # one selected lane one point too small: every n written, nothing copied
    for which in WHICH:
        caps = [n[which][0], n[which][1] - 1]
        r, got_n, bufs = raw_host(L, lvo, which, caps)
        assert r == L.LVO_E_CAPACITY and got_n == n[which] and untouched(bufs), which
        assert raw_dev(which, caps) == (L.LVO_E_CAPACITY, n[which]) and dev_untouched()
        # the short lane not selected: fine
        r, got_n, bufs = raw_host(L, lvo, which, [n[which][0], None])
        assert r == L.LVO_OK and got_n == n[which] and same(bufs[0][:n[which][0]], single(L, lvo, 0, which))
    # an *_async step in flight
    lvo.step_batch_async([sweeps(l, 3) for l in range(2)])
    for which in WHICH:
        r, got_n, bufs = raw_host(L, lvo, which, big[which])
        assert r == L.LVO_E_STATE and got_n == [12345, 12345] and untouched(bufs)
        assert raw_dev(which, big[which]) == (L.LVO_E_STATE, [777, 777]) and dev_untouched()
    lvo.wait()
    check_outputs(L, lvo, [True, True])
    # the single depth call runs in its own arena: the registered clouds stay available, bit for bit
    pts = sweeps(0, 3)
    before = lvo.map_cloud_batch(2)
    lvo.depth_associate(pts, np.zeros((4, 2), np.float32))
    assert all(len(b) > 1000 and same(a, b) for a, b in zip(lvo.map_cloud_batch(2), before))
    assert all(same(a, b) for a, b in zip(dev_call(lvo, 2), before))
    # which 2 after the two calls that overwrite the registered clouds; the next step makes it valid again
    one = L.Lvo(lanes=1, **CAPS)
    ex = one.extract_features(pts)[1]
    one.close()
    overwriters = {
        "knn": lambda: lvo.knn(pts[:5000], pts[:100], 5, 1.0),
        "scan_to_map": lambda: lvo.scan_to_map(ex["less_sharp"], ex["less_flat"], ex["full"], np.array([0, 0, 0, 1, 0, 0, 0.0]), want_registered=True),
    }
    for f, (name, call) in enumerate(overwriters.items()):
        call()
        r, got_n, bufs = raw_host(L, lvo, 2, big[2])
        assert r == L.LVO_E_STATE and got_n == [12345, 12345] and untouched(bufs), name
        assert b"registered" in lvo.lib.lvo_last_error(lvo.h)
        assert raw_dev(2, big[2]) == (L.LVO_E_STATE, [777, 777]) and dev_untouched(), name
        for which in (0, 1):   # the map clouds are not affected
            assert all(same(a, lvo.map_cloud(l, which)) for l, a in enumerate(lvo.map_cloud_batch(which)))
        lvo.step_batch([sweeps(l, 4 + f) for l in range(2)])
        check_outputs(L, lvo, [True, True])
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
def test_no_effect_on_pipeline(lvo_mod, sweeps, skip, graphs):
    L = lvo_mod
    ctx = [make(L, 2, graphs, skip_frame=skip) for _ in range(2)]   # ctx[0] fetches every output between its steps, ctx[1] does not
    frames = [[sweeps(lane, f) for lane in range(2)] for f in range(11)]
    for f in range(10):
        outs = []
        for i, c in enumerate(ctx):
            r = c.step_batch_pipelined(frames[f], frames[f + 1]) if f < 6 else dev_step(c, frames[f])
            launches = c.timings().kernel_launches
            if i == 0:   # all three outputs in both forms, checked against the single-lane routes, after pipelined and device steps
                check_outputs(L, c, [f % skip == 0] * 2)
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


def test_launch_count_is_independent_of_lanes(lvo_mod, sweeps):
    L = lvo_mod
    counts = set()
    for lanes in (1, 8, 32):
        lvo = make(L, lanes)
        for f in range(2):
            dev_step(lvo, [sweeps(l % 8, f) for l in range(lanes)])
        for which in WHICH:
            lvo.map_cloud_batch(which)
            counts.add(("host", which, lvo.timings().kernel_launches))
            dev_call(lvo, which)
            counts.add(("dev", which, lvo.timings().kernel_launches))
        lvo.close()
    assert counts == {(form, w, 1 if w == 2 else 2) for form in ("host", "dev") for w in WHICH}, counts


def test_arena_growth(lvo_mod, sweeps):
    L = lvo_mod
    lvo = make(L, 3)
    lvo.step_batch([sweeps(l, 0) for l in range(3)])

    def check(lanes):
        for which in WHICH:
            got = lvo.map_cloud_batch(which, lanes=lanes)
            for l in range(3):
                assert (got[l] is None) == (l not in lanes)
                if got[l] is not None:
                    assert same(got[l], single(L, lvo, l, which)), (which, l)

    check([0])                                             # first use: small
    for f in range(1, 4):
        lvo.step_batch([sweeps(l, f) for l in range(3)])
    check([0, 1, 2])                                       # larger maps, every lane: the point buffers grow
    check([1])                                             # smaller again
    assert len(lvo.map_cloud_batch(1)[2]) > 1000
    lvo.close()
    lvo = make(L, 1)                                       # the device is healthy after lvo_destroy of a grown arena
    lvo.step_batch([sweeps(0, 0)])
    check_outputs(L, lvo, [True])
    lvo.close()
