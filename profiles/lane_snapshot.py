"""Cost of lane snapshots (lvo_lane_save / lvo_lane_load) at bench.py's configuration.

128 lanes, max_points 131072, maps of 256 k corner / 512 k surf points, debug_probes 0, plain launches; lane l runs seeded synthetic
HDL-64 sequence l // 8 from its frame l % 8 (bench.py's lane plan), through lvo_step_batch_dev.  After 100 steps:
  1. snapshot bytes per lane;
  2. host time of lvo_lane_save / lvo_lane_load per lane, to and from pageable host memory and device memory of the same GPU (the
     loads put each lane's own snapshot back, which leaves the state as it was; every call returns after its copies are done);
  3. checkpoint of all 128 lanes to host memory, restore into a new context, and that context's first step (which rebuilds the
     odometry grids once) against its following steps; the restored context's poses are compared with the original's;
  4. consolidation: the context and a second one built the same way (the same lane plan, so both do the same kind of work) with lanes
     64-127 idle; the step time of both against the time of one context after the second's 64 active lanes have been moved into the
     first's idle lanes through a device buffer, and the time the moves took.
Step times are host clocks around the synchronous lvo_step_batch_dev call, plus the device time of its stages (lvo_timings) where it
applies.  The GPU's name and power limit are read in the same run.

Usage:  python profiles/lane_snapshot.py [--warm 100] [--steps 10] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import sys
import time
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from lane_lifecycle import ROOT, gpu_identity, load_pkg  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))


def stats_ms(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=128)
    ap.add_argument("--warm", type=int, default=100)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle_py import Synth
    L = load_pkg()
    lanes, n_seq = args.lanes, 16
    per_seq = lanes // n_seq
    half = lanes // 2
    plan = [(l // per_seq, l % per_seq) for l in range(lanes)]
    R = 6                                                                 # steps after the restore
    frames = per_seq + args.warm + R + 2 * (2 + args.steps) + 2
    synth = Synth()
    jobs = [(s, f) for s in range(n_seq) for f in range(frames)]
    dev = {}
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        for j, h in zip(jobs, ex.map(lambda j: synth.sweep(64, j[0], j[1])[0], jobs)):
            dev[j] = torch.from_numpy(h).cuda()
    torch.cuda.synchronize()
    cfg = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=lanes, max_points=131072, max_map_corner=1 << 18,
               max_map_surf=1 << 19, debug_probes=0)

    def new_ctx():
        c = L.Lvo(**cfg)
        c.set_option(L.LVO_OPT_GRAPHS, 0)
        c.set_option(L.LVO_OPT_STAGE_TIMING, 0)
        return c

    def step(ctx, frame, active):
        """One step; returns (host ms, device stage ms, odometry rows, mapping rows)."""
        ptrs, ns = [], []
        for l in range(lanes):
            if active[l]:
                t = dev[(plan[l][0], plan[l][1] + frame[l])]
                ptrs.append(t.data_ptr()); ns.append(t.shape[0])
                frame[l] += 1
            else:
                ptrs.append(None); ns.append(None)
        t0 = time.perf_counter()
        st, o, m = ctx.step_batch_dev(ptrs, ns)
        host = (time.perf_counter() - t0) * 1e3
        assert st >= 0, st
        t = ctx.timings()
        return host, t.extract_ms + t.odometry_ms + t.mapping_ms, o, m

    out = {"config": {**cfg, "warm_steps": args.warm, "timed_steps": args.steps, "entry": "lvo_step_batch_dev", "graphs": 0}}
    out.update(gpu_identity(torch))
    all_on = [True] * lanes
    a = new_ctx()
    fa = [0] * lanes
    for _ in range(args.warm):
        step(a, fa, all_on)
    lib = a.lib

    # 1 + 2: sizes, per-lane save / load to and from host and device memory
    sizes = []
    for l in range(lanes):
        n = L.C.c_size_t(0)
        assert lib.lvo_lane_save(a.h, l, None, 0, L.C.byref(n)) == L.LVO_E_CAPACITY
        sizes.append(n.value)
    host_bufs = [np.empty(n, np.uint8) for n in sizes]
    for b in host_bufs:
        b.fill(0)                                                          # fault the pages in before timing
    offs = np.concatenate([[0], np.cumsum(sizes)]).tolist()
    dbuf = torch.empty(offs[-1], dtype=torch.uint8, device="cuda")
    n = L.C.c_size_t(0)
    t_save_h, t_save_d, t_load_h, t_load_d = [], [], [], []
    for l in range(lanes):
        t0 = time.perf_counter()
        assert lib.lvo_lane_save(a.h, l, host_bufs[l].ctypes.data, sizes[l], L.C.byref(n)) == 0
        t_save_h.append((time.perf_counter() - t0) * 1e3)
    for l in range(lanes):
        t0 = time.perf_counter()
        assert lib.lvo_lane_save(a.h, l, L.C.c_void_p(dbuf.data_ptr() + offs[l]), sizes[l], L.C.byref(n)) == 0
        t_save_d.append((time.perf_counter() - t0) * 1e3)
    assert all(np.array_equal(dbuf[offs[l]:offs[l + 1]].cpu().numpy(), host_bufs[l]) for l in range(lanes))
    for l in range(lanes):
        t0 = time.perf_counter()
        assert lib.lvo_lane_load(a.h, l, host_bufs[l].ctypes.data, sizes[l]) == 0
        t_load_h.append((time.perf_counter() - t0) * 1e3)
    for l in range(lanes):
        t0 = time.perf_counter()
        assert lib.lvo_lane_load(a.h, l, L.C.c_void_p(dbuf.data_ptr() + offs[l]), sizes[l]) == 0
        t_load_d.append((time.perf_counter() - t0) * 1e3)
    out["snapshot_bytes"] = {"min": min(sizes), "median": statistics.median(sizes), "max": max(sizes), "total": offs[-1]}
    out["per_lane_ms"] = {"save_to_host": stats_ms(t_save_h), "save_to_device": stats_ms(t_save_d),
                          "load_from_host": stats_ms(t_load_h), "load_from_device": stats_ms(t_load_d)}
    print(json.dumps({k: out[k] for k in ("snapshot_bytes", "per_lane_ms")}), flush=True)

    # 3: checkpoint all lanes to host, restore into a new context; a's own first step after the reloads above also rebuilds its grids
    t0 = time.perf_counter()
    snaps = [a.lane_save(l) for l in range(lanes)]
    ckpt_ms = (time.perf_counter() - t0) * 1e3
    b = new_ctx()
    t0 = time.perf_counter()
    for l in range(lanes):
        b.lane_load(l, snaps[l])
    restore_ms = (time.perf_counter() - t0) * 1e3
    fb = list(fa)
    same, b_host, b_dev = True, [], []
    for k in range(R):
        _, _, ao, am = step(a, fa, all_on)
        h, d, bo, bm = step(b, fb, all_on)
        b_host.append(h); b_dev.append(d)
        same = same and np.array_equal(ao, bo) and np.array_equal(am, bm)
    b.close()
    out["checkpoint_restore"] = {"checkpoint_all_lanes_to_host_ms": ckpt_ms, "restore_all_lanes_from_host_ms": restore_ms,
                                 "first_step_after_restore_host_ms": b_host[0], "later_steps_host_ms": stats_ms(b_host[1:]),
                                 "first_step_extra_host_ms": b_host[0] - statistics.median(b_host[1:]),
                                 "first_step_device_stage_ms": b_dev[0], "later_steps_device_stage_ms": stats_ms(b_dev[1:]),
                                 "restored_poses_bitwise_equal": bool(same)}
    print(json.dumps(out["checkpoint_restore"]), flush=True)

    # 4: consolidation
    y = new_ctx()
    fy = [0] * lanes
    for _ in range(args.warm):
        step(y, fy, all_on)
    half_on = [l < half for l in range(lanes)]
    for ctx in (a, y):
        for l in range(half, lanes):
            ctx.set_lane_active(l, False)
    two_host, two_dev = [], []
    for k in range(2 + args.steps):
        ha, da, _, _ = step(a, fa, half_on)
        hy, dy, _, _ = step(y, fy, half_on)
        if k >= 2:
            two_host.append(ha + hy); two_dev.append(da + dy)
    need = []
    for j in range(half):
        assert lib.lvo_lane_save(y.h, j, None, 0, L.C.byref(n)) == L.LVO_E_CAPACITY
        need.append(n.value)
    moff = np.concatenate([[0], np.cumsum(need)]).tolist()
    mbuf = torch.empty(moff[-1], dtype=torch.uint8, device="cuda")
    t0 = time.perf_counter()
    for j in range(half):
        assert lib.lvo_lane_save(y.h, j, L.C.c_void_p(mbuf.data_ptr() + moff[j]), need[j], L.C.byref(n)) == 0
        assert lib.lvo_lane_load(a.h, half + j, L.C.c_void_p(mbuf.data_ptr() + moff[j]), need[j]) == 0
        fa[half + j] = fy[j]
    move_ms = (time.perf_counter() - t0) * 1e3
    for l in range(half, lanes):
        a.set_lane_active(l, True)
    one_host, one_dev = [], []
    for k in range(2 + args.steps):
        h, d, _, _ = step(a, fa, all_on)
        if k >= 2:
            one_host.append(h); one_dev.append(d)
    y.close(); a.close()
    out["consolidation"] = {"active_lanes": half, "two_contexts_step_host_ms": stats_ms(two_host), "two_contexts_step_device_stage_ms": stats_ms(two_dev),
                            "one_context_step_host_ms": stats_ms(one_host), "one_context_step_device_stage_ms": stats_ms(one_dev),
                            "move_lanes": half, "move_bytes": moff[-1], "move_all_lanes_ms": move_ms,
                            "one_vs_two_step_time": statistics.median(one_host) / statistics.median(two_host)}
    print(json.dumps(out["consolidation"]), flush=True)
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
