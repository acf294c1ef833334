"""Cost of localising lanes (lvo_set_lane_map_update off) in the batched device-resident pipeline (lvo_step_batch_dev).

One 128-lane context with bench.py's configuration and lane plan (16 seeded synthetic HDL-64 sequences, 8 lanes each, entering their
sequence one frame apart), max_points 131072, maps of 256 k corner / 512 k surf points, debug_probes 0, plain launches.  `--warm`
steps with every lane mapping grow the maps.  Then, for each of `--steps` frames, three set-ups run the same frame from the same
state: 0, 64 (the odd lanes) and 128 lanes with map updates off.  Before each set-up every lane is restored from a device-memory
snapshot of that state (lvo_lane_load); the all-updating set-up's result is the state of the next frame.  The order of the set-ups
rotates from frame to frame.  Per set-up and frame:
  - step ms: host clock around the synchronous lvo_step_batch_dev, stage timing off;
  - map_add_points_ms / map_filter_ms ("add points time" / "filter time" of laserMapping.cpp:784 / :802) of a second run of the same
    step from the same state with the context's sub-stage events on;
  - the poses of the lanes with updates on, which must be bitwise equal across the set-ups.
The GPU's name and power limit are read in the same run.

Usage:  python profiles/map_fixed.py [--warm 20] [--steps 20] [--out FILE.json]"""
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
    ap.add_argument("--warm", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle_py import Synth
    L = load_pkg()
    C = L.C
    lanes, n_seq = 128, 16
    per_seq = lanes // n_seq
    plan = [(l // per_seq, l % per_seq) for l in range(lanes)]          # bench.lane_plan
    frames = per_seq + args.warm + args.steps
    synth = Synth()
    jobs = [(s, f) for s in range(n_seq) for f in range(frames)]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        host = list(ex.map(lambda j: synth.sweep(64, j[0], j[1])[0], jobs))
    dev = {j: torch.from_numpy(h).cuda() for j, h in zip(jobs, host)}
    torch.cuda.synchronize()
    ctx = L.Lvo(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=lanes, max_points=131072, max_map_corner=1 << 18,
                max_map_surf=1 << 19, debug_probes=0)
    ctx.set_option(L.LVO_OPT_GRAPHS, 0)
    ctx.set_option(L.LVO_OPT_STAGE_TIMING, 0)

    def step(k):
        ptrs = (C.c_void_p * lanes)(*[dev[(s, f + k)].data_ptr() for s, f in plan])
        ns = (C.c_size_t * lanes)(*[dev[(s, f + k)].shape[0] for s, f in plan])
        po, pm = (L.Pose * lanes)(), (L.Pose * lanes)()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ctx.lib.lvo_step_batch_dev(ctx.h, ptrs, ns, po, pm)
        ms = (time.perf_counter() - t0) * 1e3
        assert r >= 0, (r, ctx.lib.lvo_last_error(ctx.h))
        return ms, np.frombuffer(pm, np.float64).reshape(lanes, 7).copy()

    for k in range(args.warm):
        step(k)
    # device-memory snapshots of every lane (lvo_lane_save / lvo_lane_load of device memory)
    snap_cap = 64 << 20
    snap = torch.empty(lanes * snap_cap, dtype=torch.uint8, device="cuda")
    snap_n = [0] * lanes

    def save():
        for l in range(lanes):
            snap_n[l] = ctx.lane_save_dev(l, snap.data_ptr() + l * snap_cap, snap_cap)

    def load():
        for l in range(lanes):
            ctx.lane_load_dev(l, snap.data_ptr() + l * snap_cap, snap_n[l])

    setups = {0: [], 64: [l for l in range(lanes) if l % 2], 128: list(range(lanes))}
    res = {n: {"step_ms": [], "map_add_points_ms": [], "map_filter_ms": [], "map_corner_total": [], "map_surf_total": []} for n in setups}
    mismatches = 0
    for j in range(args.steps):
        k = args.warm + j
        save()
        order = list(setups)[j % 3:] + list(setups)[:j % 3]
        poses, next_state = {}, None
        for n in order:
            for l in range(lanes):
                ctx.set_lane_map_update(l, l not in setups[n])
            load()
            ms, pm = step(k)
            poses[n] = pm
            res[n]["step_ms"].append(ms)
            res[n]["map_corner_total"].append(sum(ctx.stats(l).map_corner_total for l in range(lanes)))
            res[n]["map_surf_total"].append(sum(ctx.stats(l).map_surf_total for l in range(lanes)))
            load()
            ctx.set_option(L.LVO_OPT_STAGE_TIMING, 1)
            step(k)
            ctx.set_option(L.LVO_OPT_STAGE_TIMING, 0)
            t = ctx.timings()
            res[n]["map_add_points_ms"].append(float(t.map_add_points_ms))
            res[n]["map_filter_ms"].append(float(t.map_filter_ms))
            if n == 0:   # the state of the next frame: every lane mapping
                next_state = torch.empty_like(snap)
                next_n = [ctx.lane_save_dev(l, next_state.data_ptr() + l * snap_cap, snap_cap) for l in range(lanes)]
        for n in setups:
            on = [l for l in range(lanes) if l not in setups[n]]
            mismatches += int(not np.array_equal(poses[n][on], poses[0][on]))
        snap.copy_(next_state)
        snap_n[:] = next_n
        del next_state
        load()
    for l in range(lanes):
        ctx.set_lane_map_update(l, True)
    out = {"config": {"lanes": lanes, "sequences": n_seq, "warm_steps": args.warm, "timed_steps": args.steps, "entry": "lvo_step_batch_dev",
                      "max_points": 131072, "map_caps": [1 << 18, 1 << 19], "graphs": 0, "fixed_lanes_64": "odd lanes"},
           "update_on_poses_bitwise_equal_across_setups": mismatches == 0, "pose_mismatching_steps": mismatches}
    out.update(gpu_identity(torch))
    out["setups"] = {}
    for n, r in res.items():
        out["setups"][f"{n}_fixed"] = {"step_ms": stats_ms(r["step_ms"]), "map_add_points_ms": stats_ms(r["map_add_points_ms"]),
                                       "map_filter_ms": stats_ms(r["map_filter_ms"]),
                                       "map_points_all_lanes_median": statistics.median([a + b for a, b in zip(r["map_corner_total"], r["map_surf_total"])]),
                                       "raw_step_ms": r["step_ms"]}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(s)
    ctx.close()


if __name__ == "__main__":
    main()
