"""Per-lane sensor settings (lvo_lane_configure): one mixed context against one dedicated context per sensor model.

  1. A 128-lane context with n_scans 64 whose lanes 0-63 run HDL-64 sequences with the HDL-64 launch values and whose lanes 64-127 are
     configured with the VLP-16 launch values and run VLP-16 sequences, against two 64-lane contexts, one created with each model's
     values, on streams of their own: both are enqueued (lvo_step_batch_dev_async) before either is waited for.  Lane l of each half
     runs seeded synthetic sequence (l % 64) // 8 of its model from frame l % 8 (bench.py's lane plan), through lvo_step_batch_dev,
     max_points 131072, maps of 256 k corner / 512 k surf points, debug_probes 0, plain launches.  Step time is a host clock around
     the synchronous call (mixed) or around both enqueues and both waits (dedicated pair); the two set-ups alternate step by step, and
     their poses are compared bit for bit.
  2. Device memory from cudaMemGetInfo before and after creating each context, and the memory of a 64-lane
     context with n_scans 64 against one with n_scans 16: what a VLP-16 lane costs more in a context sized for the HDL-64.
  3. Host time of lvo_lane_configure (a synchronous call: it resets the lane and uploads its settings) per lane of the mixed context.
The GPU's name and power limit are read in the same run.

Usage:  python profiles/lane_config.py [--warm 20] [--steps 20] [--out FILE.json]"""
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

HDL64 = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, skip_frame=1)   # launch/aloam_velodyne_HDL_64.launch
VLP16 = dict(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4, skip_frame=1)   # launch/aloam_velodyne_VLP_16.launch


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
    half, per_seq = 64, 8
    plan = [(l // per_seq, l % per_seq) for l in range(half)]   # (sequence, first frame) of lane l of each half
    frames = per_seq + args.warm + args.steps + 1
    synth = Synth()
    jobs = [(m, s, f) for m in (64, 16) for s in range(half // per_seq) for f in range(frames)]
    dev = {}
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        for j, h in zip(jobs, ex.map(lambda j: synth.sweep(j[0], j[1], j[2])[0], jobs)):
            dev[j] = torch.from_numpy(h).cuda()
    torch.cuda.synchronize()
    caps = dict(max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 19, debug_probes=0)

    def free_bytes():
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info()[0]

    def new_ctx(lanes, **cfg):
        before = free_bytes()
        c = L.Lvo(lanes=lanes, **caps, **cfg)
        c.set_option(L.LVO_OPT_GRAPHS, 0)
        c.set_option(L.LVO_OPT_STAGE_TIMING, 0)
        return c, before - free_bytes()

    def inputs(models, k):
        """Device pointers and counts of step k for lanes running `models` (one entry per lane)."""
        ts = [dev[(m, plan[l % half][0], plan[l % half][1] + k)] for l, m in enumerate(models)]
        return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts]), (C.c_size_t * len(ts))(*[t.shape[0] for t in ts])

    out = {"config": {**caps, "lanes_per_model": half, "warm_steps": args.warm, "timed_steps": args.steps, "entry": "lvo_step_batch_dev",
                      "graphs": 0, "hdl64": HDL64, "vlp16": VLP16}}
    out.update(gpu_identity(torch))

    # 1 + 2: the mixed context and the two dedicated ones, all alive at once
    mixed, mem_mixed = new_ctx(2 * half, **HDL64)
    for l in range(half, 2 * half):
        mixed.lane_configure(l, **VLP16)
    ded64, mem64 = new_ctx(half, **HDL64)
    ded16, mem16 = new_ctx(half, **VLP16)
    models_mixed = [64] * half + [16] * half
    po = lambda n: ((L.Pose * n)(), (L.Pose * n)())

    def step_mixed(k):
        p, n = inputs(models_mixed, k)
        a, b = po(2 * half)
        t0 = time.perf_counter()
        st = mixed.lib.lvo_step_batch_dev(mixed.h, p, n, a, b)
        dt = (time.perf_counter() - t0) * 1e3
        assert st >= 0, mixed.lib.lvo_last_error(mixed.h)
        return dt, np.frombuffer(a, np.float64).copy(), np.frombuffer(b, np.float64).copy()

    def step_pair(k):
        (p64, n64), (p16, n16) = inputs([64] * half, k), inputs([16] * half, k)
        a64, b64 = po(half)
        a16, b16 = po(half)
        t0 = time.perf_counter()
        assert ded64.lib.lvo_step_batch_dev_async(ded64.h, p64, n64) == 0
        assert ded16.lib.lvo_step_batch_dev_async(ded16.h, p16, n16) == 0
        r64 = ded64.lib.lvo_wait(ded64.h, a64, b64)
        r16 = ded16.lib.lvo_wait(ded16.h, a16, b16)
        dt = (time.perf_counter() - t0) * 1e3
        assert r64 >= 0 and r16 >= 0, (r64, r16)
        cat = lambda x, y: np.concatenate([np.frombuffer(x, np.float64), np.frombuffer(y, np.float64)])
        return dt, cat(a64, a16), cat(b64, b16)

    t_mixed, t_pair, same = [], [], True
    for k in range(args.warm + args.steps):
        tm, om, mm = step_mixed(k)
        tp, op, mp = step_pair(k)
        same = same and np.array_equal(om, op) and np.array_equal(mm, mp)
        if k >= args.warm:
            t_mixed.append(tm); t_pair.append(tp)
    out["step"] = {"mixed_128_lane_context_ms": stats_ms(t_mixed), "two_64_lane_contexts_concurrent_ms": stats_ms(t_pair),
                   "mixed_vs_pair_step_time": statistics.median(t_mixed) / statistics.median(t_pair),
                   "poses_bitwise_equal": bool(same)}
    print(json.dumps(out["step"]), flush=True)

    # 3: lvo_lane_configure per lane (the VLP-16 half again: each call resets its lane)
    t_cfg = []
    for l in range(half, 2 * half):
        t0 = time.perf_counter()
        mixed.lane_configure(l, **VLP16)
        t_cfg.append((time.perf_counter() - t0) * 1e3)
    out["lane_configure_ms"] = stats_ms(t_cfg)
    print(json.dumps(out["lane_configure_ms"]), flush=True)
    for c in (mixed, ded64, ded16):
        c.close()
    # memory of the n_scans a context is sized for: 64 lanes at n_scans 64 (what a VLP-16 lane of a mixed context holds) and at 16
    wide, mem_wide = new_ctx(half, **HDL64)
    wide.close()
    narrow, mem_narrow = new_ctx(half, **VLP16)
    narrow.close()
    out["device_memory_bytes"] = {"mixed_128_lanes": mem_mixed, "dedicated_hdl64_64_lanes": mem64, "dedicated_vlp16_64_lanes": mem16,
                                  "dedicated_pair": mem64 + mem16, "mixed_minus_pair": mem_mixed - (mem64 + mem16),
                                  "repeat_64_lanes_n_scans_64": mem_wide,
                                  "repeat_64_lanes_n_scans_16": mem_narrow,
                                  "per_vlp16_lane_in_a_64_beam_context_extra": (mem_wide - mem_narrow) / half}
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
