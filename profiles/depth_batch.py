"""Throughput of the batched camera-lidar depth association (lvo_depth_associate_batch / _dev) at the config-5 shape.

Every lane brings a seeded synthetic HDL-64 sweep (~119.4 k points; lane l: sequence l % 16, frame l // 16) and 1120 keypoints (uniform
over the image inside the 20 / 15 pixel borders, normalised with KITTI00_CAMERA).  For 8, 32 and 128 lanes it measures:
  - the device-resident form: CUDA events on the context's stream around --calls calls, after --warm warm-up calls;
  - the host form: host clock around each synchronous call (median);
  - the baseline: a loop of lvo_depth_associate over the same lanes in the same context (host clock around the loop, median).
It reports sweeps/s and keypoints/s, launches per call, the bytes the arena took (cudaMemGetInfo around the first call), and the
algorithmic bytes 16 N + 16 N_dc + 8 K (sweep read, depth cloud written, keypoints read; DESIGN §4) over the call time as a fraction
of 6554.2 GB/s.  That fraction is a whole-call figure, not a kernel's.  A torch.profiler run of its own then gives the per-kernel
device times of the device form at the largest lane count.  Results of the batched forms are checked against the baseline, bitwise.
The GPU's name and power limit are read in the same run.

Usage:  python profiles/depth_batch.py [--lanes 8 32 128] [--warm 5] [--calls 50] [--out FILE.json]"""
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
PEAK_GBS = 6554.2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, nargs="+", default=[8, 32, 128])
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--loops", type=int, default=5, help="timed loops of the single-call baseline")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle_py import Synth
    L = load_pkg()
    cam = L.KITTI00_CAMERA
    synth = Synth()
    top = max(args.lanes)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        sweeps = list(ex.map(lambda l: synth.sweep(64, l % 16, l // 16)[0], range(top)))
    rng = np.random.default_rng(5)
    kps = []
    for _ in range(top):
        px = np.stack([rng.uniform(20, cam["width"] - 20, 1120), rng.uniform(15, cam["height"] - 15, 1120)], 1)
        kps.append(np.stack([(px[:, 0] - cam["cx"]) / cam["fx"], (px[:, 1] - cam["cy"]) / cam["fy"]], 1).astype(np.float32))
    d_sw = [torch.from_numpy(s).cuda() for s in sweeps]
    d_kp = [torch.from_numpy(k).cuda() for k in kps]
    d_depth = [torch.empty(1120, device="cuda") for _ in range(top)]
    d_valid = [torch.empty(1120, dtype=torch.int32, device="cuda") for _ in range(top)]
    d_nn = [torch.empty((1120, 3), dtype=torch.int32, device="cuda") for _ in range(top)]
    torch.cuda.synchronize()
    res = {"gpu": gpu_identity(torch), "shape": {"points_per_sweep_mean": float(np.mean([len(s) for s in sweeps[:top]])), "keypoints_per_lane": 1120},
           "peak_gbs": PEAK_GBS, "runs": []}
    for lanes in args.lanes:
        ctx = L.Lvo(lanes=lanes, max_points=131072, max_map_corner=1 << 16, max_map_surf=1 << 17, debug_probes=0)
        st = torch.cuda.Stream()
        ctx.set_stream(st.cuda_stream)
        sw, kp = sweeps[:lanes], kps[:lanes]
        N = sum(len(s) for s in sw)
        K = 1120 * lanes
        # baseline: the single call, lane after lane (also the reference results and depth-cloud sizes)
        base, n_dc = [], 0
        for l in range(lanes):
            dc, d, v, nn = ctx.depth_associate(sw[l], kp[l])
            base.append((d.copy(), v.copy(), nn.copy()))
            n_dc += len(dc)
        single_launches = ctx.timings().kernel_launches
        loop_s = []
        for _ in range(args.loops):
            t0 = time.perf_counter()
            for l in range(lanes):
                ctx.depth_associate(sw[l], kp[l])
            loop_s.append(time.perf_counter() - t0)
        # device form
        ptrs = lambda ts: [t.data_ptr() for t in ts[:lanes]]
        dev_args = (ptrs(d_sw), [len(s) for s in sw], ptrs(d_kp), [1120] * lanes, ptrs(d_depth), ptrs(d_valid), ptrs(d_nn))
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        ctx.depth_associate_batch_dev(*dev_args)
        free1 = torch.cuda.mem_get_info()[0]
        dev_launches = ctx.timings().kernel_launches
        ok_dev = all(np.array_equal(d_depth[l].cpu().numpy().view(np.uint32), base[l][0].view(np.uint32)) and
                     np.array_equal(d_valid[l].cpu().numpy(), base[l][1]) and np.array_equal(d_nn[l].cpu().numpy(), base[l][2]) for l in range(lanes))
        for _ in range(args.warm):
            ctx.depth_associate_batch_dev(*dev_args)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(args.calls):
            ctx.depth_associate_batch_dev(*dev_args)
        e1.record(st)
        e1.synchronize()
        dev_s = e0.elapsed_time(e1) / 1e3 / args.calls
        # host form (its arena growth happens in the first call)
        free2 = torch.cuda.mem_get_info()[0]
        out = ctx.depth_associate_batch(sw, kp)
        free3 = torch.cuda.mem_get_info()[0]
        host_launches = ctx.timings().kernel_launches
        ok_host = all(np.array_equal(out[l][0].view(np.uint32), base[l][0].view(np.uint32)) and np.array_equal(out[l][1], base[l][1]) and
                      np.array_equal(out[l][2], base[l][2]) for l in range(lanes))
        for _ in range(args.warm):
            ctx.depth_associate_batch(sw, kp)
        host_s = []
        for _ in range(args.calls):
            t0 = time.perf_counter()
            ctx.depth_associate_batch(sw, kp)
            host_s.append(time.perf_counter() - t0)
        alg = 16 * N + 16 * n_dc + 8 * K
        t_loop, t_host = statistics.median(loop_s), statistics.median(host_s)
        run = {"lanes": lanes, "points": N, "depth_cloud_points": n_dc, "keypoints": K, "valid_fraction": float(np.mean([b[1].mean() for b in base])),
               "bitwise_equal_to_single_call": {"device_form": ok_dev, "host_form": ok_host},
               "launches_per_call": {"device_form": dev_launches, "host_form": host_launches, "single_call": single_launches},
               "arena_bytes_cudaMemGetInfo": {"device_form_first_call": free0 - free1, "host_form_growth": free2 - free3},
               "algorithmic_bytes": alg}
        for name, t in (("device_form", dev_s), ("host_form", t_host), ("single_call_loop", t_loop)):
            run[name] = {"ms_per_call": t * 1e3, "sweeps_per_s": lanes / t, "keypoints_per_s": K / t,
                         "whole_call_fraction_of_peak_bw": alg / t / (PEAK_GBS * 1e9)}
        run["device_form_over_single_call_loop"] = t_loop / dev_s
        run["host_form_over_single_call_loop"] = t_loop / t_host
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
        if args.out:
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
        if lanes == top:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(10):
                    ctx.depth_associate_batch_dev(*dev_args)
                torch.cuda.synchronize()
            kern = {}
            for e in prof.key_averages():
                if e.device_type.name == "CUDA" and e.count:
                    kern[e.key] = {"us_per_call": e.device_time_total / 10, "launches_per_call": e.count / 10}
            res["kernels_device_form_lanes%d" % top] = dict(sorted(kern.items(), key=lambda kv: -kv[1]["us_per_call"]))
            print(json.dumps(res["kernels_device_form_lanes%d" % top]), flush=True)
        ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
