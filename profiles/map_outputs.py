"""Cost of the batched map outputs (lvo_map_cloud_batch / _dev) against the single-lane routes.

For 8, 32 and 128 lanes a context (max_points 131072, the map capacities of bench.py: max_map_corner 2^18 and max_map_surf 2^19,
debug_probes 0, skip_frame 1) steps 20 seeded
synthetic HDL-64 sweeps per lane through lvo_step_batch_dev (lane l: sequence l % 16, frames 0 .. 19), so that the maps have grown.
Then, for each `which` (0 surround, 1 whole map, 2 registered) and form:
  - the device form: CUDA events on the context's stream around --calls calls into per-lane device buffers, after --warm calls;
  - the host form: host clock around each synchronous call into per-lane numpy buffers (median);
  - the baseline: a per-lane loop of lvo_map_cloud (which 0 / 1) or lvo_probe_fetch(LVO_P_REGISTERED) (which 2), host clock
    around the loop (median);
  - the other host-form strategy, which the library does not use: the device form gathers every lane's cloud back to back into
    one device buffer, ONE copy brings it to pinned host memory, and a host memcpy scatters it into the per-lane numpy buffers
    (host clock, median).  The library's host form instead copies each lane's cloud into the caller's buffer with one
    cudaMemcpyAsync; both move each point over PCIe once.
It reports ms per call, the point bytes delivered (16 bytes per point) over that time, launches per call, and the arena's device
bytes (cudaMemGetInfo around the first call of each form).  Every output of both forms is checked bitwise against its single-lane
counterpart in the same run.  The GPU's name and power limit are read in the same run.

Usage:  python profiles/map_outputs.py [--lanes 8 32 128] [--frames 20] [--warm 3] [--calls 20] [--out FILE.json]"""
import argparse
import ctypes as C
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, nargs="+", default=[8, 32, 128])
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--warm", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--loops", type=int, default=3, help="timed loops of the single-lane baselines")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle_py import Synth
    L = load_pkg()
    synth = Synth()
    nseq = min(16, max(args.lanes))
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        sweeps = {(s, f): p for (s, f), p in zip([(s, f) for s in range(nseq) for f in range(args.frames)],
                                                 ex.map(lambda sf: synth.sweep(64, sf[0], sf[1])[0], [(s, f) for s in range(nseq) for f in range(args.frames)]))}
    d_sweeps = {k: torch.from_numpy(v).cuda() for k, v in sweeps.items()}
    torch.cuda.synchronize()
    res = {"gpu": gpu_identity(torch), "library": os.environ.get("LVO_LIB_PATH") or "liblvo.so", "frames": args.frames, "runs": []}
    for lanes in args.lanes:
        ctx = L.Lvo(lanes=lanes, max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 19, debug_probes=0, skip_frame=1)
        st = torch.cuda.Stream()
        ctx.set_stream(st.cuda_stream)
        for f in range(args.frames):
            ctx.step_batch_dev([d_sweeps[(l % nseq, f)].data_ptr() for l in range(lanes)], [len(sweeps[(l % nseq, f)]) for l in range(lanes)])
        step_launches = ctx.timings().kernel_launches
        run = {"lanes": lanes, "step_launches_last_frame": step_launches, "outputs": {}}
        for which in (0, 1, 2):
            name = ["surround", "whole_map", "registered"][which]
            # single-lane route: reference results and the baseline
            if which < 2:
                outs = [L.CloudOut(None, 0, 0) for _ in range(lanes)]
                for l in range(lanes):   # size query of the single call: LVO_E_CAPACITY with n
                    ctx.lib.lvo_map_cloud(ctx.h, l, which, C.byref(outs[l]))
                bufs = [np.empty((max(o.n, 1), 4), np.float32) for o in outs]
                outs = [L.CloudOut(b.ctypes.data, len(b), 0) for b in bufs]
                single = lambda: [ctx.lib.lvo_map_cloud(ctx.h, l, which, C.byref(outs[l])) for l in range(lanes)]
                single()
                ref = [bufs[l][:outs[l].n].copy() for l in range(lanes)]
            else:
                ref = [ctx.probe(L.P_REGISTERED, l) for l in range(lanes)]
                bufs = [np.empty((len(r), 4), np.float32) for r in ref]
                nb = C.c_size_t(0)
                single = lambda: [ctx.lib.lvo_probe_fetch(ctx.h, l, L.P_REGISTERED, bufs[l].ctypes.data, bufs[l].nbytes, C.byref(nb)) for l in range(lanes)]
            loop_s = []
            for _ in range(args.loops):
                t0 = time.perf_counter()
                single()
                loop_s.append(time.perf_counter() - t0)
            n = [len(r) for r in ref]
            pts_bytes = 16 * sum(n)
            # device form
            d_out = [torch.empty((max(k, 1), 4), device="cuda") for k in n]
            torch.cuda.synchronize()
            ptrs, caps = [t.data_ptr() for t in d_out], [len(t) for t in d_out]
            free0 = torch.cuda.mem_get_info()[0]
            ctx.map_cloud_batch_dev(which, ptrs, caps)
            free1 = torch.cuda.mem_get_info()[0]
            dev_launches = ctx.timings().kernel_launches
            ok_dev = all(np.array_equal(d_out[l][:n[l]].cpu().numpy().view(np.uint32), ref[l].view(np.uint32)) for l in range(lanes))
            for _ in range(args.warm):
                ctx.map_cloud_batch_dev(which, ptrs, caps)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(args.calls):
                ctx.map_cloud_batch_dev(which, ptrs, caps)
            e1.record(st)
            e1.synchronize()
            dev_s = e0.elapsed_time(e1) / 1e3 / args.calls
            # host form, called through ctypes with buffers allocated once
            h_out = [np.full((max(k, 1), 4), np.nan, np.float32) for k in n]
            arr = (L.CloudOut * lanes)(*[L.CloudOut(b.ctypes.data, len(b), 0) for b in h_out])
            free2 = torch.cuda.mem_get_info()[0]
            assert ctx.lib.lvo_map_cloud_batch(ctx.h, which, arr) == 0, ctx.lib.lvo_last_error(ctx.h)
            free3 = torch.cuda.mem_get_info()[0]
            host_launches = ctx.timings().kernel_launches
            ok_host = all(arr[l].n == n[l] and np.array_equal(h_out[l][:n[l]].view(np.uint32), ref[l].view(np.uint32)) for l in range(lanes))
            for _ in range(args.warm):
                ctx.lib.lvo_map_cloud_batch(ctx.h, which, arr)
            host_s = []
            for _ in range(args.calls):
                t0 = time.perf_counter()
                ctx.lib.lvo_map_cloud_batch(ctx.h, which, arr)
                host_s.append(time.perf_counter() - t0)
            # the packed-download strategy, through the device form into one buffer
            off = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
            d_packed = torch.empty((max(int(off[-1]), 1), 4), device="cuda")
            h_packed = torch.empty((max(int(off[-1]), 1), 4), pin_memory=True)
            hp = h_packed.numpy()
            a_out = [np.full((max(k, 1), 4), np.nan, np.float32) for k in n]
            VP, NS = C.c_void_p * lanes, C.c_size_t * lanes
            p_ptrs = VP(*[d_packed.data_ptr() + 16 * int(off[l]) for l in range(lanes)])
            p_caps, p_n = NS(*n), NS()
            torch.cuda.synchronize()

            def packed():
                assert ctx.lib.lvo_map_cloud_batch_dev(ctx.h, which, p_ptrs, p_caps, p_n) == 0
                with torch.cuda.stream(st):
                    h_packed.copy_(d_packed, non_blocking=True)
                st.synchronize()
                for l in range(lanes):
                    a_out[l][:n[l]] = hp[off[l]:off[l + 1]]

            packed()
            ok_packed = all(np.array_equal(a_out[l][:n[l]].view(np.uint32), ref[l].view(np.uint32)) for l in range(lanes))
            for _ in range(args.warm):
                packed()
            packed_s = []
            for _ in range(args.calls):
                t0 = time.perf_counter()
                packed()
                packed_s.append(time.perf_counter() - t0)
            del d_packed, h_packed
            t_loop, t_host, t_packed = statistics.median(loop_s), statistics.median(host_s), statistics.median(packed_s)
            out = {"points": sum(n), "points_per_lane_mean": sum(n) / lanes,
                   "bitwise_equal_to_single_lane": {"device_form": ok_dev, "host_form": ok_host, "packed_download_alternative": ok_packed},
                   "launches_per_call": {"device_form": dev_launches, "host_form": host_launches},
                   "arena_device_bytes_cudaMemGetInfo": {"device_form_first_call": free0 - free1, "host_form_first_call": free2 - free3}}
            for form, t in (("device_form", dev_s), ("host_form", t_host), ("packed_download_alternative", t_packed), ("single_lane_loop", t_loop)):
                out[form] = {"ms_per_call": t * 1e3, "point_GB_per_s": pts_bytes / t / 1e9}
            out["host_form_over_single_lane_loop"] = t_loop / t_host
            out["device_form_over_single_lane_loop"] = t_loop / dev_s
            run["outputs"][name] = out
            print(json.dumps({"lanes": lanes, name: out}), flush=True)
        res["runs"].append(run)
        if args.out:
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
        ctx.close()
    print(json.dumps(res["gpu"]))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
