"""Cost of idle lanes and of lvo_lane_reset in the batched device-resident pipeline (lvo_step_batch_dev).

One 128-lane context with bench.py's configuration and sweeps (16 seeded synthetic HDL-64 sequences, 8 lanes each, entering their
sequence one frame apart).  For 0, 1/4, 1/2 and 3/4 of the lanes idle (lanes l with l % 4 below the idle quarter count, so every
sequence keeps active lanes), after warm-up steps, each of `--steps` steps is timed:
  - device step time: the context's stage events (lvo_timings extract + odometry + mapping, plain launches), and
  - active-lane scans/s = active lanes / device step time.
Then the host time of lvo_lane_reset (the call returns after the stream has finished the reset).  The GPU's name and power limit are
read in the same run.  An idle lane still pays its odometry grid rebuild and the copy of its map into the other generation; how much of
an active lane's cost it saves is what the numbers show.

Usage:  python profiles/lane_lifecycle.py [--steps 20] [--warmup 5] [--out FILE.json]"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def load_pkg():
    spec = importlib.util.spec_from_file_location("lvo_b200", os.path.join(ROOT, "lidar-visual-odometry_b200", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lvo_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def gpu_identity(torch):
    """Name, power limit and top SM clock of the card the context runs on.  nvidia-smi numbers GPUs without regard to
    CUDA_VISIBLE_DEVICES, so the card is selected by the PCI bus id of CUDA device 0."""
    p = torch.cuda.get_device_properties(0)
    bus = f"{p.pci_domain_id:08X}:{p.pci_bus_id:02X}:{p.pci_device_id:02X}.0"
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,pci.bus_id", "--format=csv,noheader", "-i", bus],
                       capture_output=True, text=True, check=True)
    name, power, clock, smi_bus = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "gpu_torch_name": p.name, "pci_bus_id": smi_bus, "power_limit": power, "sm_clock_max": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--resets", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from oracle_py import Synth
    L = load_pkg()
    lanes, n_seq = args.lanes, 16
    per_seq = lanes // n_seq
    plan = [(l // per_seq, l % per_seq) for l in range(lanes)]          # bench.lane_plan
    idle_quarters = (0, 1, 2, 3)
    frames = len(idle_quarters) * (args.warmup + args.steps) + per_seq
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
    frame = [0] * lanes                     # each lane's own position in its sequence: idle lanes do not advance
    out = {"config": {"lanes": lanes, "sequences": n_seq, "steps": args.steps, "warmup": args.warmup, "entry": "lvo_step_batch_dev",
                      "max_points": 131072, "map_caps": [1 << 18, 1 << 19], "graphs": 0}, "runs": []}
    out.update(gpu_identity(torch))
    for q in idle_quarters:
        active = [l % 4 >= q for l in range(lanes)]
        for l in range(lanes):
            ctx.set_lane_active(l, active[l])
        dev_ms, wall_ms = [], []
        for k in range(args.warmup + args.steps):
            ptrs, ns = [], []
            for l in range(lanes):
                if active[l]:
                    s, off = plan[l]
                    t = dev[(s, off + frame[l])]
                    ptrs.append(t.data_ptr()); ns.append(t.shape[0])
                    frame[l] += 1
                else:
                    ptrs.append(None); ns.append(None)
            w0 = time.perf_counter()
            st, _, _ = ctx.step_batch_dev(ptrs, ns)
            w1 = time.perf_counter()
            assert st >= 0, st
            if k >= args.warmup:
                t = ctx.timings()
                dev_ms.append(t.extract_ms + t.odometry_ms + t.mapping_ms)
                wall_ms.append((w1 - w0) * 1e3)
        n_act = sum(active)
        med = statistics.median(dev_ms)
        out["runs"].append({"idle_fraction": q / 4, "active_lanes": n_act, "device_step_ms_median": med,
                            "device_step_ms_min": min(dev_ms), "device_step_ms_max": max(dev_ms), "host_step_ms_median": statistics.median(wall_ms),
                            "active_scans_per_s": n_act / (med / 1e3), "device_ms_per_active_lane": med / n_act})
        print(json.dumps(out["runs"][-1]), flush=True)
    base = out["runs"][0]["device_step_ms_median"]
    for r in out["runs"]:
        r["step_time_vs_all_active"] = r["device_step_ms_median"] / base
    reset_ms = []
    for i in range(args.resets):
        lane = (i * 37) % lanes
        t0 = time.perf_counter()
        ctx.lane_reset(lane)
        reset_ms.append((time.perf_counter() - t0) * 1e3)
    out["lane_reset_host_ms"] = {"median": statistics.median(reset_ms), "min": min(reset_ms), "max": max(reset_ms), "calls": len(reset_ms)}
    ctx.close()
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
