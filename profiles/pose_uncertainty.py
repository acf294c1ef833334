"""Cost of reading pose uncertainty (LVO_P_ODO_UNCERTAINTY / LVO_P_MAP_UNCERTAINTY) and the bench headline before / after the feature.

Fetch cost: contexts of 1, 32 and 128 lanes with bench.py's HDL-64 settings (max_points 131072, maps of 256 k corner / 512 k surf
points, debug_probes 0, plain launches), lane l running synthetic HDL-64 sequence l % 16.  After `--warm` steps, for each of `--steps`
further steps, host clock around
  - the first fetch after the step (one k_pose_uncertainty launch for every lane and stage, one device-to-host copy, a synchronise);
  - a later fetch of the same record (served from the host mirror);
  - reading both records of every lane after the step (the fleet pattern: one launch and one copy in all).
`--bench`: bench.py with default arguments, alternating the build under test and `--parent-lib` (LVO_LIB_PATH), two runs of each.
The GPU's name and power limit are read in the same run.

Usage:  python profiles/pose_uncertainty.py [--warm 5] [--steps 20] [--bench] [--parent-lib PATH] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from lane_lifecycle import ROOT, gpu_identity, load_pkg  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))


def stats_us(xs):
    return {"median_us": statistics.median(xs) * 1e6, "min_us": min(xs) * 1e6, "max_us": max(xs) * 1e6, "n": len(xs)}


def fetch_cost(L, synth, lanes, warm, steps):
    import torch
    n_seq = min(lanes, 16)
    frames = warm + steps
    jobs = [(s, f) for s in range(n_seq) for f in range(frames + steps)]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        host = list(ex.map(lambda j: synth.sweep(64, j[0], j[1])[0], jobs))
    dev = {j: torch.from_numpy(h).cuda() for j, h in zip(jobs, host)}
    torch.cuda.synchronize()
    ctx = L.Lvo(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=lanes, max_points=131072, max_map_corner=1 << 18,
                max_map_surf=1 << 19, debug_probes=0)
    ctx.set_option(L.LVO_OPT_GRAPHS, 0)
    first, later, fleet = [], [], []
    for f in range(frames):
        d = [dev[(l % n_seq, f)] for l in range(lanes)]
        ctx.step_batch_dev([t.data_ptr() for t in d], [t.shape[0] for t in d])
        if f < warm:
            continue
        t0 = time.perf_counter()
        ctx.pose_uncertainty(0, "odometry")
        t1 = time.perf_counter()
        ctx.pose_uncertainty(0, "odometry")
        t2 = time.perf_counter()
        first.append(t1 - t0)
        later.append(t2 - t1)
    # the fleet pattern: one more step, then every record of every lane
    for f in range(steps):
        d = [dev[(l % n_seq, frames + f)] for l in range(lanes)]
        ctx.step_batch_dev([t.data_ptr() for t in d], [t.shape[0] for t in d])
        t0 = time.perf_counter()
        for l in range(lanes):
            ctx.pose_uncertainty(l, "odometry")
            ctx.pose_uncertainty(l, "mapping")
        fleet.append(time.perf_counter() - t0)
    ctx.close()
    return {"lanes": lanes, "first_fetch": stats_us(first), "later_fetch": stats_us(later), "all_records_after_step": stats_us(fleet)}


def bench_line(lib):
    env = dict(os.environ)
    if lib:
        env["LVO_LIB_PATH"] = lib
    else:
        env.pop("LVO_LIB_PATH", None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], capture_output=True, text=True, env=env, cwd=ROOT, check=True)
    line = [x for x in r.stdout.strip().splitlines() if x.startswith("{")][-1]
    return json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from oracle_py import Synth
    L = load_pkg()
    out = {"identity": gpu_identity(torch), "fetch": [fetch_cost(L, Synth(), n, args.warm, args.steps) for n in (1, 32, 128)]}
    if args.bench:
        runs = []
        for rep in range(2):
            for name, lib in (("this", None), ("parent", args.parent_lib)):
                d = bench_line(lib)
                runs.append({"build": name, "rep": rep, "value": d.get("value"), "ms_per_step": d.get("ms_per_step"), "line": d})
        out["bench"] = runs
    out["identity_after"] = gpu_identity(torch)
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
