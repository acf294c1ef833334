#!/usr/bin/env python
"""bench.py — scan-to-map throughput of the B200 hot path (BASELINE.json metric) on synthetic HDL-64-shaped sweeps.

A "step" advances every lane (independent sequence) of this rank by `--frames-per-step` (default 5) sweeps through the full per-frame
path: lvo_extract_features -> lvo_scan_to_scan -> lvo_scan_to_map (device-resident chain).  With the driver's K = 20 steps the timed
region is 100 frames per lane (~2 s).  The lanes of a rank are split over `--groups` contexts, each with its own CUDA stream and host
thread, so that the stages of different groups overlap on the GPU.
  value : scans/s, whole job (all ranks, all lanes), inputs already resident in HBM (`lvo_step_batch_dev`), timed with one CUDA event
          pair on the main stream around all K steps of all contexts (inputs larger than L2: every frame reads new sweeps), max over ranks.
  e2e   : the same metric through `lvo_step_batch_pipelined` with HOST (pinned) sweep buffers — packed x,y,z records in one slab per
          sequence: every frame uploads one frame of sweeps (the next frame's, on a copy stream, overlapping this frame's compute)
          and reads the poses / lane state back, all inside the timed region.
  single_trajectory : BASELINE configs[0] literally — ONE sequence, one lane, host API: scans/s, latency percentiles, and the per-stage
          milliseconds under the reference's TicToc printf names, next to the CPU arm's per-stage milliseconds.
  roofline     : the 5-NN map-search kernel (k_map_knn) — algorithmic bytes 16 M + 56 Q per launch (SURVEY §8d) / its CUDA-event
                 duration, vs the measured HBM peak; `traffic` only from an ncu capture of the same launch state (profiles/r2_traffic.json).
  cpu_baseline : the reference's own node sources (oracle/_ref, kind "reference") when they were built, else the restated port, on one
                 host core, bounded sample, rank 0 at N=1 only.
`--impl reference` times that CPU implementation with all host threads (one independent sequence per thread).
Multi-GPU (torchrun): one process per GPU, lanes sharded across ranks with no data-path collective ("weak" scaling,
per-GPU work fixed); torch.distributed (NCCL) is used only for the barrier and the max-over-ranks of the timing.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def load_pkg():
    spec = importlib.util.spec_from_file_location("lvo_b200", os.path.join(ROOT, "lidar-visual-odometry_b200", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lvo_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def gen_sweeps(n_seq, n_frames, threads):
    from oracle_py import Synth
    synth = Synth()
    jobs = [(s, f) for s in range(n_seq) for f in range(n_frames)]
    with ThreadPoolExecutor(max_workers=threads) as ex:
        res = list(ex.map(lambda j: synth.sweep(64, j[0], j[1])[0], jobs))
    return {j: r for j, r in zip(jobs, res)}


def lane_plan(lanes, n_seq):
    """lane -> (sequence, frame offset).  Lanes are grouped by sequence: `lanes / n_seq` consecutive lanes follow one sequence, each
    entering it one frame later than its neighbour, so that at any step the sweeps of those lanes are ADJACENT frames of the
    per-sequence host slab (one merged upload per sequence, lvo_step_batch* stage_sweeps) while every lane still is its own trajectory."""
    per_seq = max(1, -(-lanes // n_seq))
    return [(l // per_seq, l % per_seq) for l in range(lanes)]


N_SEQ = 16


def rank_sequence_base(rank):
    """Sequence ids of a rank: distinct data per rank, no overlap (N_SEQ sequences per rank)."""
    return N_SEQ * rank


def max_over_ranks(values, world, device="cuda"):
    """The only cross-rank exchange of the bench: element-wise max of per-rank timings."""
    if world <= 1:
        return [float(v) for v in values]
    import torch
    import torch.distributed as dist
    t = torch.tensor(values, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def traffic_record(kernel):
    """DRAM bytes per launch of `kernel` from an `ncu --set full` capture, with the launch state it was taken in
    (profiles/r2_traffic.json: written from the committed ncu CSVs by profiles/ncu_traffic.py).  None when absent."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def knn_throughput(L, frames, reps, device, peak):
    """SURVEY §8d throughput mode of the graded kernel: many independent (map, query set) 5-NN problems in ONE launch, >= 1 GiB of
    map data, cold L2.  Two workloads:
      config3  : `frames` x (corner, surf) problems of config-3 size (~100 k corner + ~390 k surf map points, ~8 k queries of one
                 sweep per frame, all within ~60 m of the sensor) — the queries touch a quarter of the map;
      covering : the same maps with the queries spread over the WHOLE map (one query per ~5 map points, in the voxel-index order a
                 pcl::VoxelGrid output has), so that the algorithmic bytes 16 M + 56 Q are bytes the search really needs."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(1234)
    ax = torch.arange(-125.0, 125.0, 0.4, device="cuda")
    gx, gy = torch.meshgrid(ax, ax, indexing="ij")
    n_s = gx.numel()
    surf = torch.stack([gx.reshape(-1), gy.reshape(-1), torch.full((n_s,), -1.73, device="cuda"), torch.zeros(n_s, device="cuda")], 1)
    surf[:, :2] += (torch.rand(n_s, 2, device="cuda", generator=g) - 0.5) * 0.3
    surf[:, 2] += torch.randn(n_s, device="cuda", generator=g) * 0.02
    nl = 4000
    lx = (torch.rand(nl, 2, device="cuda", generator=g) - 0.5) * 250.0
    lz = torch.arange(-1.7, 8.3, 0.4, device="cuda")
    corner = torch.cat([lx[:, None, :].expand(nl, len(lz), 2), lz[None, :, None].expand(nl, len(lz), 1), torch.zeros(nl, len(lz), 1, device="cuda")], 2).reshape(-1, 4).contiguous()
    r = torch.rand(3000, device="cuda", generator=g).sqrt() * 40.0
    th = torch.rand(3000, device="cuda", generator=g) * 6.2831853
    q_s = torch.stack([r * torch.cos(th), r * torch.sin(th), torch.full((3000,), -1.70, device="cuda"), torch.zeros(3000, device="cuda")], 1)
    near = corner[(corner[:, 0].abs() < 60) & (corner[:, 1].abs() < 60)]
    q_c = near[torch.randint(0, len(near), (5000,), device="cuda", generator=g)].clone()
    q_c[:, :3] += torch.randn(5000, 3, device="cuda", generator=g) * 0.1
    # covering queries: every 5th map point, displaced by ~0.2 m
    qc_s = surf[torch.randperm(n_s, device="cuda", generator=g)[:n_s // 5]].clone()
    qc_s[:, :3] += torch.randn(len(qc_s), 3, device="cuda", generator=g) * 0.2
    qc_c = corner[torch.randperm(len(corner), device="cuda", generator=g)[:len(corner) // 5]].clone()
    qc_c[:, :3] += torch.randn(len(qc_c), 3, device="cuda", generator=g) * 0.1

    def voxel_order(q, leaf):
        # the order pcl::VoxelGrid leaves a cloud in (z, y, x voxel index ascending): what the stack of laserMapping.cpp:543-549 looks like
        v = torch.floor(q[:, :3] / leaf).to(torch.int64)
        v -= v.min(0).values
        key = (v[:, 2] * (int(v[:, 1].max()) + 1) + v[:, 1]) * (int(v[:, 0].max()) + 1) + v[:, 0]
        return q[torch.argsort(key, stable=True)].contiguous()
    qc_s, qc_c = voxel_order(qc_s, 0.8), voxel_order(qc_c, 0.4)
    out = {}
    for name, (qa, qb), nfr in (("config3", (q_c, q_s), frames), ("covering", (qc_c, qc_s), max(1, frames // 2))):
        maps, queries, mc, qc = [], [], [], []
        for f in range(nfr):
            off = torch.tensor([0.013 * f, -0.007 * f, 0.0, 0.0], device="cuda")
            for m, q in ((corner, qa), (surf, qb)):
                maps.append(m + off); queries.append(q + off); mc.append(len(m)); qc.append(len(q))
        maps = torch.cat(maps).contiguous(); queries = torch.cat(queries).contiguous()
        ind = torch.empty((len(queries), 5), dtype=torch.int32, device="cuda")
        sq = torch.empty((len(queries), 5), dtype=torch.float32, device="cuda")
        ctx = L.Lvo(lanes=1, device=device, max_points=65536, max_map_corner=1 << 16, max_map_surf=1 << 16, debug_probes=0)
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        ms = ctx.knn5_throughput(maps.data_ptr(), mc, queries.data_ptr(), qc, reps, ind.data_ptr(), sq.data_ptr())
        ctx.close()
        alg = 16.0 * sum(mc) + 56.0 * sum(qc)
        found = float((ind[:, 0] >= 0).float().mean())
        tr = traffic_record(f"k_knn5_batch/{name}")
        ok = tr is not None and tr.get("problems") == len(mc)
        dram = float(tr["dram_bytes_per_launch"]) if ok else None
        out[name] = {"kernel": "k_knn5_batch (same search as k_map_knn; L2 flushed before every timed launch)",
                     "problems": len(mc), "map_points_total": int(sum(mc)), "queries_total": int(sum(qc)), "map_bytes": 16 * int(sum(mc)), "kernel_ms": ms,
                     "algorithmic_bytes_per_launch": alg, "achieved_gbs": alg / 1e9 / (ms * 1e-3), "frac_algorithmic": alg / 1e9 / (ms * 1e-3) / peak,
                     "traffic": dram, "traffic_source": tr.get("source") if ok else None,
                     "frac_dram": (dram / 1e9 / (ms * 1e-3) / peak) if dram else None,
                     "queries_with_5_neighbours": found, "reps": reps}
        del maps, queries, ind, sq
        torch.cuda.empty_cache()
    return out


def extra_configs(L, device):
    """BASELINE configs 2 and 5 (reported next to the headline, not part of it).
    config 2: VLP-16 extract + scan-to-scan latency per frame through the host API (one trajectory, wall clock).
    config 5: camera-lidar depth association of 1120 keypoints against HDL-64 sweeps (wall clock, host API)."""
    from oracle_py import Synth
    synth = Synth()
    out = {}
    ctx = L.Lvo(n_scans=16, minimum_range=0.3, line_res=0.2, plane_res=0.4, device=device, max_points=65536, max_map_corner=1 << 16, max_map_surf=1 << 17)
    sweeps = [synth.sweep(16, 0, k)[0] for k in range(60)]
    lat = []
    for k, sw in enumerate(sweeps):
        t0 = time.perf_counter()
        _, f = ctx.extract_features(sw)
        ctx.scan_to_scan(f["sharp"], f["less_sharp"], f["flat"], f["less_flat"])
        if k >= 10:
            lat.append(1e3 * (time.perf_counter() - t0))
    ctx.close()
    out["config2_vlp16_scan_to_scan_latency_ms"] = {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)), "frames": len(lat),
                                                     "what": "lvo_extract_features + lvo_scan_to_scan per frame, host API incl. python binding"}
    ctx = L.Lvo(device=device, max_points=131072, max_map_corner=1 << 16, max_map_surf=1 << 17)
    cam = L.KITTI00_CAMERA
    rng = np.random.default_rng(5)
    px = np.stack([rng.uniform(20, cam["width"] - 20, 1120), rng.uniform(15, cam["height"] - 15, 1120)], 1)
    uv = np.stack([(px[:, 0] - cam["cx"]) / cam["fx"], (px[:, 1] - cam["cy"]) / cam["fy"]], 1).astype(np.float32)
    sweeps = [synth.sweep(64, 0, k)[0] for k in range(12)]
    for sw in sweeps[:2]:
        ctx.depth_associate(sw, uv)
    t0 = time.perf_counter()
    valid = 0
    for sw in sweeps[2:]:
        _, d, v, _ = ctx.depth_associate(sw, uv)
        valid += int(v.sum())
    dt = time.perf_counter() - t0
    ctx.close()
    # ---- config 3: dense map stress (tests/dense_map.py: ~100 k corner + ~385 k surf points that survive the per-cube re-filter;
    # parity at this size: tests/test_gpu_dense_map.py)
    import torch
    from dense_map import make_dense_map
    corner_np, cc_np, surf_np, sc_np = make_dense_map()
    ctx = L.Lvo(device=device, max_points=131072, max_map_corner=1 << 18, max_map_surf=1 << 20, debug_probes=0)
    # (a) voxel-downsample kernels in isolation on a 1.15 M-point cloud (3 jittered copies of the surf map), leaf 0.8
    surf = torch.from_numpy(surf_np).cuda()
    big = torch.cat([surf + torch.tensor([0.05 * i, 0.03 * i, 0.0, 0.0], device="cuda") for i in range(3)]).contiguous()
    dout = torch.empty_like(big)
    times = []
    for _ in range(6):
        n_out, ms = ctx.voxel_downsample_dev(big.data_ptr(), len(big), 0.8, dout.data_ptr())
        times.append(ms)
    ms = float(np.median(times[1:]))
    alg = 16.0 * (len(big) + n_out)
    out["config3_voxel_downsample"] = {"points_in": int(len(big)), "points_out": int(n_out), "kernel_ms": ms, "algorithmic_bytes": alg,
                                        "achieved_gbs": alg / 1e9 / (ms * 1e-3), "launches": int(ctx.timings().kernel_launches),
                                        "what": "lvo_voxel_downsample_dev (bbox + keys + LSD radix sort + centroids), leaf 0.8 m"}
    # (b) whole lvo_scan_to_map against the imported map
    ctx.map_import(0, corner_np, cc_np, surf_np, sc_np)
    from oracle_py import Oracle
    orc = Oracle()
    ident = np.array([0, 0, 0, 1, 0, 0, 0], float)
    tms, knn_us, stages = [], [], []
    for k in range(5):
        feats = orc.extract(synth.sweep(64, 0, k)[0])
        st, pose, _ = ctx.scan_to_map(feats["less_sharp"], feats["less_flat"], feats["full"], ident)
        tm = ctx.timings()
        tms.append(tm.mapping_ms); knn_us.append(1e3 * tm.knn_ms / max(tm.knn_launches, 1)); stages.append(ctx.stage_timings())
    stt = ctx.stats(0)
    out["config3_scan_to_map_dense_map"] = {"map_points_in_neighbourhood": [stt.map_corner_from_map, stt.map_surf_from_map], "queries": [stt.map_corner_stack, stt.map_surf_stack],
                                            "scan_to_map_ms": float(np.median(tms[1:])), "knn_launch_us": float(np.median(knn_us[1:])),
                                            "stage_ms": {k: float(np.median([s_[k] for s_ in stages[1:]])) for k in stages[0] if k.startswith("m") or k in ("add points time", "filter time", "build tree time")},
                                            "what": "one lvo_scan_to_map call (1 lane, host API, incl. uploads and the per-cube re-filter of the whole neighbourhood); "
                                                    "the map is re-filtered by every call and keeps its size (one point per voxel)"}
    ctx.close()
    out["config5_depth_association"] = {"sweeps_per_s": 10 / dt, "keypoints_per_s": 11200 / dt, "valid_fraction": valid / 11200.0,
                                        "what": "lvo_depth_associate, 120k-point sweep + 1120 keypoints per call, host API"}
    return out


def cpu_impl(kind):
    """The CPU implementation behind the reference arm / cpu_baseline.  "reference": the reference's OWN node sources
    (src/scanRegistration.cpp, src/laserOdometry.cpp, src/laserMapping.cpp compiled unmodified into oracle/_ref against shim ROS / PCL /
    Ceres headers whose back ends — VoxelGrid, kd-tree, trust-region LM — are restated; autodiff Jacobians as in the reference);
    "port": the hand restatement (oracle/liblvo_oracle.so: analytic Jacobians, own kd-tree + LM).  Returns (kind, factory, note)."""
    import refnode_py
    from oracle_py import Oracle
    if kind in ("auto", "reference") and refnode_py.available():
        return ("reference", lambda: refnode_py.RefPipeline(64, 5.0, 0.4, 0.8),
                "the reference's own scanRegistration / laserOdometry / laserMapping sources compiled unmodified (oracle/_ref); PCL VoxelGrid, FLANN kd-tree "
                "and Ceres LM back ends are restatements, not the PCL/Ceres binaries; one sequence = one worker process (the three nodes run one after the other)")
    if kind == "reference":
        raise SystemExit("bench.py: oracle/_ref/libref_*.so not built")
    return ("port", lambda: Oracle(64, 5.0, 0.4, 0.8), "restated reference (oracle/: own kd-tree + own LM, analytic Jacobians), not the PCL/Ceres binaries")


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path with all host threads: one independent sequence per thread."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, args.ref_threads or cores))
    F = args.frames_per_step
    total = (args.warmup + args.steps) * F
    nseq = min(threads, N_SEQ)
    sweeps = gen_sweeps(nseq, total, threads)
    kind, make, note = cpu_impl(args.ref_impl)

    def work(t):
        o = make()
        for k in range(args.warmup * F):
            o.step(sweeps[(t % nseq, k)])
        t0 = time.perf_counter()
        for k in range(args.warmup * F, total):
            o.step(sweeps[(t % nseq, k)])
        dt = time.perf_counter() - t0
        if hasattr(o, "close"):
            o.close()
        return dt

    with ThreadPoolExecutor(max_workers=threads) as ex:
        times = list(ex.map(work, range(threads)))
    dt = max(times)
    value = threads * args.steps * F / dt
    line = {"impl": "reference", "metric": "scan-to-map scans/sec (HDL-64 synthetic)", "value": value, "unit": "scans/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
            "data": "synthetic",
            "config": {"workload": "HDL-64 full pipeline (extract + scan-to-scan + scan-to-map), one sequence per host thread", "points_per_sweep": 120000,
                       "outer_iters": 10, "lm_iters": 4, "frames_per_step": F, "sequences": threads, "distinct_sequences": nseq},
            "cpu_baseline": {"value": value, "unit": "scans/s", "cores": threads, "kind": kind,
                             "sample": f"{threads} sequences ({nseq} distinct) x {args.steps} steps x {F} frames after {args.warmup * F} warm-up frames; {note}"},
            "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def dump_last_step(out_dir, record, groups, frames, total, suffix=""):
    """What lvo_step_batch_dev returned for the frames of the last timed step, as float64 .npy files: status[frame, context] and
    odometry_pose / mapping_pose[frame, lane, 7] (q x, y, z, w, t x, y, z; lanes in context order).  Two builds run with the same
    arguments see the same seeded sweeps, so their files can be compared array for array."""
    ks = range(total - frames, total)
    out = {"status": np.array([[record[(g, k)][0] for g in range(groups)] for k in ks], np.float64),
           "odometry_pose": np.stack([np.concatenate([record[(g, k)][1] for g in range(groups)]) for k in ks]).astype(np.float64),
           "mapping_pose": np.stack([np.concatenate([record[(g, k)][2] for g in range(groups)]) for k in ks]).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def quiet_stdout():
    """fd 1 -> fd 2 for everything else (NCCL prints its version banner on stdout, torchrun children share it)."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=int(os.environ.get("LVO_BENCH_FRAMES_PER_STEP", "5")),
                    help="sweeps every lane advances per step (5: the driver's 20 steps time 100 frames per lane, ~2 s)")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("LVO_BENCH_LANES", "0")),
                    help="independent sequences per GPU (0 = 384 when the GPU has >= 150 GB, else 128)")
    ap.add_argument("--groups", type=int, default=int(os.environ.get("LVO_BENCH_GROUPS", "0")),
                    help="contexts per GPU, each with lanes/groups sequences, its own CUDA stream and host thread (0 = one per 128 lanes)")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--ref-impl", default=os.environ.get("LVO_BENCH_REF_IMPL", "auto"), choices=["auto", "reference", "port"],
                    help="CPU implementation of the reference arm / cpu_baseline: the reference's own node sources (oracle/_ref) or the restated port")
    ap.add_argument("--cpu-sample-frames", type=int, default=40)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling aid: only the device-resident arm")
    ap.add_argument("--knn-frames", type=int, default=128, help="throughput-mode 5-NN: number of config-3 frames in one launch (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-2 / 3 / 5 side measurements")
    ap.add_argument("--no-single", action="store_true", help="skip the single-trajectory measurement")
    ap.add_argument("--map-caps", type=int, nargs=2, default=[1 << 18, 1 << 19], help="max_map_corner / max_map_surf of the timed contexts (points per lane)")
    ap.add_argument("--e2e-order", default=os.environ.get("LVO_BENCH_E2E_ORDER", "first"), choices=["first", "last"],
                    help="run the host-buffer arm before or after the device-resident arm")
    ap.add_argument("--graphs", type=int, default=int(os.environ.get("LVO_BENCH_GRAPHS", "-1")),
                    help="LVO_OPT_GRAPHS for the timed contexts: 1 = replay each frame from a CUDA graph, 0 = plain launches, -1 = graphs in the e2e arm only")
    ap.add_argument("--fixpoint-skip", type=int, default=int(os.environ.get("LVO_BENCH_FIXPOINT_SKIP", "1")),
                    help="LVO_OPT_FIXPOINT_SKIP of the timed contexts (library default 1): outer iterations after a bit-exact fixed point of the pose "
                         "are exact repeats and are not run; 0 = always run all ten")
    ap.add_argument("--no-full-schedule", action="store_true", help="skip the extra device-resident arm with LVO_OPT_FIXPOINT_SKIP = 0")
    ap.add_argument("--only-knn", action="store_true", help="profiling aid: only the throughput-mode 5-NN measurement")
    ap.add_argument("--profile-iso", type=int, default=0, help="profiling aid: bracket this many of the isolated frames after the timed region with "
                    "cudaProfilerStart / cudaProfilerStop (use with `ncu --profile-from-start off`: nothing before them is profiled or serialised)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the status and poses the device-resident arm returned in its last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    F = max(1, args.frames_per_step)
    args.frames_per_step = F

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sampler = ClockSampler(local_rank)
    sampler.start()   # early: nvidia-smi's start-up (NVML init takes a driver lock) must not fall into a timed region
    if args.lanes <= 0:
        args.lanes = 384 if torch.cuda.get_device_properties(local_rank).total_memory >= 150e9 else 128
    if args.groups <= 0:
        args.groups = max(1, args.lanes // 128)
    while args.lanes % args.groups:
        args.groups -= 1
    L = load_pkg()
    peak, peak_src = measured_peak_gbs()
    if args.only_knn:
        emit({"knn_throughput": knn_throughput(L, args.knn_frames, 5, local_rank, peak)})
        return
    lanes = args.lanes
    total = (args.warmup + args.steps) * F          # frames per lane in one arm
    n_seq = min(lanes, N_SEQ)
    plan = lane_plan(lanes, n_seq)
    max_off = max(o for _, o in plan)
    host_threads = os.cpu_count() or 1
    t_gen = time.perf_counter()
    # distinct data per rank: sequence ids are offset by N_SEQ * rank
    from oracle_py import Synth
    synth = Synth()
    iso_extra = 4   # frames after the timed region for the isolated kernel timing
    n_frames = total + max_off + iso_extra
    jobs = [(s, f) for s in range(n_seq) for f in range(n_frames)]
    with ThreadPoolExecutor(max_workers=host_threads) as ex:
        res = list(ex.map(lambda j: synth.sweep(64, rank_sequence_base(rank) + j[0], j[1])[0], jobs))
    sweeps = {j: r for j, r in zip(jobs, res)}
    t_gen = time.perf_counter() - t_gen

    stream = torch.cuda.current_stream()
    G = args.groups
    per = lanes // G
    mk = dict(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=per, device=local_rank, max_points=131072, max_map_corner=args.map_caps[0],
              max_map_surf=args.map_caps[1], debug_probes=0)
    # One context per group of `per` lanes, each on its own CUDA stream and driven by its own host thread (include/lvo.h: a context
    # is single-threaded, distinct contexts run concurrently — the reference's multi-sequence mechanism, SURVEY 8b "Threading").
    # The stages of different groups overlap on the GPU (sort-bound extraction next to latency-bound association / LM).
    gstreams = [torch.cuda.Stream(device=local_rank) for _ in range(G)]
    # LVO_OPT_GRAPHS: the host-buffer arm replays each frame from a CUDA graph (the host thread is free for the uploads);
    # the device-resident arm uses plain launches because the in-situ per-launch kNN events need them (same device time either way)
    graphs_e2e = args.graphs if args.graphs >= 0 else 1
    graphs_dev = args.graphs if args.graphs >= 0 else 0

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_groups(fn, k0, k1, after=None):
        """fn(g, k) for frames k in [k0, k1) on one host thread per group; after(g) runs on that thread at the end."""
        errs = []

        def work(g):
            try:
                torch.cuda.set_device(local_rank)
                for k in range(k0, k1):
                    fn(g, k)
                if after:
                    after(g)
            except Exception as e:  # noqa: BLE001
                errs.append(e)
        ths = [threading.Thread(target=work, args=(g,)) for g in range(G)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]

    def timed_run(step_fn, ctxs):
        """W warm-up steps, then K steps (K * F frames) of every group inside ONE event pair on the main stream: the group streams wait
        for the start event and the end event waits for every group's last kernel (device time of the whole region, all groups)."""
        acc = {"launches": 0, "knn_ms": 0.0, "knn_launches": 0, "knn_bytes": 0.0}
        lock = threading.Lock()

        def timed_step(g, k):
            step_fn(g, k)
            t = ctxs[g].timings()
            with lock:
                acc["launches"] += t.kernel_launches
                acc["knn_ms"] += t.knn_ms; acc["knn_launches"] += t.knn_launches; acc["knn_bytes"] += t.knn_bytes
        run_groups(step_fn, 0, args.warmup * F)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        done = [torch.cuda.Event() for _ in range(G)]
        wall0 = time.perf_counter()
        e0.record(stream)
        for gs in gstreams:
            gs.wait_event(e0)
        run_groups(timed_step, args.warmup * F, total, after=lambda g: done[g].record(gstreams[g]))
        for d in done:
            stream.wait_event(d)
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - wall0
        return e0.elapsed_time(e1), wall, acc["launches"], acc["knn_ms"], acc["knn_launches"], acc["knn_bytes"]

    # ---- e2e arm: host (pinned) sweeps through lvo_step_batch_pipelined ------------------------------------------------
    # One pinned slab per sequence, frames back to back as packed x,y,z records (12 bytes per point: the path never reads a sweep's
    # intensity, scanRegistration.cpp:132-133).  Lanes that follow one sequence one frame apart are adjacent in the slab and go up in one copy.
    nmax = max(len(a) for a in sweeps.values())
    slabs = []
    for s_ in range(n_seq):
        t = torch.zeros((n_frames, nmax, 3), dtype=torch.float32).pin_memory()
        for f in range(n_frames):
            a = sweeps[(s_, f)]
            t[f, :len(a)] = torch.from_numpy(a[:, :3])
        slabs.append(t.numpy())
    counts = {j: len(a) for j, a in sweeps.items()}
    gplan = [plan[g * per:(g + 1) * per] for g in range(G)]
    h2d = [0] * G

    def run_e2e():
        ctx_e = [L.Lvo(**mk) for _ in range(G)]
        for g in range(G):
            ctx_e[g].set_stream(gstreams[g].cuda_stream)
            ctx_e[g].set_option(L.LVO_OPT_GRAPHS, graphs_e2e)
            ctx_e[g].set_option(L.LVO_OPT_FIXPOINT_SKIP, args.fixpoint_skip)
        host_views = [dict() for _ in range(G)]

        def views_of(g, k):
            if k not in host_views[g]:
                host_views[g][k] = [slabs[s_][k + o, :counts[(s_, k + o)]] for s_, o in gplan[g]]
            return host_views[g][k]

        def step_host(g, k):
            # every frame uploads exactly one frame of sweeps from pinned host memory: frame k+1 goes up on the copy stream
            # while frame k computes (lvo_step_batch_pipelined), and the poses / lane state of frame k come back before it returns
            views = views_of(g, k)
            nxt = views_of(g, k + 1) if k + 1 < total else None
            h2d[g] = sum(v.nbytes for v in views)
            st, odo, mp = ctx_e[g].step_batch_pipelined(views, nxt)
            assert st >= 0
            host_views[g].pop(k - 1, None)

        ms, wall, _, _, _, _ = timed_run(step_host, ctx_e)
        for c in ctx_e:
            c.close()
        return ms, wall

    ms_e, wall_e = float("nan"), float("nan")
    if not args.skip_e2e and args.e2e_order == "first":
        ms_e, wall_e = run_e2e()

    # ---- device-resident arm ------------------------------------------------------------------------------------------
    dev = {j: torch.from_numpy(a).cuda() for j, a in sweeps.items()}

    def make_dev_contexts(fixpoint_skip):
        cs = [L.Lvo(**mk) for _ in range(G)]
        for g in range(G):
            cs[g].set_stream(gstreams[g].cuda_stream)
            cs[g].set_option(L.LVO_OPT_GRAPHS, graphs_dev)
            cs[g].set_option(L.LVO_OPT_STAGE_TIMING, 0)
            cs[g].set_option(L.LVO_OPT_FIXPOINT_SKIP, fixpoint_skip)
        return cs

    def dev_stepper(cs, record=None):
        def step_dev(g, k):
            ptrs = [dev[(s_, k + o)].data_ptr() for s_, o in gplan[g]]
            ns = [dev[(s_, k + o)].shape[0] for s_, o in gplan[g]]
            st, odo, mp = cs[g].step_batch_dev(ptrs, ns)
            assert st >= 0
            if record is not None and total - F <= k < total:
                record[(g, k)] = (st, odo, mp)
        return step_dev

    last_step = {} if args.dump_outputs else None
    ctx_d = make_dev_contexts(args.fixpoint_skip)
    step_dev = dev_stepper(ctx_d, last_step)

    ms_d, wall_d, launches, knn_ms_situ, knn_launches_situ, knn_bytes_situ = timed_run(step_dev, ctx_d)
    if args.dump_outputs:
        dump_last_step(args.dump_outputs, last_step, G, F, total, f"_rank{rank}" if world > 1 else "")
    st0 = ctx_d[0].stats(0)
    # outer iterations that ran in the last timed frame, mean over all lanes (10 = the reference's full schedule)
    ex = [(c.stats(l).odo_outer_executed, c.stats(l).map_outer_executed) for c in ctx_d for l in range(per)]
    outer_ran = [float(np.mean([e[0] for e in ex])), float(np.mean([e[1] for e in ex]))]
    map_sizes = np.array([[c.stats(l).map_corner_from_map, c.stats(l).map_surf_from_map] for c in ctx_d for l in range(per)])
    # LVO_OPT_KNN_REUSE: share of the scan-to-map queries that were searched in full, per outer iteration (iteration 0: all), last timed frame
    st_all = [c.stats(l) for c in ctx_d for l in range(per)]
    q_tot = float(sum(x.map_corner_stack + x.map_surf_stack for x in st_all if x.map_outer_executed > 0)) or 1.0
    knn_full_frac = [float(sum(x.map_knn_full[o] for x in st_all if x.map_outer_executed > o)) /
                     (float(sum(x.map_corner_stack + x.map_surf_stack for x in st_all if x.map_outer_executed > o)) or 1.0) for o in range(10)]
    # Roofline of the graded kernel: inside the timed region the contexts overlap, so a per-launch event time of k_map_knn includes
    # whatever the other streams were running.  It is therefore taken from context 0 advancing ALONE for a few more frames right
    # after the timed region (same maps, same library path, per-launch CUDA events inside the library); the in-situ average is
    # reported next to it.
    knn_ms = knn_bytes = 0.0
    knn_launches = 0
    iso_frames = 0
    ctx_d[0].set_option(L.LVO_OPT_GRAPHS, 0)   # the per-launch events need plain launches
    ctx_d[0].set_option(L.LVO_OPT_STAGE_TIMING, 1)
    ctx_d[0].set_option(L.LVO_OPT_FIXPOINT_SKIP, 0)   # ... and every one of the ten launches should search all lanes (kernel property)
    stage_batch = None
    for k in range(total, total + iso_extra):
        if args.profile_iso and k == total + iso_extra - args.profile_iso:
            torch.cuda.synchronize(); torch.cuda.profiler.start()
        step_dev(0, k)
        t = ctx_d[0].timings()
        knn_ms += t.knn_ms; knn_launches += t.knn_launches; knn_bytes += t.knn_bytes
        iso_frames += 1
        stage_batch = ctx_d[0].stage_timings()
    if args.profile_iso:
        torch.cuda.synchronize(); torch.cuda.profiler.stop()
    for c in ctx_d:
        c.close()
    # the same device-resident arm with the reference's full schedule (every lane runs all ten outer iterations), for comparison
    ms_f = float("nan")
    if args.fixpoint_skip and not args.no_full_schedule:
        ctx_f = make_dev_contexts(0)
        ms_f = timed_run(dev_stepper(ctx_f), ctx_f)[0]
        for c in ctx_f:
            c.close()
    if not args.skip_e2e and args.e2e_order == "last":
        ms_e, wall_e = run_e2e()
    clocks = sampler.stop()

    # max over ranks
    ms_d, ms_e, ms_f = max_over_ranks([ms_d, ms_e, ms_f], world)
    scans = lanes * args.steps * F * world
    value = scans / (ms_d * 1e-3)
    e2e = scans / (ms_e * 1e-3)
    achieved = (knn_bytes / 1e9) / (knn_ms * 1e-3) if knn_ms > 0 else 0.0

    # ---- single trajectory (BASELINE configs[0] literally): one sequence, one lane, host buffers through the public API ----------
    single = None
    if rank == 0 and world == 1 and not args.no_single:
        seq0 = [slabs[0][f, :counts[(0, f)]] for f in range(min(n_frames, 110))]
        c1 = L.Lvo(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=1, device=local_rank, max_points=131072, max_map_corner=1 << 18,
                   max_map_surf=1 << 19, debug_probes=0)
        lat = []
        for k, sw in enumerate(seq0):                      # CUDA-graph replay (the default for <= 8 lanes), one pinned sweep up, poses back
            t0 = time.perf_counter()
            st, odo, mp = c1.step_batch([sw])
            if k >= 10:
                lat.append(1e3 * (time.perf_counter() - t0))
        c1.close()
        c2 = L.Lvo(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=1, device=local_rank, max_points=131072, max_map_corner=1 << 18,
                   max_map_surf=1 << 19, debug_probes=0)
        c2.set_option(L.LVO_OPT_GRAPHS, 0)                 # plain launches: the sub-stage events need them
        stages = []
        for k, sw in enumerate(seq0[:60]):
            c2.step_batch([sw])
            if k >= 10:
                stages.append(c2.stage_timings())
        launches_frame = int(c2.timings().kernel_launches)
        c2.close()
        single = {"what": "ONE synthetic HDL-64 sequence (sequence 0, ~119.4 k returns per sweep), one lane, lvo_step_batch with a pinned host sweep per frame "
                          "(H2D of the sweep + D2H of the lane state inside the timing), wall clock; frame = extract + scan-to-scan + scan-to-map",
                  "scans_per_s": 1e3 / float(np.mean(lat)), "frames": len(lat),
                  "latency_ms": {"mean": float(np.mean(lat)), "p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99))},
                  "cuda_graph": True, "kernel_launches_per_frame": launches_frame,
                  "stage_ms_gpu": {k_: float(np.mean([s_[k_] for s_ in stages])) for k_ in stages[0]},
                  "stage_ms_note": "CUDA-event milliseconds per frame (mean of 50 frames, plain launches, so the sum exceeds the graph-replay latency) under the "
                                   "reference's TicToc printf names: scanRegistration.cpp:254,409,410,456; laserOdometry.cpp:564,577,665; "
                                   "laserMapping.cpp:552,560,710,721,728,784,802,850,852"}

    knn_tp = None
    if rank == 0 and world == 1 and args.knn_frames > 0:
        del dev
        torch.cuda.empty_cache()
        try:
            knn_tp = knn_throughput(L, args.knn_frames, 5, local_rank, peak)
        except Exception as e:  # noqa: BLE001 — a side measurement must not lose the headline
            knn_tp = {"error": repr(e)}
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            extras = extra_configs(L, local_rank)
        except Exception as e:  # noqa: BLE001
            extras = {"error": repr(e)}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nf = min(args.cpu_sample_frames, n_frames)
        legs = {}
        for want in ("auto", "port"):
            kind, make, note = cpu_impl(want)
            if kind in legs:
                continue
            o = make()
            stage = np.zeros(3)
            t0 = time.perf_counter()
            for k in range(nf):
                r = o.step(sweeps[(0, k)])
                if k >= nf // 2:
                    stage += np.array(r["times"]) * 1e3 if isinstance(r, dict) else np.array(o.timings())
            dt = time.perf_counter() - t0
            if hasattr(o, "close"):
                o.close()
            stage /= max(1, nf - nf // 2)
            legs[kind] = {"value": nf / dt, "unit": "scans/s", "cores": 1, "kind": kind,
                          "stage_ms": {"scan registration time": float(stage[0]), "whole laserOdometry time": float(stage[1]), "whole mapping time": float(stage[2])},
                          "sample": f"first {nf} frames of sequence 0, one sequence on one host core; {note}; host has {host_threads} cores"}
        cpu = legs.get("reference") or legs["port"]
        if "reference" in legs:
            cpu["port"] = {k_: legs["port"][k_] for k_ in ("value", "stage_ms", "sample")}

    if rank == 0:
        d2h = lanes * int(L.load_library().lvo_state_bytes())  # LaneState record per lane (poses, counters, status)
        tr = traffic_record("k_map_knn")
        tr_ok = tr is not None and tr.get("lanes_per_launch") == per
        line = {"metric": "scan-to-map scans/sec (HDL-64 synthetic)", "value": value, "unit": "scans/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_d / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": f"HDL-64 full pipeline (extract + scan-to-scan + scan-to-map), {lanes} independent sequences per GPU "
                                       f"in {G} contexts of {per} lanes (one CUDA stream + host thread each), {F} frames per step",
                           "lanes_per_gpu": lanes, "contexts_per_gpu": G, "frames_per_step": F, "timed_frames_per_lane": args.steps * F,
                           "distinct_sequences_per_gpu": n_seq, "lane_plan": f"{lanes // n_seq} lanes per sequence, entering it one frame apart",
                           "cuda_graphs": {"e2e_arm": graphs_e2e, "device_arm": graphs_dev}, "points_per_sweep": 120000, "outer_iters": 10, "lm_iters": 4,
                           "map_points_in_neighbourhood_last_frame": {"corner_mean": float(map_sizes[:, 0].mean()), "surf_mean": float(map_sizes[:, 1].mean()),
                                                                      "corner_max": int(map_sizes[:, 0].max()), "surf_max": int(map_sizes[:, 1].max())},
                           "fixpoint_skip": {"enabled": args.fixpoint_skip, "outer_iterations_run_mean": {"scan_to_scan": outer_ran[0], "scan_to_map": outer_ran[1]},
                                             "what": "LVO_OPT_FIXPOINT_SKIP (include/lvo.h): an outer iteration that returns the pose bit for bit unchanged makes "
                                                     "the remaining ones exact repeats; they are not run. Poses / maps / counters are bitwise those of the full "
                                                     "schedule (tests/test_gpu_mapping.py::test_fixpoint_skip_is_bitwise_identical)"},
                           "knn_reuse": {"full_search_fraction_per_outer_iteration": knn_full_frac,
                                         "what": "LVO_OPT_KNN_REUSE (include/lvo.h): share of a lane's 5-NN queries searched in full in each outer iteration of the "
                                                 "last timed frame; the others re-rank their five known neighbours under a guard-radius certificate (bitwise the "
                                                 "same rows: tests/test_gpu_mapping.py::test_knn_reuse_is_bitwise_identical)"},
                           "l2": f"inputs larger than L2: every frame reads {lanes} new sweeps ({lanes * 1.92:.0f} MB) and rebuilds every grid; no flush",
                           "timing": "one CUDA event pair on the main stream around all K steps of all contexts (context streams wait for the start event, "
                                     "the end event waits for every context's last kernel)"},
                "e2e": {"value": e2e, "unit": "scans/s", "h2d_bytes_per_step": sum(h2d) * F * world, "d2h_bytes_per_step": d2h * F * world,
                        "per_gpu_h2d_bytes_per_frame": sum(h2d), "ms_per_step": ms_e / args.steps,
                        "host_layout": "packed x,y,z float32 records (12 B / point), one pinned slab per sequence; merged uploads (one copy per run of adjacent lanes)"},
                "gpu_launches": launches,
                "full_schedule": None if ms_f != ms_f else {"value": scans / (ms_f * 1e-3), "unit": "scans/s", "ms_per_step": ms_f / args.steps,
                                                            "what": "device-resident arm with LVO_OPT_FIXPOINT_SKIP = 0: all ten outer iterations run for every lane"},
                "single_trajectory": single,
                "roofline": {"bound": "hbm", "kernel": "k_map_knn_reuse (5-NN grid search of lvo_scan_to_map; LVO_OPT_KNN_REUSE carries certified neighbour sets across outer iterations)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak if peak else None,
                             # dram__bytes_read.sum + dram__bytes_write.sum per launch of an `ncu --set full` capture taken in the SAME launch state
                             # (lanes per launch, frame index, commit recorded in profiles/r2_traffic.json); null when no such capture exists
                             "traffic": float(tr["dram_bytes_per_launch"]) if tr_ok else None, "traffic_source": tr.get("source") if tr_ok else None,
                             "peak_source": peak_src, "launches": knn_launches,
                             "avg_launch_us": 1e3 * knn_ms / max(knn_launches, 1), "algorithmic_bytes_per_launch": knn_bytes / max(knn_launches, 1),
                             "lanes_per_launch": per,
                             "how": f"context 0 alone for {iso_frames} frames after the timed region (frame {total} on), LVO_OPT_FIXPOINT_SKIP = 0 so that every launch "
                                    "searches all lanes (per-launch CUDA events inside the library)",
                             "in_situ_avg_launch_us": (1e3 * knn_ms_situ / knn_launches_situ) if knn_launches_situ else None,
                             "in_situ_note": "per-launch events are off inside the timed region (LVO_OPT_STAGE_TIMING = 0): there the launch overlaps the other contexts' kernels",
                             "stage_ms_per_frame_batched": stage_batch},
                "knn_throughput": knn_tp, "other_configs": extras, "cpu_baseline": cpu, "clocks": clocks,
                "host": {"wall_ms_per_step_dev": 1e3 * wall_d / args.steps, "wall_ms_per_step_e2e": 1e3 * wall_e / args.steps, "gen_s": t_gen, "cores": host_threads}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
