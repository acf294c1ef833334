"""bench.py --dump-outputs: the files hold what the timed device-resident path returned in its last timed step, lane for lane and bit
for bit, and --steps sets how many steps are timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_dump_outputs_hold_the_last_timed_step(lvo_mod, synth, tmp_path):
    import torch
    L = lvo_mod
    lanes, steps, warmup, F = 2, 2, 3, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                        "--frames-per-step", str(F), "--lanes", str(lanes), "--skip-e2e", "--no-full-schedule", "--no-single", "--no-extras",
                        "--knn-frames", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == steps and line["config"]["timed_frames_per_lane"] == steps * F
    status, odo, mp = (np.load(tmp_path / f"{n}.npy") for n in ("status", "odometry_pose", "mapping_pose"))
    assert status.dtype == odo.dtype == mp.dtype == np.float64
    assert status.shape == (F, 1) and odo.shape == mp.shape == (F, lanes, 7)
    # the same lanes replayed: with 2 lanes and 2 sequences (bench.lane_plan) lane l follows sequence l from frame 0, one context
    lvo = L.Lvo(n_scans=64, minimum_range=5.0, line_res=0.4, plane_res=0.8, lanes=lanes, max_points=131072, max_map_corner=1 << 18,
                max_map_surf=1 << 19, debug_probes=0)
    lvo.set_option(L.LVO_OPT_GRAPHS, 0)
    lvo.set_option(L.LVO_OPT_STAGE_TIMING, 0)
    lvo.set_option(L.LVO_OPT_FIXPOINT_SKIP, 1)
    total = (warmup + steps) * F
    for k in range(total):
        dev = [torch.from_numpy(synth.sweep(64, l, k)[0]).cuda() for l in range(lanes)]
        torch.cuda.synchronize()
        st, o, m = lvo.step_batch_dev([d.data_ptr() for d in dev], [d.shape[0] for d in dev])
        j = k - (total - F)
        if j >= 0:
            assert st == status[j, 0] and np.array_equal(o, odo[j]) and np.array_equal(m, mp[j]), k
    lvo.close()
