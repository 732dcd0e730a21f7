"""GPU box: cost of frame groups (ssd_gpu_process_groups_* / ssd_gpu_process_depth_groups_*) on BASELINE.json configs[2]'s shape --
4096 device-resident 1024 x 768 frames of eight cameras, vertex and z16 input. Arms, alternated round by round in one process:
    (a) one camera call (every frame detected on its own), (b) 512 groups of 8 frames, (c) 128 groups of 32 frames.
The eight table entries are one camera's record, so the point kernels do the same work in every arm; what differs is that a group
accumulates its members into one histogram, one set of BEV images and one set of step sums, and that the per-group kernels run once
per group. Also: the single-stream per-stage times of each arm, and the latency of one 3-frame group against a 3-frame camera call
(host clock).
    python tools/groups_bench.py [--frames 4096] [--rounds 5] [--out profiles/groups/b200_groups_bench.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import stair_step_detector_b200 as S  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--latency-reps", type=int, default=200)
ap.add_argument("--out", default="")
args = ap.parse_args()
W, H = 1024, 768
N, F = W * H, args.frames
out = open(args.out, "a") if args.out else None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": F, "size": f"{W}x{H}", "tool": "tools/groups_bench.py"})

cfg = S.default_config(W, H)
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
cam = S.scene_camera(base)
det = S.Detector(cfg, cam.xf, max_frames=F)
d_xyz = det.malloc(F * N * 12)
d_z16 = det.malloc(F * N * 2)
det.synth_frames(base, 1, 0, F, 3, 8, d_xyz, d_z16)
det.set_cameras([cam] * 8)
order = (np.arange(F, dtype=np.int32) % 8)
arms = {"a": None, "b": np.full(F // 8, 8, np.int32), "c": np.full(F // 32, 32, np.int32)}


def call(arm, inp, flags=0):
    g = arms[arm]
    if inp == "xyz":
        if g is None:
            det.process_cameras_device(d_xyz, order, F, flags)
        else:
            det.process_groups_device(d_xyz, order, g, flags)
    else:
        if g is None:
            det.process_depth_cameras_device(d_z16, order, F)
        else:
            det.process_depth_groups_device(d_z16, order, g, flags)
    return det.timing().total_ms


for inp in ("xyz", "z16"):
    ref = {}
    for arm in arms:  # warm-up of every arm; each arm gives the same results call after call
        call(arm, inp)
        ref[arm] = det.n_steps_all(F).tobytes()
        call(arm, inp)
        assert det.n_steps_all(F).tobytes() == ref[arm], (inp, arm)
    times = {a: [] for a in arms}
    for r in range(args.rounds):
        for arm in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            times[arm].append(call(arm, inp))
    med = {a: float(np.median(v)) for a, v in times.items()}
    for arm in arms:
        emit({"input": inp, "arm": arm, "group_frames": 1 if arms[arm] is None else int(arms[arm][0]), "ms_median": round(med[arm], 3),
              "ms_all": [round(t, 3) for t in times[arm]], "kfps": round(F / med[arm], 2),
              "vs_camera_call_pct": round(100.0 * (med[arm] / med["a"] - 1.0), 2)})
    for arm in arms:  # per-stage device time, one stream (the kernels' own durations; the z16 camera call takes no flags)
        if inp == "z16" and arm == "a":
            continue
        call(arm, inp, A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM)
        emit({"input": inp, "arm": arm, "serial_stage_ms": {k: round(v[0], 3) for k, v in det.stage_times().items()}})

# latency: one 3-frame group against a 3-frame camera call, host clock
det3 = S.Detector(cfg, cam.xf, max_frames=3)
det3.set_cameras([cam] * 3)
order3 = np.arange(3, dtype=np.int32)
fns = {"camera_call_3_frames": lambda: det3.process_cameras_device(d_xyz, order3, 3),
       "group_of_3_frames": lambda: det3.process_groups_device(d_xyz, order3, [3])}
for _ in range(20):
    for fn in fns.values():
        fn()
lat = {k: [] for k in fns}
for r in range(args.latency_reps):
    for name, fn in fns.items():
        t0 = time.perf_counter()
        fn()
        lat[name].append((time.perf_counter() - t0) * 1e6)
emit({"latency_us_median": {k: round(float(np.median(v)), 1) for k, v in lat.items()},
      "latency_us_p10": {k: round(float(np.percentile(v, 10)), 1) for k, v in lat.items()}})
det3.close()
det.free(d_xyz)
det.free(d_z16)
det.close()
