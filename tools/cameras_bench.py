"""GPU box: cost of per-frame cameras (ssd_gpu_set_cameras) on BASELINE.json configs[2]'s shape -- 4096 device-resident
1024 x 768 frames, vertex and z16 input. Arms, alternated round by round in one process:
    (a) the plain call, (b) a camera call with one camera, (c) eight cameras interleaved, (d) one camera per frame.
The frames are seeded synthetic scenes of one camera pose and every table entry is that camera's record, so all arms do the
same work and must give the same results: the difference is the cost of the per-frame lookup alone. Also: the host time of
ssd_gpu_set_cameras for 8 and 4096 cameras, and one 8-frame camera call against eight single-frame plain calls.
    python tools/cameras_bench.py [--frames 4096] [--rounds 5]     (one JSON line per measurement)"""
import argparse
import ctypes
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
args = ap.parse_args()
W, H = 1024, 768
N, F = W * H, args.frames


def emit(d):
    print(json.dumps(d), flush=True)


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": F, "size": f"{W}x{H}"})

cfg = S.default_config(W, H)
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
xf = S.scene_transform(base)
intr = S.scene_intrinsics(base)
cam = S.scene_camera(base)
det = S.Detector(cfg, xf, max_frames=F)
d_xyz = det.malloc(F * N * 12)
d_z16 = det.malloc(F * N * 2)
det.synth_frames(base, 1, 0, F, 3, 8, d_xyz, d_z16)

set_ms = {}
for n_cam in (8, F):
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        det.set_cameras([cam] * n_cam)
        ts.append((time.perf_counter() - t0) * 1e3)
    set_ms[n_cam] = min(ts)
emit({"set_cameras_host_ms": {str(k): round(v, 3) for k, v in set_ms.items()}})

tables = {"b": (1, np.zeros(F, np.int32)), "c": (8, np.arange(F, dtype=np.int32) % 8), "d": (F, np.arange(F, dtype=np.int32))}


def call(arm, inp, flags=0):
    if arm == "a":
        if inp == "xyz":
            det.process_device(d_xyz, F, flags)
        else:
            det.process_depth_device(d_z16, intr, F)
    else:
        n_cam, order = tables[arm]
        if det.n_cameras != n_cam:
            det.set_cameras([cam] * n_cam)
        if inp == "xyz":
            det.process_cameras_device(d_xyz, order, F, flags)
        else:
            det.process_depth_cameras_device(d_z16, order, F)
    return det.timing().total_ms


arms = ["a", "b", "c", "d"]
for inp in ("xyz", "z16"):
    ref = None
    for arm in arms:  # warm-up of every arm, and the same results everywhere
        call(arm, inp)
        out = (det.n_steps_all(F).tobytes(), bytes(det.stats()))
        ref = ref or out
        assert out[0] == ref[0], (inp, arm)
    times = {a: [] for a in arms}
    for r in range(args.rounds):
        for arm in (arms if r % 2 == 0 else arms[::-1]):
            times[arm].append(call(arm, inp))
    med = {a: float(np.median(v)) for a, v in times.items()}
    for arm in arms:
        emit({"input": inp, "arm": arm, "n_cameras": 0 if arm == "a" else tables[arm][0], "ms_median": round(med[arm], 3),
              "ms_all": [round(t, 3) for t in times[arm]], "kfps": round(F / med[arm], 2),
              "vs_plain_pct": round(100.0 * (med[arm] / med["a"] - 1.0), 2)})
    if inp == "xyz":
        for arm in ("a", "d"):  # per-stage device time, one stream (the kernels' own durations)
            call(arm, inp, A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM)
            emit({"input": inp, "arm": arm, "serial_stage_ms": {k: round(v[0], 3) for k, v in det.stage_times().items()}})

# latency: one 8-frame camera call (eight cameras, one frame each) against eight single-frame plain calls, host clock
det8 = S.Detector(cfg, xf, max_frames=8)
det8.set_cameras([cam] * 8)
order8 = np.arange(8, dtype=np.int32)
frame = lambda i: ctypes.c_void_p(d_xyz.value + i * N * 12)  # noqa: E731


def one_cam_call():
    det8.process_cameras_device(d_xyz, order8, 8)


def eight_plain_calls():
    for i in range(8):
        det8.process_device(frame(i), 1)


lat = {}
for name, fn in (("camera_call_8_frames", one_cam_call), ("eight_plain_single_frame_calls", eight_plain_calls)):
    for _ in range(20):
        fn()
lat = {"camera_call_8_frames": [], "eight_plain_single_frame_calls": []}
for r in range(args.latency_reps):
    for name, fn in (("camera_call_8_frames", one_cam_call), ("eight_plain_single_frame_calls", eight_plain_calls)):
        t0 = time.perf_counter()
        fn()
        lat[name].append((time.perf_counter() - t0) * 1e6)
emit({"latency_us_median": {k: round(float(np.median(v)), 1) for k, v in lat.items()},
      "latency_us_p10": {k: round(float(np.percentile(v, 10)), 1) for k, v in lat.items()}})
det8.close()
det.free(d_xyz)
det.free(d_z16)
det.close()
