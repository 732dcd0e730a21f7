"""GPU box: cost of the step surfaces (ssd_gpu_set_step_surfaces) on BASELINE.json configs[2]'s shape -- 4096 device-resident
1024 x 768 frames, vertex and z16 input -- and on one-frame latency. Arms, alternated round by round in one process: step labels on
with surfaces off, and step labels on with surfaces on (one more pass: the map is read again, 1 B per pixel, and the vertices of
the step pixels). Also the single-stream stage times of each arm (the surface pass is not a stage: it shows as the difference of
the call totals), and the card's name and power limit, read in the same call.
    python tools/step_surfaces_bench.py [--frames 4096] [--rounds 7] [--out FILE]
Appends its JSON lines to profiles/step_surfaces/b200_step_surfaces_bench.jsonl unless --out names another file."""
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
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--latency-reps", type=int, default=300)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "step_surfaces", "b200_step_surfaces_bench.jsonl"))
args = ap.parse_args()
W, H = 1024, 768
N, F = W * H, args.frames
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
out = open(args.out, "a") if args.out else None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": F, "size": f"{W}x{H}", "tool": "tools/step_surfaces_bench.py"})

cfg = S.default_config(W, H)
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
xf = S.scene_transform(base)
intr = S.scene_intrinsics(base)
det = S.Detector(cfg, xf, max_frames=F)
d_xyz = det.malloc(F * N * 12)
d_z16 = det.malloc(F * N * 2)
det.synth_frames(base, 1, 0, F, 3, 8, d_xyz, d_z16)


det.set_step_labels(True)


def call(on, inp, flags=0, n=F):
    det.set_step_surfaces(on)
    if inp == "xyz":
        det.process_device(d_xyz, n, flags)
    else:
        det.process_depth_device(d_z16, intr, n)
    return det.timing().total_ms


for inp in ("xyz", "z16"):
    ref = None
    for on in (False, True):  # warm-up of both arms; the results are the same either way
        call(on, inp)
        lines = [det.line(f) for f in range(0, F, 97)]
        ref = ref or lines
        assert lines == ref, (inp, on)
    times = {False: [], True: []}
    launches = {}
    for r in range(args.rounds):
        for on in ((False, True) if r % 2 == 0 else (True, False)):
            times[on].append(call(on, inp))
            launches[on] = det.timing().n_launches
    med = {on: float(np.median(v)) for on, v in times.items()}
    for on in (False, True):
        emit({"input": inp, "step_surfaces": on, "ms_median": round(med[on], 3), "ms_all": [round(t, 3) for t in times[on]],
              "kfps": round(F / med[on], 2), "n_launches": launches[on], "vs_off_pct": round(100.0 * (med[on] / med[False] - 1.0), 2),
              "vs_off_ms": round(med[on] - med[False], 3)})
    if inp == "xyz":  # per-stage device time, one stream (the depth device call takes no flags)
        for on in (False, True):
            q, tot = [], []
            for r in range(3):
                tot.append(call(on, inp, A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM))
                q.append(det.stage_times())
            emit({"input": inp, "step_surfaces": on, "serial_stage_ms_median_of_3":
                  {k: round(float(np.median([s[k][0] for s in q])), 3) for k in q[0]}})

# latency: one frame, host clock around the synchronous call
det1 = S.Detector(cfg, xf, max_frames=1)
det1.set_step_labels(True)


def one(on):
    det1.set_step_surfaces(on)
    t0 = time.perf_counter()
    det1.process_device(d_xyz, 1)
    return (time.perf_counter() - t0) * 1e6


for on in (False, True):
    for _ in range(30):
        one(on)
lat = {False: [], True: []}
for r in range(args.latency_reps):
    for on in ((False, True) if r % 2 == 0 else (True, False)):
        lat[on].append(one(on))
emit({"latency_us_median": {str(k): round(float(np.median(v)), 1) for k, v in lat.items()},
      "latency_us_p10": {str(k): round(float(np.percentile(v, 10)), 1) for k, v in lat.items()}})
det1.close()
det.free(d_xyz)
det.free(d_z16)
det.close()
