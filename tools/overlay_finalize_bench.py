"""GPU box: device time of the finalize stage (k_finalize) with the overlay on (ssd_gpu_set_overlay), on 1024 device-resident
1024 x 768 vertex frames generated on the device. k_finalize projects every step corner of every frame into the overlay, through the
pin-hole or through the lens of the call. Arms, alternated round by round in one process:
    plain-pinhole   plain call, no lens                 plain-lens   plain call, Brown-Conrady lens (ssd_gpu_set_distortion)
    cameras-pinhole camera call, four pin-hole cameras  cameras-lens camera call, four cameras of mixed lenses (pin-hole, BC, IBC)
Each value is the median over --rounds of the finalize stage's summed device time (SSD_FLAG_STAGE_TIMING) over the call's chunks.
Run it once per build (SSD_GPU_LIB selects the library) to compare them. One JSON line per arm; --out also appends them to a file.
    python tools/overlay_finalize_bench.py [--frames 1024] [--rounds 7] [--tag NAME] [--out profiles/process_call/b200_finalize.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import stair_step_detector_b200 as S  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=1024)
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--tag", default=os.environ.get("SSD_GPU_LIB", "this build"))
ap.add_argument("--out", default=None)
args = ap.parse_args()
W, H = 1024, 768
N, F = W * H, args.frames
BC = S.make_distortion(A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
IBC = S.make_distortion(A.DISTORTION_INVERSE_BROWN_CONRADY, (-0.11, 0.06, -0.0012, 0.0018, -0.02))
PIN = S.make_distortion(A.DISTORTION_NONE)

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
cfg, xf, cam = S.default_config(W, H), S.scene_transform(base), S.scene_camera(base)
cof = np.arange(F, dtype=np.int32) % 4
with S.Detector(cfg, xf, max_frames=F) as det:
    d_xyz = det.malloc(F * N * 12)
    det.synth_frames(base, 1, 0, F, 3, 8, d_xyz)
    det.set_overlay(np.array(cam.a_inv[:]).reshape(3, 3), S.scene_intrinsics(base))

    def run(arm):
        if arm.startswith("plain"):
            det.set_distortion(BC if arm == "plain-lens" else None)
            det.process_device(d_xyz, F, A.FLAG_STAGE_TIMING)
        else:
            det.set_cameras([cam] * 4, [PIN] * 4 if arm == "cameras-pinhole" else [PIN, BC, IBC, BC])
            det.process_cameras_device(d_xyz, cof, F, A.FLAG_STAGE_TIMING)
        return det.stage_times()["finalize"][0]

    arms = ["plain-pinhole", "plain-lens", "cameras-pinhole", "cameras-lens"]
    for arm in arms:  # warm-up: module load, ray tables, staging
        run(arm)
    ms = {arm: [] for arm in arms}
    for r in range(args.rounds):
        for arm in (arms if r % 2 == 0 else arms[::-1]):
            ms[arm].append(run(arm))
    det.free(d_xyz)
out_f = open(args.out, "a") if args.out else None
for arm in arms:
    line = json.dumps({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "build": args.tag, "arm": arm, "frames": F,
                       "size": f"{W}x{H}", "finalize_ms_median": round(float(np.median(ms[arm])), 4),
                       "finalize_ms": [round(v, 4) for v in ms[arm]]})
    print(line, flush=True)
    if out_f:
        out_f.write(line + "\n")
