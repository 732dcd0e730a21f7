"""GPU box: device-resident z16 depth frames through the chain, deprojection inside the point kernels (SrcDepth), next to the
packed-vertex input.
    python tools/depth_bench.py --frames 2048"""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import stair_step_detector_b200 as S
from stair_step_detector_b200 import _abi as A

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=2048)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()
W, H = 1024, 768
N = W * H
cfg = S.default_config(W, H)
base = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
xf = S.scene_transform(base)
intr = S.scene_intrinsics(base)
det = S.Detector(cfg, xf, max_frames=args.frames)
d_xyz = det.malloc(args.frames * N * 12)
d_depth = det.malloc(args.frames * N * 2)
det.synth_frames(base, 1, 0, args.frames, 3, 8, d_xyz, d_depth)


def run(name, fn, flags_fn=None):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(args.reps):
        fn()
        ts.append(det.timing().total_ms)
    ms = min(ts)
    out = {"input": name, "frames": args.frames, "ms_best": round(ms, 3), "kfps": round(args.frames / ms, 2),
           "Gpoints_s": round(args.frames * N / ms / 1e6, 1), "steps": int(det.n_steps_all(args.frames).sum())}
    if flags_fn:
        flags_fn()
        out["serial_stage_ms"] = {k: round(v[0], 3) for k, v in det.stage_times().items()}
    print(json.dumps(out), flush=True)


run("packed vertices (12 B/point)", lambda: det.process_device(d_xyz, args.frames),
    lambda: det.process_device(d_xyz, args.frames, flags=A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM))
run("z16 depth (2 B/point), deprojected inside the point kernels", lambda: det.process_depth_device(d_depth, intr, args.frames))
