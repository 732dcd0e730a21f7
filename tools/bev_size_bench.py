"""GPU box: a BEV size of its own (ssd_gpu_create_bev) against the frame-size BEV, on device-resident synthetic frames generated on
the device. Two workloads, each with two arms alternated round by round in one process (median of --rounds):
    (1) --frames 1024x768 z16 frames (bench.py configs[2]'s scene), BEV 1024x768 (the default) against BEV 640x480
    (2) 64 4096x3072 vertex frames (bench.py configs[4]), BEV 4096x3072 (the default) against BEV 1024x768; also the chain's
        per-stage device times on one stream (SSD_FLAG_STAGE_TIMING | SSD_FLAG_SINGLE_STREAM)
Every arm reports the chunk size its context chose and the mean number of steps it detects. Card name and power limit are read in
the same process.
    python tools/bev_size_bench.py [--frames 4096] [--rounds 5] [--out profiles/bev_size/b200_bev_size_bench.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import stair_step_detector_b200 as S  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()
out_f = open(args.out, "a") if args.out else None
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out_f:
        out_f.write(line + "\n")
        out_f.flush()


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": args.frames, "rounds": args.rounds})


def compare(name, dets, run, n, stage_cfg=None):
    """alternate the arms of dets {arm: Detector} over --rounds, report medians, chunk sizes and mean steps"""
    arms = list(dets)
    steps = {}
    for a in arms:
        run(dets[a])
        steps[a] = dets[a].n_steps_all(n)
    times = {a: [] for a in arms}
    for r in range(args.rounds):
        for a in (arms if r % 2 == 0 else arms[::-1]):
            run(dets[a])
            times[a].append(dets[a].timing().total_ms)
    med = {a: float(np.median(v)) for a, v in times.items()}
    for a in arms:
        emit({"workload": name, "arm": a, "bev": "%dx%d" % dets[a].bev, "ms_median": round(med[a], 3), "ms_all": [round(t, 3) for t in times[a]],
              "frames_per_s": round(n / med[a] * 1e3, 1), "vs_default_pct": round(100.0 * (med[a] / med[arms[0]] - 1.0), 2),
              "chunk_frames": dets[a].chunk_frames, "mean_steps": float(steps[a].mean())})
    if stage_cfg:
        for a in arms:
            run(dets[a], A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM)
            st = dets[a].stage_times()
            emit({"workload": name, "arm": a, "single_stream_stage_ms": {k: round(v[0], 3) for k, v in st.items()},
                  "sum_ms": round(sum(v[0] for v in st.values()), 3)})


# (1) 1024x768 z16 frames, device resident
W, H, F = 1024, 768, args.frames
cfg = S.default_config(W, H)
sc = S.default_scene(W, H, **NOISY)
xf, intr = S.scene_transform(sc), S.scene_intrinsics(sc)
dets = {"bev_1024x768": S.Detector(cfg, xf, max_frames=F), "bev_640x480": S.Detector(cfg, xf, max_frames=F, bev=(640, 480))}
z16 = torch.empty(F * W * H, dtype=torch.int16, device="cuda")
dets["bev_1024x768"].synth_frames(sc, 1, 0, F, 3, 8, None, z16.data_ptr())
torch.cuda.synchronize()
compare("1024x768_z16", dets, lambda d, fl=0: d.process_depth_device(z16.data_ptr(), intr, F), F)
for d in dets.values():
    d.close()
del z16
torch.cuda.empty_cache()

# (2) 64 4096x3072 vertex frames (bench.py configs[4])
W, H, F = 4096, 3072, 64
cfg = S.default_config(W, H, y_max=3.7, z_max=2.3)
sc = S.default_scene(W, H, n_steps=12, riser=0.17, tread=0.26, cam_height=3.2, cam_pitch_deg=48.0, first_riser_y=0.5, **NOISY)
xf = S.scene_transform(sc)
dets = {"bev_4096x3072": S.Detector(cfg, xf, max_frames=F), "bev_1024x768": S.Detector(cfg, xf, max_frames=F, bev=(1024, 768))}
xyz = torch.empty(F * W * H * 3, dtype=torch.float32, device="cuda")
dets["bev_4096x3072"].synth_frames(sc, 1, 0, F, 12, 12, xyz.data_ptr(), None)
torch.cuda.synchronize()
compare("4096x3072_vertices", dets, lambda d, fl=0: d.process_device(xyz.data_ptr(), F, fl), F, stage_cfg=True)
for d in dets.values():
    d.close()
del xyz
torch.cuda.empty_cache()

# the chunk each BEV size chooses for a large device-resident batch of 4096x3072 frames: the BEV bitmaps (2 streams x 32 slots per
# frame) are held to 8 GB
for bev in ((4096, 3072), (1024, 768)):
    with S.Detector(cfg, xf, max_frames=1024, bev=bev) as d:
        emit({"workload": "4096x3072_chunk", "bev": "%dx%d" % bev, "max_frames": 1024, "chunk_frames": d.chunk_frames})
