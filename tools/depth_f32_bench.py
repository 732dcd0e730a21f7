"""GPU box: float depth frames (ssd_gpu_process_depth_f32_*) against z16 and vertex input, 1024 x 768. The frames are generated on
the device; the float frames are converted from the z16 ones on the device (u16 -> f32 is exact), so every arm sees the same
scene. Arms, alternated round by round in one process, median of --rounds:
    z16       pin-hole z16, plain call                      f32       the same frames as float samples
    z16_bc    z16 frames rendered through a BC lens         f32_bc    the same frames as float samples
    vertices  the pin-hole frames as packed vertices (what the library's synthetic source deprojects)
(1) --frames device-resident frames per call; (2) per-kernel device time of each arm on one stream (torch.profiler);
(3) end to end from pinned host memory (--host-frames frames) for z16, f32 and vertices; (4) one-frame latency from pageable
host memory (median of --latency-calls calls). Card name and power limit are read in the same process.
    python tools/depth_f32_bench.py [--frames 4096] [--rounds 5] [--out profiles/depth_f32/b200_depth_f32_bench.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import stair_step_detector_b200 as S  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=4096)
ap.add_argument("--host-frames", type=int, default=512)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--latency-calls", type=int, default=200)
ap.add_argument("--out", default=None)
args = ap.parse_args()
W, H = 1024, 768
N, F, FH = W * H, args.frames, args.host_frames
BC = (A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
out_f = open(args.out, "a") if args.out else None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out_f:
        out_f.write(line + "\n")
        out_f.flush()


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": F, "host_frames": FH, "size": f"{W}x{H}",
      "bytes_per_pixel": {"z16": 2, "f32": 4, "vertices": 12}})
cfg = S.default_config(W, H)


def scene(lens):
    s = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
    if lens:
        s.distortion_model = lens[0]
        for i, c in enumerate(lens[1]):
            s.coeffs[i] = c
    return s


def to_f32(z16):
    """u16 -> f32 on the device, in slices (int16 storage read as unsigned)"""
    out = torch.empty(z16.numel(), dtype=torch.float32, device="cuda")
    step = 64 * N
    for i in range(0, z16.numel(), step):
        out[i:i + step] = (z16[i:i + step].to(torch.int32) & 0xffff).to(torch.float32)
    return out


pin, bc = scene(None), scene(BC)
xf, intr = S.scene_transform(pin), S.scene_intrinsics(pin)
dets = {a: S.Detector(cfg, xf, max_frames=F) for a in ("z16", "f32", "z16_bc", "f32_bc", "vertices")}
z16 = torch.empty(F * N, dtype=torch.int16, device="cuda")
z16_bc = torch.empty(F * N, dtype=torch.int16, device="cuda")
xyz = torch.empty(F * N * 3, dtype=torch.float32, device="cuda")
dets["z16"].synth_frames(pin, 1, 0, F, 3, 8, xyz.data_ptr(), z16.data_ptr())
dets["z16_bc"].synth_frames(bc, 1, 0, F, 3, 8, None, z16_bc.data_ptr())
torch.cuda.synchronize()
f32, f32_bc = to_f32(z16), to_f32(z16_bc)
torch.cuda.synchronize()
for a in ("z16_bc", "f32_bc"):
    dets[a].set_distortion(S.scene_distortion(bc))
ptr = {"z16": z16.data_ptr(), "f32": f32.data_ptr(), "z16_bc": z16_bc.data_ptr(), "f32_bc": f32_bc.data_ptr(), "vertices": xyz.data_ptr()}


def run(det, arm, p, n):
    if arm.startswith("z16"):
        det.process_depth_device(p, intr, n)
    elif arm.startswith("f32"):
        det.process_depth_f32_device(p, intr, n)
    else:
        det.process_device(p, n)


arms = list(dets)
steps = {}
for a in arms:  # warm-up; the float arms detect what the z16 arms detect
    run(dets[a], a, ptr[a], F)
    steps[a] = dets[a].n_steps_all(F)
assert np.array_equal(steps["z16"], steps["f32"]) and np.array_equal(steps["z16_bc"], steps["f32_bc"]), "float and z16 disagree"
emit({"mean_steps": {a: float(steps[a].mean()) for a in arms}})
times = {a: [] for a in arms}
for r in range(args.rounds):
    for a in (arms if r % 2 == 0 else arms[::-1]):
        run(dets[a], a, ptr[a], F)
        times[a].append(dets[a].timing().total_ms)
med = {a: float(np.median(v)) for a, v in times.items()}
for a in arms:
    emit({"device_resident": a, "ms_median": round(med[a], 3), "ms_all": [round(t, 3) for t in times[a]], "kfps": round(F / med[a], 2),
          "vs_z16_pct": round(100.0 * (med[a] / med["z16_bc" if a.endswith("_bc") else "z16"] - 1.0), 2)})

# per-kernel device time, one chunk stream (torch.profiler: CUPTI sees the library's launches)
try:
    from torch.profiler import ProfilerActivity, profile
    os.environ["SSD_GPU_STREAMS"] = "1"
    for a in arms:
        d1 = S.Detector(cfg, xf, max_frames=F)
        if a.endswith("_bc"):
            d1.set_distortion(S.scene_distortion(bc))
        run(d1, a, ptr[a], F)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(d1, a, ptr[a], F)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and e.name.startswith(("void k_", "k_")):
                name = e.name.split("(")[0].replace("void ", "").split("<")[0]
                per[name] = per.get(name, 0.0) + e.device_time / 1e3
        emit({"serial_kernels": a, "kernel_ms": {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])},
              "sum_ms": round(sum(per.values()), 3)})
        d1.close()
    del os.environ["SSD_GPU_STREAMS"]
except Exception as ex:  # a diagnosis, not a result: report and go on
    emit({"profiler": "failed", "error": repr(ex)})

# end to end from pinned host memory
hz, p1 = S.pinned_empty((FH, H, W), np.uint16)
hf, p2 = S.pinned_empty((FH, H, W), np.float32)
hx, p3 = S.pinned_empty((FH, H, W, 3), np.float32)
hz[:] = z16[:FH * N].cpu().numpy().view(np.uint16).reshape(FH, H, W)
hf[:] = f32[:FH * N].cpu().numpy().reshape(FH, H, W)
hx[:] = xyz[:FH * N * 3].cpu().numpy().reshape(FH, H, W, 3)
hosts = {"z16": lambda: dets["z16"].process_depth_host(hz, intr), "f32": lambda: dets["f32"].process_depth_f32_host(hf, intr),
         "vertices": lambda: dets["vertices"].process_host(hx)}
ht = {k: [] for k in hosts}
for fn in hosts.values():
    fn()
for r in range(args.rounds):
    for k in (list(hosts) if r % 2 == 0 else list(hosts)[::-1]):
        t0 = time.perf_counter()  # each call ends in a device synchronise
        hosts[k]()
        ht[k].append((time.perf_counter() - t0) * 1e3)
hm = {k: float(np.median(v)) for k, v in ht.items()}
for k in hosts:
    emit({"pinned_host": k, "ms_median": round(hm[k], 3), "ms_all": [round(t, 3) for t in ht[k]], "kfps": round(FH / hm[k], 2),
          "vs_z16_pct": round(100.0 * (hm[k] / hm["z16"] - 1.0), 2)})

# one-frame latency (pageable host frame, as a capture loop hands it over)
one = {"z16": np.ascontiguousarray(hz[0]), "f32": np.ascontiguousarray(hf[0]), "vertices": np.ascontiguousarray(hx[0])}
lat = {k: [] for k in one}
calls1 = {"z16": lambda: dets["z16"].process_depth_host(one["z16"], intr), "f32": lambda: dets["f32"].process_depth_f32_host(one["f32"], intr),
          "vertices": lambda: dets["vertices"].process_host(one["vertices"])}
for fn in calls1.values():
    for _ in range(10):
        fn()
for i in range(args.latency_calls):
    for k in (list(calls1) if i % 2 == 0 else list(calls1)[::-1]):
        t0 = time.perf_counter()
        calls1[k]()
        lat[k].append((time.perf_counter() - t0) * 1e6)
for k in calls1:
    emit({"one_frame_latency": k, "us_median": round(float(np.median(lat[k])), 1), "us_p90": round(float(np.percentile(lat[k], 90)), 1),
          "calls": args.latency_calls})
for p in (p1, p2, p3):
    S.free_pinned(p)
for d in dets.values():
    d.close()
