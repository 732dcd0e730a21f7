"""GPU box: cost of lens distortion (ssd_gpu_set_distortion / ssd_gpu_set_cameras_ex) on 4096 device-resident 1024 x 768 z16 frames
generated on the device. Arms, alternated round by round in one process:
    (a) pin-hole z16, plain call            (b) Brown-Conrady lens, plain call      (c) inverse Brown-Conrady lens, plain call
    (d) eight cameras of mixed lenses (pin-hole, BC, IBC) in one camera call
    (e) the workaround: ssd_gpu_deproject_device with the lens into a vertex array, then ssd_gpu_process_device, timed together
    (f) end to end from pinned host memory (--host-frames frames): lens z16, pin-hole z16 and vertex input
Each lens arm's frames are rendered through its own lens. Also the per-kernel device time of (a) and (b) (torch.profiler, one
stream) and the ray-table bytes. One JSON line per measurement; --out also appends them to a file.
    python tools/distortion_bench.py [--frames 4096] [--rounds 5] [--out profiles/distortion/b200.jsonl]"""
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
ap.add_argument("--host-frames", type=int, default=512)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()
W, H = 1024, 768
N, F, FH = W * H, args.frames, args.host_frames
BC = (A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
IBC = (A.DISTORTION_INVERSE_BROWN_CONRADY, (-0.11, 0.06, -0.0012, 0.0018, -0.02))
out_f = open(args.out, "a") if args.out else None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    if out_f:
        out_f.write(line + "\n")
        out_f.flush()


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
emit({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown", "frames": F, "host_frames": FH, "size": f"{W}x{H}",
      "ray_table_bytes": N * 8})

cfg = S.default_config(W, H)


def scene(lens):
    s = S.default_scene(W, H, noise_sigma=0.0025, dropout=0.03, n_holes=3)
    if lens:
        s.distortion_model = lens[0]
        for i, c in enumerate(lens[1]):
            s.coeffs[i] = c
    return s


scenes = {"a": scene(None), "b": scene(BC), "c": scene(IBC)}
xf = S.scene_transform(scenes["a"])
intr = S.scene_intrinsics(scenes["a"])
dets, z16 = {}, {}
for arm, sc in scenes.items():
    dets[arm] = S.Detector(cfg, xf, max_frames=F)
    z16[arm] = dets[arm].malloc(F * N * 2)
    dets[arm].synth_frames(sc, 1, 0, F, 3, 8, None, z16[arm])
    if arm != "a":
        dets[arm].set_distortion(S.scene_distortion(sc))
det_d = dets["a"]
cams = [S.scene_camera(scenes[k]) for k in "abcabcab"]
dists = [S.scene_distortion(scenes[k]) for k in "abcabcab"]
d_xyz = dets["b"].malloc(F * N * 12)


def call(arm):
    if arm in "abc":
        dets[arm].process_depth_device(z16[arm], intr, F)
        return dets[arm].timing().total_ms
    if arm == "d":
        if det_d.n_cameras != 8:
            det_d.set_cameras(cams, dists)
        det_d.process_depth_cameras_device(z16["b"], np.arange(F, dtype=np.int32) % 8, F)
        return det_d.timing().total_ms
    t0 = time.perf_counter()  # (e): both calls end in a device synchronise
    dets["b"].deproject_device(z16["b"], intr, F, d_xyz)
    dets["b"].process_device(d_xyz, F)
    return (time.perf_counter() - t0) * 1e3


arms = ["a", "b", "c", "d", "e"]
steps = {}
for arm in arms:  # warm-up, and the lens z16 path gives the workaround's results
    call(arm)
    steps[arm] = (dets["b"] if arm == "e" else det_d if arm == "d" else dets[arm]).n_steps_all(F)
assert np.array_equal(steps["b"], steps["e"]), "lens z16 and deprojected vertices disagree"
emit({"ray_tables": {a: dets[a].n_ray_tables for a in "abc"} | {"d": det_d.n_ray_tables}, "mean_steps": {a: float(steps[a].mean()) for a in arms}})
times = {a: [] for a in arms}
for r in range(args.rounds):
    for arm in (arms if r % 2 == 0 else arms[::-1]):
        times[arm].append(call(arm))
med = {a: float(np.median(v)) for a, v in times.items()}
for arm in arms:
    emit({"arm": arm, "ms_median": round(med[arm], 3), "ms_all": [round(t, 3) for t in times[arm]], "kfps": round(F / med[arm], 2),
          "vs_pinhole_pct": round(100.0 * (med[arm] / med["a"] - 1.0), 2)})

# per-kernel device time of (a) and (b), one chunk stream at a time (torch.profiler, CUPTI sees the library's launches)
try:
    import torch
    from torch.profiler import ProfilerActivity, profile
    os.environ["SSD_GPU_STREAMS"] = "1"
    for arm in ("a", "b"):
        d1 = S.Detector(cfg, xf, max_frames=F)
        if arm == "b":
            d1.set_distortion(S.scene_distortion(scenes["b"]))
        d1.process_depth_device(z16[arm], intr, F)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            d1.process_depth_device(z16[arm], intr, F)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and e.name.startswith(("void k_", "k_")):
                name = e.name.split("(")[0].replace("void ", "")
                per[name] = per.get(name, 0.0) + e.device_time / 1e3
        emit({"arm": arm, "serial_kernel_ms": {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])},
              "sum_ms": round(sum(per.values()), 3)})
        d1.close()
    del os.environ["SSD_GPU_STREAMS"]
except Exception as ex:  # the stage times are a diagnosis, not a result: report and go on
    emit({"profiler": "failed", "error": repr(ex)})

# (f) end to end from pinned host memory
dev = dets["b"]
hz_lens, p1 = S.pinned_empty((FH, H, W), np.uint16)
hz_pin, p2 = S.pinned_empty((FH, H, W), np.uint16)
hxyz, p3 = S.pinned_empty((FH, H, W, 3), np.float32)
dev.d2h(hz_lens, z16["b"])
dets["a"].d2h(hz_pin, z16["a"])
dev.deproject_device(z16["b"], intr, FH, d_xyz)
dev.d2h(hxyz, d_xyz)
hosts = {"lens_z16": lambda: dets["b"].process_depth_host(hz_lens, intr), "pinhole_z16": lambda: dets["a"].process_depth_host(hz_pin, intr),
         "lens_vertices": lambda: dets["b"].process_host(hxyz)}
ht = {k: [] for k in hosts}
for k, fn in hosts.items():
    fn()
for r in range(args.rounds):
    for k in (list(hosts) if r % 2 == 0 else list(hosts)[::-1]):
        t0 = time.perf_counter()
        hosts[k]()
        ht[k].append((time.perf_counter() - t0) * 1e3)
hm = {k: float(np.median(v)) for k, v in ht.items()}
for k in hosts:
    emit({"arm": "f", "input": k, "ms_median": round(hm[k], 3), "ms_all": [round(t, 3) for t in ht[k]], "kfps": round(FH / hm[k], 2),
          "vs_pinhole_z16_pct": round(100.0 * (hm[k] / hm["pinhole_z16"] - 1.0), 2)})
for p in (p1, p2, p3):
    S.free_pinned(p)
for arm, d in dets.items():
    d.free(z16[arm])
dets["b"].free(d_xyz)
for d in dets.values():
    d.close()
