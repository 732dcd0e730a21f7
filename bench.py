#!/usr/bin/env python
"""bench.py -- headline benchmark of the stair-step geometry hot path (BASELINE.json metric:
Mpoints/s and frames/s at 1024x768 on 1/2/4/8 B200, % of HBM roofline).

    python bench.py --gpus N --steps K --warmup W          # our CUDA path
    python bench.py --impl reference ...                   # the reference's own CPU code on the host cores
    python bench.py --config {0..4}                        # another BASELINE.json config (default 2, the metric's)
    python bench.py --scaling weak                         # 4096 frames PER GPU instead of 4096/G (default: strong)
    python bench.py --dump-outputs DIR                     # also write the last timed step's results to DIR/*.npy

A "step" is one pass of the whole chain (transform -> height-band labels -> per-step reductions -> Stairs
records on the host) over one batch of synthetic frames that is already resident in HBM. BASELINE.json configs[2]
(the config the metric is quoted on): a batch of 4096 frames of 3-8-step staircases with L515-class noise, SHARDED
over the GPUs -- rank r of G owns the contiguous frames sharding.frame_range(r, G, 4096) (strong scaling; SURVEY.md
8(e)). One process per GPU under torchrun; no collective on the data path (frames are independent), the per-frame
step counts are gathered to rank 0; the timed region is bracketed by barrier + synchronize and the MAX over ranks is
reported. Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only: nothing is cached in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ALGO_BYTES_PER_POINT = 13  # 12 B packed f32 xyz read + 1 B u8 label written (SURVEY.md 8(d))
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
BASE_SEED = 20261017
DUMP_SEED = 7  # which frames / pixels --dump-outputs samples when the results exceed its budget
DUMP_MAX_FRAMES = 4096  # per-frame results (steps, plateaus, histograms, frame info) of at most this many frames
DUMP_LABEL_VALUES = 1 << 21  # labels: at most this many (frame, pixel) values (all dumped arrays stay below 64 MB)
# BASELINE.json configs (SURVEY.md 8(d)). frames: the batch of the config (global); steps: range of the staircase's
# step count per frame, (0, 0) = the base scene itself.
CONFIGS = {
    0: dict(name="configs[0]: single clean synthetic 1024x768 L515-resolution frame of a 3-step staircase", size=(1024, 768), cfg={}, scene={},
            frames=1, steps=(0, 0)),
    1: dict(name="configs[1]: the same 3-step staircase with L515 depth noise (sigma 2.5 mm), 3 % zero-depth pixels and 3 holes, 1 frame",
            size=(1024, 768), cfg={}, scene=dict(**NOISY), frames=1, steps=(0, 0)),
    2: dict(name="configs[2]: batch of 4096 synthetic 1024x768 L515-resolution frames of 3-8-step staircases (depth noise sigma 2.5 mm, "
                 "3 % dropouts, 3 holes), device-resident, sharded over the GPUs", size=(1024, 768), cfg={}, scene=dict(**NOISY),
            frames=4096, steps=(3, 8)),
    3: dict(name="configs[3]: descending-stairs view (image rotated 180 degrees) with 2 occluders and partial steps, batch of 1024 frames",
            size=(1024, 768), cfg={}, scene=dict(rotate180=1, n_occluders=2, **NOISY), frames=1024, steps=(3, 8)),
    4: dict(name="configs[4]: high-resolution 4096x3072 frames with 12 steps (measuring range extended to y < 3.7 m, z < 2.3 m: 241 height "
                 "bins), batch of 64 frames", size=(4096, 3072), cfg=dict(y_max=3.7, z_max=2.3),
            scene=dict(n_steps=12, riser=0.17, tread=0.26, cam_height=3.2, cam_pitch_deg=48.0, first_riser_y=0.5, **NOISY), frames=64,
            steps=(12, 12)),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md recipe). NVML in a sampling thread
    (every 5 ms: the timed region is a few hundred ms); `nvidia-smi -lms` as the fallback when pynvml is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, device):
        self.device, self.proc, self.path, self.thread = device, None, None, None
        self.sm, self.power, self.bits, self.smax = [], [], 0, None

    def _nvml_loop(self):
        import pynvml as nv
        h = self.handle
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                self.bits |= int(get(h))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            self.handle = nv.nvmlDeviceGetHandleByIndex(self.device)
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
            self.stop_flag = False
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=self.out, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if not self.sm:
                return {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": ["no samples"]}
            return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.smax, "power_w_max": max(self.power), "samples": len(self.sm),
                    "source": "nvml", "reasons": sorted(name for bit, name in self.REASONS if self.bits & bit)}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        sm, smax, reasons, power = [], [], set(), []
        with open(self.path) as f:
            for line in f:
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    smax.append(float(c[2]))
                    power.append(float(c[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power), "samples": len(sm),
                "source": "nvidia-smi", "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def reference_config(A, w, h, **kw):
    """ssd_gpu_config with the reference's defaults (configuration.h:27-52) WITHOUT touching the product library: the
    reference arm maps only libssd_scene.so (input source) and oracle/_ref (the reference itself)."""
    c = A.Config()
    c.width, c.height = w, h
    c.x_min, c.x_max, c.y_min, c.y_max, c.z_min, c.z_max = -0.6, 0.6, 0.1, 1.3, -0.1, 1.1
    c.height_interval, c.min_height_above_ground, c.min_step_depth, c.min_peak_points = 0.01, 0.05, 0.1, 2000
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def cpu_reference_leg(ref, xyz_sample, xf, threads, target_cpu_seconds, N):
    """The reference's own Pointcloud::process (oracle/_ref, compiled from the reference sources by path) on a bounded sample
    of the workload, frame-parallel over `threads` host threads (threading in the harness, not in reference code)."""
    import helpers
    nf = xyz_sample.shape[0]
    secs = C.c_double()
    failed = C.c_int()
    ref.ssd_ref_process_timed(C.byref(xf), helpers.ptr(xyz_sample), min(nf, threads), threads, 1, C.byref(secs), C.byref(failed))  # warm
    per_frame = max(secs.value * threads / max(1, min(nf, threads)), 1e-3)
    repeat = max(1, int(round(target_cpu_seconds / (per_frame * nf))))
    rc = ref.ssd_ref_process_timed(C.byref(xf), helpers.ptr(xyz_sample), nf, threads, repeat, C.byref(secs), C.byref(failed))
    assert rc == 0
    frames = nf * repeat
    t = secs.value
    return {"value": frames * N / t / 1e6, "unit": "Mpoints/s", "frames_per_s": frames / t, "cores": threads, "kind": "reference",
            "host_cores": os.cpu_count(),
            "sample": f"{nf} frames of the same synthetic batch x{repeat} passes, Pointcloud::process per frame, "
                      f"{threads} host thread(s) (threading in the harness; shim 3x3 close instead of OpenCV's)",
            "seconds": t, "failed_frames": failed.value}


def cpu_port_leg(cfg, xyz_sample, xf, N):
    """fallback when oracle/_ref is absent: the C restatement (oracle/ssd_oracle.c), one thread"""
    import helpers
    orc = helpers.load_oracle()
    nf = xyz_sample.shape[0]
    t0 = time.perf_counter()
    rc = orc.ssd_oracle_process_batch(C.byref(cfg), C.byref(xf), helpers.ptr(xyz_sample), nf, None)
    t = time.perf_counter() - t0
    assert rc == 0
    return {"value": nf * N / t / 1e6, "unit": "Mpoints/s", "frames_per_s": nf / t, "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
            "sample": f"{nf} frames of the same synthetic batch, C restatement of Pointcloud::process, 1 thread", "seconds": t, "failed_frames": 0}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation on the host cores, all threads, on a bounded sample of the
    same config. Loads libssd_scene.so (input) and oracle/_ref/libssd_ref_*.so (the reference) -- NOT the product library."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    import helpers
    import stair_step_detector_b200 as S
    from stair_step_detector_b200 import _abi as A
    conf = CONFIGS[args.config]
    W, H = conf["size"]
    N = W * H
    cfg = reference_config(A, W, H, **conf["cfg"])
    base = S.default_scene(W, H, **conf["scene"])
    ref = helpers.load_ref(cfg)
    nf = {0: 8, 1: 8, 2: 64, 3: 64, 4: 8}[args.config]
    smin, smax = conf["steps"]
    scenes = [S.randomize_scene(base, BASE_SEED, i, smin, smax) if smin else base for i in range(nf)]
    xyz = np.stack([S.deproject_host(sc, S.synth_depth_host(sc)) for sc in scenes]).reshape(nf, N, 3)
    threads = os.cpu_count() or 1
    if ref is not None:
        w9, c9 = (C.c_double * 9)(), (C.c_double * 9)()
        S.scene_lib().ssd_scene_calibration_points(C.byref(base), w9, c9)
        xf = A.Transform()
        assert ref.ssd_ref_make_transform(w9, c9, C.byref(xf)) == 0  # the reference's own GeometricTransformation
    else:
        xf = S.scene_transform(base)  # (the port needs the product's host-side transformation builder)
    res = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_leg(ref, xyz, xf, threads, 0.0, N) if ref is not None else cpu_port_leg(cfg, xyz, xf, N)
        if i >= args.warmup:
            res.append(r)
    t = sum(r["seconds"] for r in res)
    frames = nf * len(res)
    val = frames * N / t / 1e6
    cb = dict(res[-1])
    cb["value"] = val
    line = {"impl": "reference", "metric": "Mpoints/s", "value": val, "unit": "Mpoints/s", "frames_per_s": frames / t,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / len(res),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": conf["name"] + f" -- bounded sample: {nf} frames per step", "width": W, "height": H, "frames_per_step": nf,
                       "config_index": args.config},
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def gpu_frame_result(det, A, frame):
    """one frame of the last call as a helpers.FrameResult"""
    import helpers
    info = det.frame_info(frame)
    plats, _ = det.plateaus(frame)
    steps = (A.Step * A.MAX_STEPS)()
    n = C.c_int()
    det._ck(det._l.ssd_gpu_get_steps(det._h, frame, steps, A.MAX_STEPS, C.byref(n), None), "get_steps")
    hist = np.zeros(A.MAX_BINS, np.uint32)
    hist[:info.n_bins] = det.histogram(frame)
    return helpers._collect(det.labels(frame), hist, info, plats, steps, det.line(frame))


def parity_block(det, A, cfg, xf, ref, xyz_sample):
    """BASELINE.md 4: parity checked on the benchmarked frames in the same run. The first frames of the timed batch, as the
    GPU left them after the last timed step, against the compiled reference (oracle/_ref) run on the same vertices."""
    import helpers
    checker = "reference (oracle/_ref: the reference's translation units compiled by path)"
    orc = None
    if ref is None:
        orc = helpers.load_oracle()
        checker = "port (oracle/ssd_oracle.c)"
    lab_bad = hist_bad = count_bad = line_bad = status_bad = 0
    max_err = 0.0
    other = []
    for f in range(xyz_sample.shape[0]):
        g = gpu_frame_result(det, A, f)
        o = helpers.ref_process(ref, cfg, xf, xyz_sample[f]) if ref is not None else helpers.oracle_process(orc, cfg, xf, xyz_sample[f])
        lab_bad += int((g.labels != o.labels).sum())
        hist_bad += int(not np.array_equal(g.hist, o.hist))
        # (the harness around the compiled reference raises only NO_STEPS / DEGENERATE_QUAD; the quirk bits' effects -- all-zero
        #  ground step, NaN mean, wrapped plateaus -- are in the compared results themselves)
        smask = 0x3 if ref is not None else 0xffffffff
        status_bad += int((g.info["status"] & smask) != (o.info["status"] & smask))
        if len(g.steps) != len(o.steps):
            count_bad += 1
        else:
            for s, t in zip(g.steps, o.steps):
                if np.isnan(s["height"]) != np.isnan(t["height"]):
                    max_err = float("inf")
                elif not np.isnan(s["height"]):
                    max_err = max(max_err, abs(s["height"] - t["height"]))
                max_err = max(max_err, float(np.abs(s["quad"] - t["quad"]).max()))
        if o.line is not None and g.line != o.line:
            line_bad += 1  # (3 printed decimals: a height within 1e-6 m of a rounding boundary can print differently)
        bad = helpers.compare_results(o, g, tol=1e-4)
        if bad:
            other.append((f, bad[:3]))
    return {"frames": int(xyz_sample.shape[0]), "checker": checker, "label_mismatches": lab_bad, "histogram_mismatch_frames": hist_bad,
            "status_mismatch_frames": status_bad, "step_count_mismatch_frames": count_bad, "max_step_err_m": max_err,
            "tolerance_m": 1e-4, "serialized_line_mismatches": line_bad, "other_mismatches": other[:4],
            "ok": lab_bad == 0 and hist_bad == 0 and count_bad == 0 and status_bad == 0 and max_err < 1e-4 and not other}


def dump_outputs(det, A, out_dir, first, frames, N):
    """What the timed call hands its caller for each frame (ssd_gpu_get_frame_info / _get_steps / _get_plateaus /
    _get_histogram / _get_labels), as float64 / float32 .npy files under out_dir. Frames beyond DUMP_MAX_FRAMES and labels
    beyond DUMP_LABEL_VALUES are a fixed seeded sample (same arguments, same sample); frame_index holds the global frame ids."""
    rng = np.random.default_rng(DUMP_SEED)
    sel = np.arange(frames) if frames <= DUMP_MAX_FRAMES else np.sort(rng.choice(frames, DUMP_MAX_FRAMES, replace=False))
    n = len(sel)
    info = np.zeros((n, len(A.FrameInfo._fields_)), np.float64)
    steps = np.zeros((n, A.MAX_STEPS, 9), np.float64)  # height, then the quadrilateral's 4 corners (x, y); zero past n_steps
    pfields = ("height", "hmin", "hmax", "n_points", "valid", "outlined", "n_in_quad", "quad_status", "mean_z")
    plats = np.zeros((n, A.MAX_PLATEAUS, len(pfields) + 8), np.float64)  # the fields above, then quad_world; zero past n_plateaus
    hist = np.zeros((n, A.MAX_BINS), np.float32)  # zero past n_bins
    for i, f in enumerate(sel):
        fi = det.frame_info(int(f))
        info[i] = [getattr(fi, k) for k, _ in A.FrameInfo._fields_]
        st, _ = det.steps(int(f))
        for k, (h, q) in enumerate(st):
            steps[i, k, 0], steps[i, k, 1:] = h, np.asarray(q).ravel()
        pl, K = det.plateaus(int(f))
        p = np.ctypeslib.as_array(pl)[:K]
        plats[i, :K, :len(pfields)] = np.stack([p[k].astype(np.float64) for k in pfields], 1)
        plats[i, :K, len(pfields):] = p["quad_world"].reshape(K, 8)
        hg = det.histogram(int(f))
        hist[i, :len(hg)] = hg
    n_lab = max(1, min(n, DUMP_LABEL_VALUES // N))
    lab_frames = sel[np.sort(rng.choice(n, n_lab, replace=False))]
    pix = np.arange(N) if N <= DUMP_LABEL_VALUES else np.sort(rng.choice(N, DUMP_LABEL_VALUES, replace=False))
    pix_type = np.float32 if N <= 1 << 24 else np.float64  # float32 holds every pixel index below 2^24 exactly
    labels = np.stack([det.labels(int(f))[pix] for f in lab_frames]).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"frame_index": (first + sel).astype(np.float64), "frame_info": info, "steps": steps, "plateaus": plats, "histogram": hist,
              "labels": labels, "labels_frame_index": (first + lab_frames).astype(np.float64), "labels_pixel_index": pix.astype(pix_type)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def latency_block(S, A, conf, device, reps=60):
    """The reference's real use is one frame per call (detect-stairs.cpp:36-42): per-call latency of one frame through the C ABI,
    device-resident vertices / host vertices / host z16 depth frame (pinned). Median and min of `reps` calls, CUDA events."""
    W, H = conf["size"]
    N = W * H
    cfg = S.default_config(W, H, **conf["cfg"])
    base = S.default_scene(W, H, **conf["scene"])
    xf = S.scene_transform(base)
    intr = S.scene_intrinsics(base)
    out = {}
    with S.Detector(cfg, xf, device=device, max_frames=1) as det:
        d_xyz = det.malloc(N * 12)
        d_depth = det.malloc(N * 2)
        det.synth_frames(base, BASE_SEED, 0, 1, 0, 0, d_xyz, d_depth)
        h_xyz, hx = S.pinned_empty((1, N, 3), np.float32)
        h_z, hz = S.pinned_empty((1, N), np.uint16)
        det.d2h(h_xyz, d_xyz)
        det.d2h(h_z, d_depth)
        for name, fn in (("device_vertices", lambda: det.process_device(d_xyz, 1)), ("host_vertices", lambda: det.process_host_ptr(hx, 1)),
                         ("host_depth_z16", lambda: det.process_depth_host_ptr(hz, intr, 1))):
            for _ in range(5):
                fn()
            ts, wall = [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                wall.append((time.perf_counter() - t0) * 1e3)
                ts.append(det.timing().total_ms)
            out[name] = {"ms_median": statistics.median(ts), "ms_min": min(ts), "wall_ms_median": statistics.median(wall),
                         "launches_per_call": det.timing().n_launches}
        out["steps_found"] = int(det.n_steps_all(1)[0])
        S.free_pinned(hx)
        S.free_pinned(hz)
        det.free(d_xyz)
        det.free(d_depth)
    out["note"] = "one frame per call: ms_* = CUDA events from the first copy / kernel to the results in pinned host memory; wall_ms = the blocking C-ABI call"
    return out


def run_ours(args):
    rank, world, local = dist_env()
    import stair_step_detector_b200 as S
    from stair_step_detector_b200 import _abi as A
    from stair_step_detector_b200 import sharding

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier_sync():
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    if world > 1:
        # one process per GPU: run on the CPUs (and allocate the pinned host buffers on the memory) next to that GPU
        try:
            import pynvml as nv
            nv.nvmlInit()
            nv.nvmlDeviceSetCpuAffinity(nv.nvmlDeviceGetHandleByIndex(local))
        except Exception:
            pass

    conf = CONFIGS[args.config]
    W, H = conf["size"]
    N = W * H
    total_cfg = args.frames if args.frames > 0 else conf["frames"]
    if args.scaling == "strong":
        total_frames = total_cfg
        first, frames = sharding.frame_range(rank, world, total_frames)  # contiguous shard of the config's batch
    else:
        frames = total_cfg
        total_frames = frames * world
        first = rank * frames
    frames = max(frames, 1)
    smin, smax = conf["steps"]
    cfg = S.default_config(W, H, **conf["cfg"])
    base = S.default_scene(W, H, **conf["scene"])
    xf = S.scene_transform(base)
    det = S.Detector(cfg, xf, device=local, max_frames=frames)
    d_xyz = det.malloc(frames * N * 12)
    # global frame id = first + i: the same frame whatever the number of GPUs (camera pose fixed by the calibration, staircase
    # geometry varies per frame)
    det.synth_frames(base, BASE_SEED, first, frames, smin, smax, d_xyz)

    # ---- warm-up ----
    for _ in range(max(args.warmup, 3)):
        det.process_device(d_xyz, frames)

    # ---- timed: device-resident input -> Stairs records on the host ----
    sampler = ClockSampler(local)
    barrier_sync()
    sampler.start()
    t_wall0 = time.perf_counter()
    dev_ms, launches = [], 0
    for _ in range(args.steps):
        det.process_device(d_xyz, frames)
        t = det.timing()
        dev_ms.append(t.total_ms)
        launches += t.n_launches
    barrier_sync()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(det, A, args.dump_outputs, first, frames, N)
    my_ms = sum(dev_ms)
    step_counts = det.n_steps_all(frames)
    n_steps_found = int(step_counts.sum())
    st = det.stats()
    filter_stats = {"n_points": int(st.n_points), "n_exact_fallback": int(st.n_exact_fallback), "n_quad_fast": int(st.n_quad_fast),
                    "n_quad_exact": int(st.n_quad_exact), "n_bev_exact": int(st.n_bev_exact),
                    "exact_fallback_fraction": st.n_exact_fallback / max(1, st.n_points),
                    "note": "points within the proven f32 error bound of a range / height-bin threshold, a quadrilateral edge or a BEV pixel "
                            "boundary were decided by the exact double chain (bit-identical results either way); per GPU, last timed step"}

    # ---- parity on the benchmarked frames, same run (rank 0) ----
    parity = None
    ref = None
    n_par = min(args.parity_frames, frames) if rank == 0 else 0
    if n_par > 0:
        import helpers
        ref = helpers.load_ref(cfg)
        par_xyz = np.empty((n_par, N, 3), np.float32)
        det.d2h(par_xyz, d_xyz)
        parity = parity_block(det, A, cfg, xf, ref, par_xyz)

    # ---- roofline of the dominant kernel: per-launch CUDA events on the launching streams ----
    # (one extra pass right after the timed region, chunks serialised on one stream so that an event bracket is the
    #  kernel's own duration and not its duration while sharing the GPU with the other streams' kernels)
    det.process_device(d_xyz, frames, flags=A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM)
    stages = det.stage_times()
    stage_total = det.timing().total_ms
    det.process_device(d_xyz, frames, flags=A.FLAG_STAGE_TIMING)
    stages_overlapped = det.stage_times()

    # ---- e2e: the reference-facing call with HOST buffers (pinned), host->device copies and the device->host read of the
    # results inside the timed region. The reference's process() receives the z16 DEPTH FRAME (Camera::DepthFrame,
    # pointcloud.cpp:608,138), so that is the host buffer of the headline e2e: 2 bytes per pixel cross PCIe and the
    # deprojection runs on the GPU (ssd_gpu_process_depth_host). The same through the packed-vertex entry point
    # (12 bytes per pixel, ssd_gpu_process_host) is reported next to it.
    intr = S.scene_intrinsics(base)
    e2e_total = min(args.e2e_frames, total_cfg)
    if args.scaling == "strong":
        _, e2e_frames = sharding.frame_range(rank, world, e2e_total)
    else:
        e2e_frames = e2e_total
    e2e_frames = max(1, min(e2e_frames, frames))
    d_depth = det.malloc(e2e_frames * N * 2)
    det.synth_frames(base, BASE_SEED, first, e2e_frames, smin, smax, None, d_depth)  # same frames as the device-resident batch
    h_depth, h_depth_handle = S.pinned_empty((e2e_frames, N), np.uint16)
    det.d2h(h_depth, d_depth)
    for _ in range(2):
        det.process_depth_host_ptr(h_depth_handle, intr, e2e_frames)
    e2e_steps_found = int(det.n_steps_all(e2e_frames).sum())
    barrier_sync()
    e2e_ms = []
    for _ in range(max(3, args.steps // 2)):
        det.process_depth_host_ptr(h_depth_handle, intr, e2e_frames)
        e2e_ms.append(det.timing().total_ms)
    barrier_sync()
    my_e2e = sum(e2e_ms) / len(e2e_ms)
    # the same call with a PAGEABLE host buffer (what a librealsense frame is unless the application registers it): the driver
    # stages the copies through its own pinned buffer
    p_frames = max(1, min(256, e2e_frames))
    h_pageable = np.array(h_depth[:p_frames], copy=True)
    det.process_depth_host(h_pageable, intr)
    pg_ms = []
    for _ in range(3):
        det.process_depth_host(h_pageable, intr)
        pg_ms.append(det.timing().total_ms)
    my_pg = sum(pg_ms) / len(pg_ms)
    del h_pageable
    # H2D-only ceiling: the same pinned buffer, copies only, all ranks at the same time
    barrier_sync()
    t0 = time.perf_counter()
    reps_h2d = 3
    for _ in range(reps_h2d):
        det.h2d(d_depth, h_depth)
    my_h2d_s = (time.perf_counter() - t0) / reps_h2d
    barrier_sync()
    det.free(d_depth)
    # the same depth frames already resident in HBM (no PCIe): what the fused deprojection buys on the device
    d_depth2 = det.malloc(e2e_frames * N * 2)
    det.h2d(d_depth2, h_depth)
    for _ in range(2):
        det.process_depth_device(d_depth2, intr, e2e_frames)
    dd_ms = []
    for _ in range(3):
        det.process_depth_device(d_depth2, intr, e2e_frames)
        dd_ms.append(det.timing().total_ms)
    det.free(d_depth2)
    my_dd = sum(dd_ms) / len(dd_ms)
    # packed vertices through PCIe
    v_frames = max(1, min(256 if W * H <= 1 << 20 else 8, e2e_frames))
    h_xyz, h_handle = S.pinned_empty((v_frames, N, 3), np.float32)
    det.d2h(h_xyz, d_xyz)
    det.process_host_ptr(h_handle, v_frames)
    v_ms = []
    for _ in range(3):
        det.process_host_ptr(h_handle, v_frames)
        v_ms.append(det.timing().total_ms)
    my_e2e_v = sum(v_ms) / len(v_ms)

    # ---- max over ranks; per-frame step counts gathered to rank 0 ----
    gathered_ok = None
    if dist is not None:
        (my_ms, my_e2e, wall_ms, my_e2e_v, my_dd, my_h2d_s), (launches, n_steps_found, e2e_frames_all, frames_all) = sharding.reduce_timing(
            dist, [my_ms, my_e2e, wall_ms, my_e2e_v, my_dd, my_h2d_s], [launches, n_steps_found, e2e_frames, frames], device=f"cuda:{local}")
        if frames * world == frames_all:  # equal shards: gather the per-frame results (step counts) in global frame order
            allc = sharding.gather_step_counts(dist, step_counts, device=f"cuda:{local}")
            gathered_ok = len(allc) == frames_all and sum(allc) == n_steps_found
    else:
        e2e_frames_all, frames_all = e2e_frames, frames

    if rank == 0:
        ms_per_step = my_ms / args.steps
        fps = frames_all / (ms_per_step * 1e-3)
        mpts = fps * N / 1e6
        peak, peak_src = peaks()
        k_ms, k_n = stages["transform_bin"]
        pts_per_launch = min(det.chunk_frames, frames) * N
        achieved = ALGO_BYTES_PER_POINT * frames * N / (k_ms * 1e-3) / 1e9 if k_n and k_ms > 0 else None
        chain_achieved = ALGO_BYTES_PER_POINT * (fps / world) * N / 1e9
        roofline = {"bound": "hbm", "kernel": "k_transform_bin", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak if achieved else None, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": ALGO_BYTES_PER_POINT * pts_per_launch, "launches_timed": k_n,
                    "avg_launch_ms": k_ms / k_n if k_n else None,
                    "chain": {"achieved": chain_achieved, "frac": chain_achieved / peak, "frac_of_nominal_8000": chain_achieved / 8000.0,
                              "note": "whole chain per GPU: 13 B/point x points/s"},
                    "stage_ms_sum": {k: v[0] for k, v in stages.items()}, "stage_total_ms": stage_total,
                    "stage_ms_sum_overlapped": {k: v[0] for k, v in stages_overlapped.items()},
                    "note": "per-launch CUDA events on the launching stream; chunks serialised on one stream for this pass "
                            "(the timed region overlaps chunks on several streams)"}
        traffic_file = os.path.join(ROOT, "profiles", "traffic_latest.json")
        if os.path.exists(traffic_file) and (W, H) == (1024, 768):
            try:
                with open(traffic_file) as f:
                    tj = json.load(f)
                per = tj["per_kernel"]
                # measured DRAM bytes per frame (one ncu --set full launch) scaled to this run's launch size
                roofline["traffic"] = per["k_transform_bin"]["bytes_per_frame"] * min(det.chunk_frames, frames)
                roofline["traffic_source"] = tj.get("source")
                roofline["chain"]["traffic_bytes_per_frame"] = {k: v["bytes_per_frame"] for k, v in per.items()}
            except Exception:
                pass
        if roofline["frac"] and roofline["frac"] > 1.0:
            roofline["note"] += ("; frac > 1: the peak is the driver's COPY bandwidth (equal read and write streams), "
                                 "this kernel reads 12 bytes for every byte it writes and a read-dominated stream runs faster than a copy")
        e2e_fps = e2e_frames_all / (my_e2e * 1e-3)
        h2d_gbs = e2e_frames_all * N * 2 / my_h2d_s / 1e9
        line = {"metric": "Mpoints/s", "value": mpts, "unit": "Mpoints/s", "frames_per_s": fps, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "wall_ms_per_step": wall_ms / args.steps,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f64 decisions (f32 filter with proven bounds, exact f64 fallback); per-step mean z as order-independent integer sums of f32 z",
                "data": "synthetic",
                "config": {"workload": conf["name"], "config_index": args.config, "width": W, "height": H,
                           "frames_per_gpu": frames, "global_frames": frames_all,
                           "chunk_frames": det.chunk_frames,
                           "parallelism": f"frames sharded over {world} GPU(s) ({args.scaling} scaling), no collective on the data path; "
                                          "per-frame step counts gathered to rank 0",
                           "cache": f"inputs larger than L2 ({frames * N * 12 / 1e9:.2f} GB of vertices per GPU per step)" if frames * N * 12 > 256e6
                                    else "inputs smaller than L2: single-frame latency config, nothing is flushed between calls",
                           "stairs_found": n_steps_found, "results_gathered_ok": gathered_ok},
                "clocks": clocks,
                "e2e": {"value": e2e_fps * N / 1e6, "unit": "Mpoints/s", "frames_per_s": e2e_fps, "frames_per_step": e2e_frames_all,
                        "ms_per_step": my_e2e, "h2d_bytes_per_step": e2e_frames_all * N * 2,
                        "d2h_bytes_per_step": e2e_frames_all * (32 + 72 * A.MAX_STEPS + 16), "stairs_found_rank0": e2e_steps_found,
                        "input": "z16 depth frames in pinned host memory (what the reference's Pointcloud::process receives), "
                                 "deprojected on the GPU",
                        "call": "ssd_gpu_process_depth_host",
                        "h2d_ceiling_gbs": h2d_gbs, "h2d_ceiling_frames_per_s": h2d_gbs * 1e9 / (N * 2),
                        "frac_of_h2d_ceiling": e2e_fps / (h2d_gbs * 1e9 / (N * 2)),
                        "h2d_ceiling_note": "the same pinned buffers, cudaMemcpy host->device only, all ranks at the same time (max over ranks)",
                        "pageable_host_buffer": {"frames_per_s": p_frames / (my_pg * 1e-3), "frames_per_step": p_frames, "ms_per_step": my_pg,
                                                 "note": "rank 0, same call, the z16 frames in ordinary (pageable) host memory"},
                        "device_resident_depth": {"value": e2e_frames_all / (my_dd * 1e-3) * N / 1e6, "unit": "Mpoints/s",
                                                  "frames_per_s": e2e_frames_all / (my_dd * 1e-3), "ms_per_step": my_dd,
                                                  "call": "ssd_gpu_process_depth_device (z16 frames in HBM, 2 B/point, deprojected "
                                                          "inside the point kernels: no PCIe in this figure)"},
                        "vertices": {"value": v_frames * world / (my_e2e_v * 1e-3) * N / 1e6, "unit": "Mpoints/s",
                                     "frames_per_s": v_frames * world / (my_e2e_v * 1e-3), "frames_per_step": v_frames * world,
                                     "ms_per_step": my_e2e_v, "h2d_bytes_per_step": v_frames * N * 12,
                                     "call": "ssd_gpu_process_host (packed f32 vertices in pinned host memory; PCIe-bound)"}},
                "gpu_launches": launches,
                "roofline": roofline,
                "filter_stats": filter_stats}
        if parity is not None:
            line["parity"] = parity
        if world == 1 and not args.no_cpu_baseline:
            sample = np.ascontiguousarray(h_xyz[:min(32, v_frames)])
            if ref is None:
                import helpers
                ref = helpers.load_ref(cfg)
            if ref is not None:
                line["cpu_baseline"] = cpu_reference_leg(ref, sample, xf, os.cpu_count() or 1, 15.0, N)
                # mode A (SURVEY.md 8(d)): how the reference actually runs -- one thread, one frame per call
                line["cpu_baseline_single_thread"] = cpu_reference_leg(ref, sample[:min(4, len(sample))], xf, 1, 5.0, N)
            else:
                line["cpu_baseline"] = cpu_port_leg(cfg, sample[:4], xf, N)
        if world == 1 and not args.no_latency:
            line["latency"] = latency_block(S, A, CONFIGS[1] if args.config == 2 else conf, local)
        emit(line)

    S.free_pinned(h_handle)
    S.free_pinned(h_depth_handle)
    det.free(d_xyz)
    det.close()
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on stdout at
    communicator creation): point fd 1 at stderr for the duration of the run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configs index (2: the metric's config)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the config's batch is sharded over the GPUs (4096/G frames each); weak: the whole batch per GPU")
    ap.add_argument("--frames", type=int, default=0, help="override the config's batch size (global for strong, per GPU for weak)")
    ap.add_argument("--e2e-frames", type=int, default=1024, help="frames of the host-input (e2e) leg (global for strong scaling)")
    ap.add_argument("--parity-frames", type=int, default=16, help="benchmarked frames checked against the reference in the same run (rank 0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's frames) to DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
