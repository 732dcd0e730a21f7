"""Float depth frames (ssd_gpu_process_depth_f32_*, include/ssd_gpu.h): one float sample per pixel, deprojected as a z16 pixel with
the sample in place of (float)count. Two consequences carry the GPU tests:
  (a) depth_f32 = (float)z16 with the same intrinsics, or fl((float)z16 * unit) with depth_unit = 1, gives what the z16 call gives;
  (b) any float frame gives what vertex input gives on the vertices deprojected on the host by the same f32 operations.
Both are compared bit for bit on every getter: labels, histogram, plateaus, frame info, steps, status, overlay, vertical faces,
step labels, step surfaces, every ssd_gpu_stats counter and timing.n_launches."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A
from test_gpu_distortion import BC, IBC, NOISY, lens_scene, np_deproject

gpu = pytest.mark.gpu
f32 = np.float32
FUSE_MAX_FRAMES = 16  # SSD_FUSE_MAX_FRAMES (ssd_gpu.cu): larger chunks take the seven-launch route


def unit_one(sc):
    """a copy of scene sc whose depth unit is 1.0 (float samples in metres)"""
    c = type(sc).from_buffer_copy(sc)
    c.depth_unit = 1.0
    return c


def camera_with_unit(S, sc, unit):
    cam = S.scene_camera(sc)
    cam.intr.depth_unit = unit
    return cam


def intr_with_unit(S, sc, unit):
    intr = S.scene_intrinsics(sc)
    intr.depth_unit = unit
    return intr


def canon(x):
    """getter values with every float as its exact hex form (NaN compares equal to NaN)"""
    if isinstance(x, float):
        return x.hex()
    if isinstance(x, dict):
        return {k: canon(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [canon(v) for v in x]
    return x


def everything(S, det, n):
    """every result of the last call of det (all options on)"""
    frames = [(H.exact(H.gpu_result(det, f)), det.overlay(f).tobytes(), canon(det.vertical_faces(f)), det.step_labels(f).tobytes(),
               canon(det.step_surfaces(f))) for f in range(n)]
    return frames, bytes(det.stats()), det.timing().n_launches


def all_options(det, a_inv, intr):
    det.set_overlay(a_inv, intr)
    det.set_vertical_faces(True)
    det.set_step_labels(True)
    det.set_step_surfaces(True)


def camera_bases(S, w, h):
    """pin-hole, BC and IBC cameras of different poses"""
    d = S.default_scene(w, h)
    return [lens_scene(S, w, h, None, **NOISY),
            lens_scene(S, w, h, BC, **dict(NOISY, cam_pitch_deg=d.cam_pitch_deg + 4.0)),
            lens_scene(S, w, h, IBC, **dict(NOISY, cam_height=d.cam_height * 1.05))]


def camera_frames(S, bases, n, seed, distinct=6):
    """n frames, frame i of camera i % 3; `distinct` (a multiple of 3) are synthesised and repeat, each with its camera"""
    order = np.arange(n, dtype=np.int32) % len(bases)
    depth = [S.synth_depth_host(S.randomize_scene(bases[order[i]], seed, i, 3, 8)) for i in range(min(n, distinct))]
    return order, np.stack([depth[i % distinct] for i in range(n)])


# ---- host only ----
@pytest.mark.parametrize("lens", [None, BC, IBC], ids=["pinhole", "BC", "IBC"])
def test_float_deprojection_of_z16_is_the_host_deprojection(S, lens):
    """premise of (a) and (b): the numpy f32 deprojection of (float)z16, and of fl((float)z16 * unit) with unit 1, equals the scene
    library's host deprojection of the z16 frame bit for bit"""
    w, h = 640, 480
    sc = lens_scene(S, w, h, lens, **NOISY)
    depth = S.synth_depth_host(sc)
    want = S.deproject_host(sc, depth).tobytes()
    as_float = depth.astype(f32)
    assert np_deproject(sc, as_float, lens).tobytes() == want
    assert np_deproject(unit_one(sc), as_float * f32(sc.depth_unit), lens).tobytes() == want
    if lens is None:
        assert H.deproject_np(sc, as_float).tobytes() == want


def test_cpp_check_compiles(S, tmp_path):
    exe = str(tmp_path / "depth_f32_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "depth_f32_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    assert os.path.exists(exe)


# ---- GPU: (a) equality with the z16 call ----
@gpu
@pytest.mark.parametrize("n", [4, FUSE_MAX_FRAMES + 4], ids=["fused", "seven-launch"])
@pytest.mark.parametrize("size", [(640, 480), (848, 480), (1024, 768)])
def test_float_of_z16_equals_z16(S, monkeypatch, size, n):
    """(float)z16 and fl(z16 * unit) with unit 1 == the z16 call: plain calls (pin-hole and through a lens), a camera call over a
    pin-hole / BC / IBC table and a group call with a group larger than the host chunk; host and device input"""
    w, h = size
    monkeypatch.setenv("SSD_GPU_HOST_CHUNK_FRAMES", "2")
    bases = camera_bases(S, w, h)
    order, depth = camera_frames(S, bases, n, 40 + w)
    as_float = depth.astype(f32)
    metres = as_float * f32(bases[0].depth_unit)  # every base has the scene's depth unit
    assert all(b.depth_unit == bases[0].depth_unit for b in bases)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(bases[0])
    intr, intr1 = S.scene_intrinsics(bases[0]), intr_with_unit(S, bases[0], 1.0)
    cams = [S.scene_camera(b) for b in bases]
    cams1 = [camera_with_unit(S, b, 1.0) for b in bases]
    dists = [S.scene_distortion(b) for b in bases]
    groups = [3, 1] if n == 4 else [1, 5, 2, 3, 3, 3, 3]
    assert sum(groups) == n and max(groups) > 2
    with S.Detector(cfg, xf, max_frames=n) as det:
        all_options(det, a_inv, intr)
        d_z16, d_f, d_m = H.to_device(det, depth), H.to_device(det, as_float), H.to_device(det, metres)
        # each float call against the z16 call of the same input kind (host input runs in host chunks: other launch counts)
        plain = {"host": (lambda: det.process_depth_host(depth, intr),
                          {"": lambda: det.process_depth_f32_host(as_float, intr),
                           "unit 1": lambda: det.process_depth_f32_host(metres, intr1)}),
                 "device": (lambda: det.process_depth_device(d_z16, intr, n),
                            {"": lambda: det.process_depth_f32_device(d_f, intr, n),
                             "unit 1": lambda: det.process_depth_f32_device(d_m, intr1, n)})}
        cameras = {"host": (lambda: det.process_depth_cameras_host(depth, order),
                            {"": lambda: det.process_depth_f32_cameras_host(as_float, order),
                             "unit 1": lambda: det.process_depth_f32_cameras_host(metres, order)}),
                   "device": (lambda: det.process_depth_cameras_device(d_z16, order, n),
                              {"": lambda: det.process_depth_f32_cameras_device(d_f, order, n),
                               "unit 1": lambda: det.process_depth_f32_cameras_device(d_m, order, n)})}
        groups_ = {"host": (lambda: det.process_depth_groups_host(depth, order, groups),
                            {"": lambda: det.process_depth_f32_groups_host(as_float, order, groups),
                             "unit 1": lambda: det.process_depth_f32_groups_host(metres, order, groups)}),
                   "device": (lambda: det.process_depth_groups_device(d_z16, order, groups),
                              {"": lambda: det.process_depth_f32_groups_device(d_f, order, groups),
                               "unit 1": lambda: det.process_depth_f32_groups_device(d_m, order, groups)})}
        for lens in (None, dists[1]):
            det.set_distortion(lens)
            for kind, (z16_call, float_calls) in plain.items():
                z16_call()
                want = everything(S, det, n)
                assert sum(len(fr[0][0]["steps"]) for fr in want[0]) >= n
                for unit, run in float_calls.items():
                    run()
                    assert everything(S, det, n) == want, ("plain", lens is not None, kind, unit)
        det.set_distortion(None)
        for table, calls in (("cameras", cameras), ("groups", groups_)):
            for kind, (z16_call, float_calls) in calls.items():
                det.set_cameras(cams, dists)
                z16_call()
                want = everything(S, det, n)
                for unit, run in float_calls.items():
                    det.set_cameras(cams1 if unit else cams, dists)
                    run()
                    assert everything(S, det, n) == want, (table, kind, unit)
        for p in (d_z16, d_f, d_m):
            det.free(p)


@gpu
def test_float_of_z16_equals_z16_4096x3072(S):
    w, h, n = 4096, 3072, 2
    base = lens_scene(S, w, h, None, noise_sigma=0.0025)
    depth = np.stack([S.synth_depth_host(S.randomize_scene(base, 77, i, 3, 8)) for i in range(n)])
    cfg = S.default_config(w, h, y_max=3.7, z_max=2.3)
    xf, a_inv = S.scene_transform_ex(base)
    intr = S.scene_intrinsics(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        all_options(det, a_inv, intr)
        det.process_depth_host(depth, intr)
        want = everything(S, det, n)
        assert all(fr[0][0]["steps"] for fr in want[0])
        det.process_depth_f32_host(depth.astype(f32), intr)
        assert everything(S, det, n) == want
        d_f = H.to_device(det, depth.astype(f32))
        det.process_depth_f32_device(d_f, intr, n)
        assert everything(S, det, n) == want
        det.free(d_f)


# ---- GPU: (b) equality with vertex input of the host deprojection ----
SPECIALS = [np.nan, np.inf, -np.inf, 0.0, -0.0, -1.5, np.float32(1e-45), np.finfo(f32).max]


def jittered_frames(S, base, n, seed):
    """z16 frames with an f32 sub-count jitter on every valid pixel, as samples in depth counts"""
    depth = np.stack([S.synth_depth_host(S.randomize_scene(base, seed, i, 3, 8)) for i in range(n)])
    rng = np.random.default_rng(seed)
    jitter = rng.uniform(-0.45, 0.45, depth.shape).astype(f32)
    return np.where(depth > 0, depth.astype(f32) + jitter, f32(0))


def sprinkle(frames, seed, per_value=300):
    """every special value at per_value random pixels of every frame; returns the frames and the pixels of each value"""
    out = frames.copy()
    n = out.shape[0]
    flat = out.reshape(n, -1)
    rng = np.random.default_rng(seed)
    where = {}
    for f in range(n):
        pix = rng.choice(flat.shape[1], size=per_value * len(SPECIALS), replace=False).reshape(len(SPECIALS), per_value)
        for k, v in enumerate(SPECIALS):
            flat[f, pix[k]] = f32(v)
            where.setdefault(k, []).append(pix[k])
    return out, where


@gpu
@pytest.mark.parametrize("lens", [None, BC], ids=["pinhole", "BC"])
@pytest.mark.parametrize("size", [(640, 480), (1024, 768)])
def test_float_frames_equal_vertex_input(S, size, lens):
    """non-quantised float frames with NaN, +-inf, +-0, negatives, the smallest subnormal and FLT_MAX == vertex input of their
    numpy deprojection, in depth units of the scene, in metres (unit 1) and with a unit of 2 (FLT_MAX * 2 overflows); plain and
    camera calls, host and device input. The label rules of the header hold at every special pixel."""
    w, h = size
    n = 3
    base = lens_scene(S, w, h, lens, **NOISY)
    counts = jittered_frames(S, base, n, 11 + w)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(base)
    unit0 = f32(base.depth_unit)
    with S.Detector(cfg, xf, max_frames=n) as det:
        all_options(det, a_inv, S.scene_intrinsics(base))
        det.set_distortion(S.scene_distortion(base))
        for unit, frames in ((unit0, counts), (f32(1.0), counts * unit0), (f32(2.0), counts * unit0 / f32(2.0))):
            frames, where = sprinkle(frames.astype(f32), int(unit * 1000) + w)
            sc = type(base).from_buffer_copy(base)
            sc.depth_unit = float(unit)
            assert f32(sc.depth_unit) == unit
            with np.errstate(all="ignore"):
                xyz = np.stack([np_deproject(sc, frames[f], lens) for f in range(n)])
            det.process_host(xyz)
            want = everything(S, det, n)
            if unit == unit0:
                assert sum(len(fr[0][0]["steps"]) for fr in want[0]) >= n
            intr = intr_with_unit(S, base, float(unit))
            det.set_cameras([camera_with_unit(S, base, float(unit))], [S.scene_distortion(base)])
            d_f = H.to_device(det, frames)
            for kind, run in {"host": lambda: det.process_depth_f32_host(frames, intr),
                              "device": lambda: det.process_depth_f32_device(d_f, intr, n),
                              "camera host": lambda: det.process_depth_f32_cameras_host(frames, np.zeros(n, np.int32)),
                              "camera device": lambda: det.process_depth_f32_cameras_device(d_f, np.zeros(n, np.int32), n)}.items():
                run()
                assert everything(S, det, n) == want, (float(unit), kind)
            det.free(d_f)
            for f in range(n):
                labels = det.labels(f)
                info = det.frame_info(f)
                assert info.n_nonzero == int((labels != A.LABEL_INVALID).sum()), (float(unit), f)
                for k, v in enumerate(SPECIALS):
                    lab = labels[where[k][f]]
                    with np.errstate(all="ignore"):
                        z = f32(v) * unit
                    if not z > 0:
                        # NaN, -inf, +-0, negatives, and the subnormal when its product rounds to 0: the invalid pixel
                        assert (lab == A.LABEL_INVALID).all(), (float(unit), v)
                    elif not np.isfinite(z) or v == np.finfo(f32).max:
                        # +inf, FLT_MAX * 2 (overflow): a non-finite world point; FLT_MAX * unit <= 1: far outside the range
                        assert (lab == A.LABEL_OUT_OF_RANGE).all(), (float(unit), v)
                    else:
                        assert v < 1e-37 and (lab != A.LABEL_INVALID).all(), (float(unit), v)  # the subnormal is kept: z > 0


# ---- GPU: errors ----
@gpu
def test_rejected_calls_leave_the_results_readable(S):
    w, h, n = 640, 480, 2
    base = lens_scene(S, w, h, None, **NOISY)
    depth = np.stack([S.synth_depth_host(S.randomize_scene(base, 5, i, 3, 8)) for i in range(n)]).astype(f32)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(base)
    intr = S.scene_intrinsics(base)
    N = w * h
    with S.Detector(cfg, xf, max_frames=n) as det:
        all_options(det, a_inv, intr)
        L, h_ = det._l, det._h
        cams = np.zeros(n, np.int32)
        grp = np.array([n], np.int32)

        def calls(p_host, p_dev):
            return [lambda: L.ssd_gpu_process_depth_f32_host(h_, p_host, C.byref(intr), n),
                    lambda: L.ssd_gpu_process_depth_f32_device(h_, p_dev, C.byref(intr), n),
                    lambda: L.ssd_gpu_process_depth_f32_cameras_host(h_, p_host, H.ptr(cams), n),
                    lambda: L.ssd_gpu_process_depth_f32_cameras_device(h_, p_dev, H.ptr(cams), n),
                    lambda: L.ssd_gpu_process_depth_f32_groups_host(h_, p_host, H.ptr(cams), H.ptr(grp), 1),
                    lambda: L.ssd_gpu_process_depth_f32_groups_device(h_, p_dev, H.ptr(cams), H.ptr(grp), 1, 0)]

        # no camera table: SSD_E_STATE from the camera and group calls, before any result is touched
        det.process_depth_f32_host(depth, intr)
        want = everything(S, det, n)

        def unchanged():
            assert everything(S, det, n) == want

        d_f = det.malloc(depth.nbytes + 64)
        det.h2d(d_f, depth)
        for call in calls(H.ptr(depth), d_f)[2:]:
            assert call() == A.E_STATE
            unchanged()
        det.set_cameras([S.scene_camera(base), camera_with_unit(S, base, 0.0)])
        det.process_depth_f32_cameras_host(depth, cams)
        want = everything(S, det, n)
        # misaligned input, 4 and 8 bytes off (host and device)
        buf = np.zeros(depth.size + 16, f32)
        off0 = (-buf.ctypes.data % 16) // 4
        for off in (1, 2):
            mis = buf[off0 + off:off0 + off + depth.size]
            mis[:] = depth.ravel()
            assert mis.ctypes.data % 16 == 4 * off
            d_mis = C.c_void_p(d_f.value + 4 * off)
            for call in calls(mis.ctypes.data_as(C.c_void_p), d_mis):
                assert call() == A.E_INVALID_ARG
                assert "aligned" in det._l.ssd_gpu_last_error(det._h).decode()
                unchanged()
        # NULL arguments
        for call in calls(None, None):
            assert call() == A.E_INVALID_ARG
            unchanged()
        assert L.ssd_gpu_process_depth_f32_host(h_, H.ptr(depth), None, n) == A.E_INVALID_ARG
        assert L.ssd_gpu_process_depth_f32_cameras_host(h_, H.ptr(depth), None, n) == A.E_INVALID_ARG
        assert L.ssd_gpu_process_depth_f32_groups_host(h_, H.ptr(depth), H.ptr(cams), None, 1) == A.E_INVALID_ARG
        unchanged()
        # a camera index outside the table, more frames than max_frames: SSD_E_RANGE
        bad = np.array([0, 2], np.int32)
        assert L.ssd_gpu_process_depth_f32_cameras_host(h_, H.ptr(depth), H.ptr(bad), n) == A.E_RANGE
        assert L.ssd_gpu_process_depth_f32_groups_device(h_, d_f, H.ptr(bad), H.ptr(grp), 1, 0) == A.E_RANGE
        big = np.zeros(n + 1, np.int32)
        assert L.ssd_gpu_process_depth_f32_cameras_device(h_, d_f, H.ptr(big), n + 1) == A.E_RANGE
        assert L.ssd_gpu_process_depth_f32_host(h_, H.ptr(np.zeros((n + 1) * N, f32)), C.byref(intr), n + 1) == A.E_RANGE
        unchanged()
        # a camera without valid intrinsics (camera 1: depth_unit = 0)
        one = np.array([0, 1], np.int32)
        assert L.ssd_gpu_process_depth_f32_cameras_host(h_, H.ptr(depth), H.ptr(one), n) == A.E_INVALID_ARG
        assert L.ssd_gpu_process_depth_f32_groups_host(h_, H.ptr(depth), H.ptr(one), H.ptr(grp), 1) == A.E_INVALID_ARG
        # and a plain call with invalid intrinsics
        zero_unit = intr_with_unit(S, base, 0.0)
        assert L.ssd_gpu_process_depth_f32_device(h_, d_f, C.byref(zero_unit), n) == A.E_INVALID_ARG
        unchanged()
        det.free(d_f)


# ---- GPU: z16 and float calls alternate on one context ----
@gpu
def test_z16_and_float_calls_alternate(S, monkeypatch):
    """host calls of both sample types alternate on one context, with group calls that grow the staging buffers in between:
    every result equals a fresh context's"""
    monkeypatch.setenv("SSD_GPU_HOST_CHUNK_FRAMES", "2")
    w, h, n = 848, 480, 6
    bases = camera_bases(S, w, h)
    order, depth = camera_frames(S, bases, n, 3)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(bases[0])
    intr = S.scene_intrinsics(bases[0])
    cams, dists = [S.scene_camera(b) for b in bases], [S.scene_distortion(b) for b in bases]
    other = camera_frames(S, bases, n, 4)[1]  # different frames: a stale staging buffer would show
    calls = [("z16", lambda d, x: d.process_depth_host(x, intr)),
             ("f32", lambda d, x: d.process_depth_f32_host(x.astype(f32), intr)),
             ("z16 cameras", lambda d, x: d.process_depth_cameras_host(x, order)),
             ("f32 groups", lambda d, x: d.process_depth_f32_groups_host(x.astype(f32), order, [4, 2])),
             ("f32 cameras", lambda d, x: d.process_depth_f32_cameras_host(x.astype(f32), order)),
             ("z16 groups", lambda d, x: d.process_depth_groups_host(x, order, [1, 5])),
             ("f32", lambda d, x: d.process_depth_f32_host(x.astype(f32), intr)),
             ("z16", lambda d, x: d.process_depth_host(x, intr))]

    def fresh(call, x):
        with S.Detector(cfg, xf, max_frames=n) as d:
            all_options(d, a_inv, intr)
            d.set_cameras(cams, dists)
            call(d, x)
            return everything(S, d, n)

    with S.Detector(cfg, xf, max_frames=n) as det:
        all_options(det, a_inv, intr)
        det.set_cameras(cams, dists)
        for i, (kind, call) in enumerate(calls):
            x = depth if i % 2 == 0 else other
            call(det, x)
            assert everything(S, det, n) == fresh(call, x), (i, kind)


# ---- GPU: the C++ host classes ----
@gpu
def test_cpp_pointcloud_over_float_frames(S, tmp_path):
    """tests/native/depth_f32_check.cpp: Pointcloud over DepthFrame(const float *, ...) prints the line of the z16 DepthFrame, for
    plain (pin-hole, BC lens), camera and group processing"""
    exe = str(tmp_path / "depth_f32_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "depth_f32_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([exe, "640", "480"], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == 16
    for i in range(0, 16, 2):
        assert out[i] == out[i + 1], i // 2
    assert sum(l.count("height") >= 2 for l in out) >= 12
