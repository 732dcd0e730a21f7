"""Per-frame cameras (ssd_gpu_set_cameras / ssd_gpu_process_*cameras*): frames of several camera mountings in one batched
call. Frame i of a camera call must be processed exactly as a context created with camera camera_of_frame[i]'s transform
processes it: against the stored reference runs, the oracle with each frame's transform, and per-camera contexts."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

TOL = 1e-4  # metres: 0.1 mm, as tests/test_gpu_parity.py
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
gpu = pytest.mark.gpu


# ---- layout and binding (no GPU) ----
def test_camera_struct_layout():
    assert C.sizeof(A.Camera) == 19 * 8 + 9 * 8 + C.sizeof(A.Intrinsics) == 256
    assert A.Camera.a_inv.offset == 152 and A.Camera.intr.offset == 224


def test_camera_entry_points_are_declared_bound_and_versioned(S):
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    assert re.search(r"#define SSD_GPU_ABI_VERSION 3\b", hdr)
    assert S.lib().ssd_gpu_abi_version() == 3
    for name in ("ssd_gpu_set_cameras", "ssd_gpu_n_cameras", "ssd_gpu_process_cameras_host", "ssd_gpu_process_cameras_device",
                 "ssd_gpu_process_cameras_device_ex", "ssd_gpu_process_depth_cameras_host", "ssd_gpu_process_depth_cameras_device"):
        assert re.search(r"\b%s\(" % name, hdr) and name in A.PROTOTYPES, name
        assert getattr(S.lib(), name).argtypes == A.PROTOTYPES[name][1]


def test_scene_camera_record(S):
    sc = S.default_scene(320, 240, rotate180=1, fx=300.0)
    cam = S.scene_camera(sc)
    xf, a_inv = S.scene_transform_ex(sc)
    assert bytes(cam.xf) == bytes(xf) and np.array_equal(np.array(cam.a_inv[:]), a_inv)
    assert bytes(cam.intr) == bytes(S.scene_intrinsics(sc)) and cam.intr.fx == 300.0


# ---- helpers ----
def camera_scenes(S, w, h):
    """the three synthetic camera mountings (also those of examples/detect_stairs_multicamera.cpp): default; higher, pitched,
    rolled and yawed with other intrinsics and an occluder; upside down with occluders and other intrinsics"""
    d = S.default_scene(w, h)
    return [S.default_scene(w, h, **NOISY),
            S.default_scene(w, h, cam_height=d.cam_height * 1.1, cam_pitch_deg=d.cam_pitch_deg + 4.0, cam_roll_deg=2.0, cam_yaw_deg=-3.0,
                            fx=d.fx * 1.08, fy=d.fy * 1.06, ppx=d.ppx + 7.0, ppy=d.ppy - 5.0, n_occluders=1, **NOISY),
            S.default_scene(w, h, rotate180=1, n_occluders=2, cam_roll_deg=-1.5, fx=d.fx * 0.95, fy=d.fy * 0.97, ppx=d.ppx - 4.0, **NOISY)]


def mixed_batch(S, w=1024, h=768, per_cam=3, seed=7):
    """frames of three cameras with different poses and intrinsics (camera 2: mounted upside down, occluders), interleaved in a
    shuffled order. Returns cfg, cameras, camera_of_frame, depth, xyz, per-frame transforms."""
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    order = np.random.default_rng(seed).permutation(np.repeat(np.arange(len(bases)), per_cam)).astype(np.int32)
    depth, xyz, xfs = [], [], []
    for i, c in enumerate(order):
        sc = S.randomize_scene(bases[c], 500 + seed, i, 3, 8)
        sc.rotate180, sc.n_occluders = bases[c].rotate180, bases[c].n_occluders
        xf = S.scene_transform(sc)
        assert bytes(xf) == bytes(cams[c].xf)  # the frame's calibration is its camera's
        dd = S.synth_depth_host(sc)
        depth.append(dd)
        xyz.append(S.deproject_host(sc, dd))
        xfs.append(cams[c].xf)
    return cfg, cams, order, np.stack(depth), np.stack(xyz), xfs


# ---- 1. the stored reference runs, one call per size ----
@gpu
@pytest.mark.parametrize("key", ["frames_random_scenes/320x240", "frames_random_scenes/640x480", "frames_random_scenes/1024x768",
                                 "frames_hires/2560x1920", "frames_hires/4096x3072"])
def test_camera_call_against_the_reference_runs(S, key):
    """every frame with its own pose (or, hires, identical cameras) in ONE camera call, against the reference's stored results"""
    import test_oracle_vs_ref as R
    kind, size = key.split("/")
    w, h = (int(v) for v in size.split("x"))
    if kind == "frames_hires":
        _, _, ck, sk, n = next(c for c in R.HIRES_CASES if c[:2] == (w, h))
        inputs = list(R.frames_hires_inputs(S, w, h, ck, sk, n))
    else:
        inputs = list(R.frames_random_scenes_inputs(S, w, h, {320: 10, 640: 6, 1024: 3}[w]))
    want = R.stored(key)
    cfg = inputs[0][0]
    xyz = np.stack([x for _, _, x in inputs])
    # the context's own transform is deliberately none of the frames'
    with S.Detector(cfg, S.scene_transform(S.default_scene(w, h)), max_frames=len(inputs)) as det:
        det.set_cameras([S.make_camera(xf) for _, xf, _ in inputs])
        det.process_cameras_host(xyz, np.arange(len(inputs)))
        for i in range(len(inputs)):
            g = H.gpu_result(det, i)
            assert not H.compare_with_record(want[i], g, tol=TOL), (i, H.compare_with_record(want[i], g, tol=TOL))
            assert (g.info["status"] & ~R.QUIRKS) == want[i]["info"]["status"], i


# ---- 2. oracle parity, mixed cameras, every input kind ----
@gpu
def test_mixed_cameras_equal_the_oracle(S, oracle):
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S)
    n = len(order)
    want = [H.oracle_process(oracle, cfg, xfs[f], xyz[f]) for f in range(n)]
    runs = {}
    with S.Detector(cfg, cams[1].xf, max_frames=n) as det:
        det.set_cameras(cams)
        assert det.n_cameras == 3
        d_xyz, d_z16 = H.to_device(det, xyz), H.to_device(det, depth)
        for kind in ("vertices/host", "vertices/device", "z16/host", "z16/device"):
            if kind == "vertices/host":
                det.process_cameras_host(xyz, order)
            elif kind == "vertices/device":
                det.process_cameras_device(d_xyz, order, n)
            elif kind == "z16/host":
                det.process_depth_cameras_host(depth, order)
            else:
                det.process_depth_cameras_device(d_z16, order, n)
            runs[kind] = []
            for f in range(n):
                g = H.gpu_result(det, f)
                bad = H.compare_results(want[f], g, tol=TOL)
                assert not bad, (kind, f, order[f], bad)
                assert g.info["status"] == want[f].info["status"], (kind, f)
                runs[kind].append(H.exact(g))
        det.free(d_xyz)
        det.free(d_z16)
    assert sum(len(w.steps) for w in want) >= 2 * n
    for kind in runs:  # the z16 input deprojects to the very vertices: identical results
        assert runs[kind] == runs["vertices/host"], kind


@gpu
def test_mixed_cameras_unfused_chain_equal_the_oracle(S, oracle):
    """more than SSD_FUSE_MAX_FRAMES (16) frames per chunk: the unfused camera kernels (k_transform_bin[_depth], k_peaks,
    k_frame_logic as launches of their own), every input kind, against the oracle"""
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S, 320, 240, per_cam=7, seed=13)
    n = len(order)
    assert n > 16
    want = [H.oracle_process(oracle, cfg, xfs[f], xyz[f]) for f in range(n)]
    with S.Detector(cfg, cams[0].xf, max_frames=n) as det:
        assert det.chunk_frames >= n
        det.set_cameras(cams)
        d_xyz, d_z16 = H.to_device(det, xyz), H.to_device(det, depth)
        for run in range(5):
            [lambda: det.process_cameras_host(xyz, order), lambda: det.process_cameras_device(d_xyz, order, n),
             lambda: det.process_cameras_device(d_xyz, order, n, A.FLAG_STAGE_TIMING | A.FLAG_SINGLE_STREAM),
             lambda: det.process_depth_cameras_host(depth, order), lambda: det.process_depth_cameras_device(d_z16, order, n)][run]()
            assert det.timing().n_launches == 7, run  # one chunk, the seven-launch chain
            for f in range(n):
                g = H.gpu_result(det, f)
                assert not H.compare_results(want[f], g, tol=TOL), (run, f)
                assert g.info["status"] == want[f].info["status"], (run, f)
        det.free(d_xyz)
        det.free(d_z16)


# ---- 3. equal to one plain context per camera ----
@gpu
def test_mixed_cameras_equal_per_camera_contexts(S):
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S, seed=11)
    n = len(order)
    with S.Detector(cfg, cams[0].xf, max_frames=n) as det:
        det.set_cameras(cams)
        det.process_cameras_host(xyz, order)
        got = [H.exact(H.gpu_result(det, f)) for f in range(n)]
        st = det.stats()
    fields = ("n_points", "n_exact_fallback", "n_quad_fast", "n_quad_exact", "n_bev_exact")
    total = dict.fromkeys(fields, 0)
    eps0 = eps1 = 0.0
    for c, cam in enumerate(cams):
        idx = np.flatnonzero(order == c)
        with S.Detector(cfg, cam.xf, max_frames=len(idx)) as one:
            one.process_host(xyz[idx])
            for j, f in enumerate(idx):
                assert H.exact(H.gpu_result(one, j)) == got[f], (c, f)
            s1 = one.stats()
            for k in fields:
                total[k] += getattr(s1, k)
            eps0, eps1 = max(eps0, s1.filter_eps0), max(eps1, s1.filter_eps1)
    assert {k: getattr(st, k) for k in fields} == total
    assert (st.filter_eps0, st.filter_eps1) == (eps0, eps1)


# ---- 4. degenerate table: camera 0 is the context's own camera ----
@gpu
def test_one_camera_table_equals_the_plain_call(S):
    w, h = 640, 480
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    scenes = [S.randomize_scene(base, 77, i, 3, 8) for i in range(5)]
    xf, a_inv = S.scene_transform_ex(base)
    intr = S.scene_intrinsics(base)
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    n = len(scenes)

    def everything(det):
        return [(H.exact(H.gpu_result(det, f)), det.overlay(f).tobytes(), det.vertical_faces(f)) for f in range(n)]

    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_overlay(a_inv, intr)
        det.set_vertical_faces(True)
        det.set_cameras([S.scene_camera(base)])
        det.process_host(xyz)
        plain = everything(det)
        plain_stats = bytes(det.stats())
        det.process_cameras_host(xyz, np.zeros(n))
        assert everything(det) == plain
        assert bytes(det.stats()) == plain_stats
        det.process_depth_cameras_host(depth, np.zeros(n))
        assert everything(det) == plain
        det.process_depth_host(depth, intr)
        assert everything(det) == plain


# ---- 5. chunks and streams: the chunk offset into camera_of_frame ----
@gpu
def test_camera_calls_over_many_chunks(S, oracle, monkeypatch):
    monkeypatch.setenv("SSD_GPU_CHUNK_FRAMES", "8")
    monkeypatch.setenv("SSD_GPU_HOST_CHUNK_FRAMES", "4")
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S, 320, 240, per_cam=7, seed=3)
    n = len(order)
    want = [H.oracle_process(oracle, cfg, xfs[f], xyz[f]) for f in range(n)]
    with S.Detector(cfg, cams[2].xf, max_frames=n) as det:
        assert det.chunk_frames == 8 and n > 8
        d_xyz, d_z16 = H.to_device(det, xyz), H.to_device(det, depth)
        det.set_cameras(cams)
        for run in range(4):
            [lambda: det.process_cameras_host(xyz, order), lambda: det.process_cameras_device(d_xyz, order, n),
             lambda: det.process_depth_cameras_host(depth, order), lambda: det.process_depth_cameras_device(d_z16, order, n)][run]()
            for f in range(n):
                g = H.gpu_result(det, f)
                assert not H.compare_results(want[f], g, tol=TOL), (run, f)
                assert g.info["status"] == want[f].info["status"], (run, f)
        det.free(d_xyz)
        det.free(d_z16)


# ---- 6. overlay and risers with each frame's camera ----
@gpu
def test_overlay_and_risers_per_camera(S, oracle):
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S, seed=5)
    n = len(order)
    with S.Detector(cfg, cams[0].xf, max_frames=n) as det:
        det.set_cameras(cams)
        # the plain call's overlay arguments: deliberately another camera's, they must not leak into the camera call
        det.set_overlay(np.array(cams[1].a_inv[:]), cams[1].intr)
        det.set_vertical_faces(True)
        for kind in ("vertices", "z16"):
            if kind == "vertices":
                det.process_cameras_host(xyz, order)
            else:
                det.process_depth_cameras_host(depth, order)
            n_px = 0
            for f in range(n):
                cam = cams[order[f]]
                H.oracle_process(oracle, cfg, cam.xf, xyz[f])
                want = H.oracle_overlay(oracle, cam.xf, np.array(cam.a_inv[:]), cam.intr)
                got = det.overlay(f)
                assert got.shape == want.shape, (kind, f)
                if len(want):
                    assert np.abs(got - want).max() < 2e-3, (kind, f)
                    n_px += want.size
                assert det.vertical_faces(f) == H.oracle_vertical_faces(oracle, cfg, cam.xf, xyz[f].reshape(-1, 3)), (kind, f)
            assert n_px >= 8 * n


# ---- 7. one camera per frame at scale, device-generated ----
@gpu
def test_per_frame_poses_at_scale(S, oracle):
    w, h, n = 640, 480, 320
    N = w * h
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, randomize_camera=1, **NOISY)
    scenes = [S.randomize_scene(base, 2024, i, 3, 8) for i in range(n)]
    with S.Detector(cfg, S.scene_transform(base), max_frames=n) as det:
        d_xyz = det.malloc(n * N * 12)
        det.synth_frames(base, 2024, 0, n, 3, 8, d_xyz)
        det.set_cameras([S.scene_camera(sc) for sc in scenes])
        det.process_cameras_device(d_xyz, np.arange(n), n)
        for f in sorted(np.random.default_rng(9).choice(n, 10, replace=False)):
            xyz = np.empty((N, 3), np.float32)
            det.d2h(xyz, C.c_void_p(d_xyz.value + int(f) * N * 12))
            xf = S.scene_transform(scenes[f])
            o = H.oracle_process(oracle, cfg, xf, xyz)
            g = H.gpu_result(det, int(f))
            assert not H.compare_results(o, g, tol=TOL), f
            assert g.info["status"] == o.info["status"], f
        det.free(d_xyz)


# ---- 8. errors leave the previous results intact; no leakage into plain calls ----
@gpu
def test_camera_call_rejections(S):
    cfg, cams, order, depth, xyz, xfs = mixed_batch(S, 320, 240, per_cam=2, seed=1)
    n = len(order)
    own = S.scene_transform(S.default_scene(320, 240))
    with S.Detector(cfg, own, max_frames=n) as det:
        with pytest.raises(S.SsdError, match=r"\(-5\).*no camera table"):
            det.process_cameras_host(xyz, order)
        det.process_host(xyz)
        plain = [H.exact(H.gpu_result(det, f)) for f in range(n)]
        with pytest.raises(S.SsdError, match=r"\(-5\)"):
            det.process_cameras_host(xyz, order)
        det.set_cameras(cams)
        for bad in (3, -1, 1 << 30):
            o = order.copy()
            o[n // 2] = bad
            with pytest.raises(S.SsdError, match=r"\(-4\)"):
                det.process_cameras_host(xyz, o)
            with pytest.raises(S.SsdError, match=r"\(-4\)"):
                det.process_depth_cameras_host(depth, o)
        no_intr = list(cams) + [S.make_camera(cams[0].xf)]
        det.set_cameras(no_intr)
        o = order.copy()
        o[-1] = 3
        with pytest.raises(S.SsdError, match=r"\(-1\).*intrinsics"):
            det.process_depth_cameras_host(depth, o)
        # rejected calls left the plain call's results readable
        assert [H.exact(H.gpu_result(det, f)) for f in range(n)] == plain
        # camera 3 has the transform of camera 0 but no intrinsics: fine for vertex input
        det.process_cameras_host(xyz, o)
        mixed = [H.exact(H.gpu_result(det, f)) for f in range(n)]
        # a plain call after a camera call uses the context's own transform
        det.process_host(xyz)
        assert [H.exact(H.gpu_result(det, f)) for f in range(n)] == plain
        # replacing the table takes effect: the reversed table with reversed indices is the same batch
        det.set_cameras(no_intr[::-1])
        det.process_cameras_host(xyz, 3 - o)
        assert [H.exact(H.gpu_result(det, f)) for f in range(n)] == mixed
        with pytest.raises(S.SsdError, match=r"\(-1\)"):
            det.process_depth_cameras_host(depth, 3 - o)  # now camera 0 lacks the intrinsics
        det.set_cameras([])
        assert det.n_cameras == 0
        with pytest.raises(S.SsdError, match=r"\(-5\)"):
            det.process_cameras_host(xyz, o)


# ---- 9. the C++ host classes: several cameras through one Pointcloud ----
@gpu
def test_cpp_host_classes_multicamera(S, oracle, tmp_path):
    """examples/detect_stairs_multicamera.cpp (Pointcloud::addCamera + processBatch with the camera of each frame): its lines
    equal the oracle's for the same frames, each with its own camera's transformation"""
    import json
    exe = str(tmp_path / "detect_stairs_multicamera")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "examples", "detect_stairs_multicamera.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h, n = 640, 480, 6
    out = subprocess.run([exe, str(w), str(h), str(n)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == n
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    n_steps = 0
    for f in range(n):
        b = bases[f % 3]
        sc = S.randomize_scene(b, 2027, f, 3, 8)
        sc.rotate180, sc.n_occluders = b.rotate180, b.n_occluders
        xf = S.scene_transform(sc)
        assert bytes(xf) == bytes(S.scene_transform(b))
        o = H.oracle_process(oracle, cfg, xf, S.deproject_host(sc, S.synth_depth_host(sc)))
        got = json.loads(out[f])
        assert got[0] == "stairs" and got[1] == ["stairSteps", len(o.steps)], f
        for s, g in zip(o.steps, got[2] if len(o.steps) else []):
            assert abs(g[0][1] - s["height"]) < 1.1e-3, f  # the line prints three decimals
            assert np.abs(np.array(g[1][1:]) - s["quad"]).max() < 1.1e-3, f
        n_steps += len(o.steps)
    assert n_steps >= 2 * n
