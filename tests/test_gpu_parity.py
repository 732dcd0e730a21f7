"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle (oracle/ssd_oracle.c)
on the same seeded inputs. Bars (BASELINE.json north_star): labels / histogram / peaks bit-exact, step
heights and corners within 0.1 mm (TOL below; in practice they agree to ~1e-12 m)."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

pytestmark = pytest.mark.gpu
TOL = 1e-4  # metres: 0.1 mm

NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)


def gpu_result(S, det, frame):
    info = det.frame_info(frame)
    plats, _ = det.plateaus(frame)
    steps = (A.Step * A.MAX_STEPS)()
    n = C.c_int()
    det._ck(det._l.ssd_gpu_get_steps(det._h, frame, steps, A.MAX_STEPS, C.byref(n), None), "get_steps")
    hist = np.zeros(A.MAX_BINS, np.uint32)
    hist[:info.n_bins] = det.histogram(frame)
    return H._collect(det.labels(frame), hist, info, plats, steps, det.line(frame))


_REFS = {}


def _ref_for(cfg):
    """the compiled reference for this configuration if its library was built (never builds here: the GPU box has no sources)"""
    import os
    key = H.ref_tag(cfg)
    if key not in _REFS:
        _REFS[key] = H.load_ref(cfg) if (os.path.exists(H.ref_path(cfg)) or H.ref_available()) else None
    return _REFS[key]


def _line_delta(a, b):
    """largest difference between the numbers of two result lines (a height within 1e-6 m of a rounding boundary may print
    a different third decimal)"""
    import re
    na, nb = [float(x) for x in re.findall(r"-?\d+\.\d+", a)], [float(x) for x in re.findall(r"-?\d+\.\d+", b)]
    if len(na) != len(nb):
        return float("inf")
    return max([abs(x - y) for x, y in zip(na, nb)], default=0.0)


def run_frames(S, oracle, cfg, scenes, max_bad=0):
    xf = S.scene_transform(scenes[0])
    xyz = np.stack([S.deproject_host(sc, S.synth_depth_host(sc)) for sc in scenes])
    with S.Detector(cfg, xf, max_frames=len(scenes)) as det:
        det.process_host(xyz)
        out = []
        for f in range(len(scenes)):
            g = gpu_result(S, det, f)
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            bad = H.compare_results(o, g, tol=TOL)
            assert g.info["status"] == o.info["status"], (f, hex(g.info["status"]), hex(o.info["status"]))
            assert not bad, (f, bad)
            # one hop less: straight against the compiled reference (oracle/_ref ships to the GPU box) where it exists for
            # this configuration; its harness does not raise the quirk bits, so the status is compared through the oracle
            ref = _ref_for(cfg)
            if ref is not None and f < 4:
                r = H.ref_process(ref, cfg, xf, xyz[f])
                bad = H.compare_results(r, g, tol=TOL)
                assert not bad, ("vs compiled reference", f, bad)
                assert g.line == r.line or abs(_line_delta(g.line, r.line)) <= 1.001e-3, (g.line, r.line)
            out.append((g, o))
        return out


@pytest.mark.parametrize("key", ["frames_random_scenes/320x240", "frames_random_scenes/640x480", "frames_random_scenes/1024x768",
                                 "frames_hires/2560x1920", "frames_hires/4096x3072"])
def test_against_the_reference_runs(S, key):
    """straight against the compiled reference without the oracle in between: the CUDA path on the seeded frames of
    test_oracle_vs_ref against the reference's results for them (tests/golden/reference_runs.json)"""
    import test_oracle_vs_ref as R
    kind, size = key.split("/")
    w, h = (int(v) for v in size.split("x"))
    if kind == "frames_hires":
        _, _, ck, sk, n = next(c for c in R.HIRES_CASES if c[:2] == (w, h))
        inputs = R.frames_hires_inputs(S, w, h, ck, sk, n)
    else:
        inputs = R.frames_random_scenes_inputs(S, w, h, {320: 10, 640: 6, 1024: 3}[w])
    want = R.stored(key)
    for i, (cfg, xf, xyz) in enumerate(inputs):
        with S.Detector(cfg, xf, max_frames=1) as det:
            det.process_host(xyz[None])
            g = gpu_result(S, det, 0)
        assert not H.compare_with_record(want[i], g, tol=TOL), (i, H.compare_with_record(want[i], g, tol=TOL))
        assert (g.info["status"] & ~R.QUIRKS) == want[i]["info"]["status"], i


@pytest.mark.parametrize("w,h", [(1024, 768), (640, 480), (320, 240)])
def test_clean_frame(S, oracle, w, h):
    cfg = S.default_config(w, h)
    (g, o), = run_frames(S, oracle, cfg, [S.default_scene(w, h)])
    assert g.info["n_steps"] == 4  # ground + 3 steps
    heights = [s["height"] for s in g.steps]
    assert np.allclose(heights, [0.004, 0.177, 0.350, 0.523], atol=2e-3)


def test_noisy_frame(S, oracle):
    cfg = S.default_config(1024, 768)
    (g, o), = run_frames(S, oracle, cfg, [S.default_scene(1024, 768, **NOISY)])
    assert g.info["n_steps"] >= 3


def test_descending_occluded(S, oracle):
    cfg = S.default_config(1024, 768)
    base = S.default_scene(1024, 768, rotate180=1, n_occluders=2, **NOISY)
    run_frames(S, oracle, cfg, [base])


def test_batch_random_scenes(S, oracle):
    """config 3 distribution, one shared calibration (camera pose fixed, stairs vary)."""
    cfg = S.default_config(1024, 768)
    base = S.default_scene(1024, 768, **NOISY)
    scenes = []
    for i in range(24):
        scenes.append(S.randomize_scene(base, 4242, i, 3, 8))  # camera pose fixed: one calibration per context
    res = run_frames(S, oracle, cfg, scenes)
    assert sum(g.info["n_steps"] for g, _ in res) > 24 * 3


def test_empty_and_garbage_frames(S, oracle):
    cfg = S.default_config(640, 480)
    sc = S.default_scene(640, 480)
    xf = S.scene_transform(sc)
    rng = np.random.default_rng(1)
    frames = np.zeros((4, 480, 640, 3), np.float32)  # frame 0: all invalid
    frames[1] = rng.uniform(-2, 2, (480, 640, 3)).astype(np.float32)  # uniform noise
    frames[2, ..., 2] = 1.0  # a fronto-parallel wall
    # frame 3: a valid scene salted with NaN / Inf / huge / denormal coordinates (the f32 filter must hand them to the exact path)
    frames[3] = S.deproject_host(sc, S.synth_depth_host(sc)).reshape(480, 640, 3)
    bad = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38, 1e-42, 1e20], np.float32)
    idx = rng.integers(0, 480 * 640 * 3, 20000)
    frames[3].reshape(-1)[idx] = bad[rng.integers(0, len(bad), idx.size)]
    with S.Detector(cfg, xf, max_frames=4) as det:
        det.process_host(frames)
        for f in range(4):
            g = gpu_result(S, det, f)
            o = H.oracle_process(oracle, cfg, xf, frames[f])
            assert not H.compare_results(o, g, tol=TOL), f
            assert g.info["status"] == o.info["status"]


@pytest.mark.parametrize("w,h", [(640, 480), (1024, 768)])
def test_depth_frame_input(S, oracle, monkeypatch, w, h):
    """The z16 depth-frame entry points (what the reference's process() receives): on-device deprojection is bit-identical
    to the host's, and host / device depth input -- deprojected inside the three point kernels, no vertex array in
    memory -- give exactly the results of the vertex path, which is checked against the oracle. The unfused A/B path
    (separate deprojection kernel) must agree too."""
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    scenes = [S.randomize_scene(base, 77, i, 3, 6) for i in range(5)]
    xf = S.scene_transform(base)
    k = S.scene_intrinsics(base)
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    n = len(scenes)
    with S.Detector(cfg, xf, max_frames=n) as det:
        # deprojection alone
        d_depth = det.malloc(depth.nbytes)
        d_xyz = det.malloc(xyz.nbytes)
        det.h2d(d_depth, depth)
        det.deproject_device(d_depth, k, n, d_xyz)
        got = np.empty_like(xyz)
        det.d2h(got, d_xyz)
        assert np.array_equal(got.view(np.uint32), xyz.view(np.uint32)), "device deprojection differs from the host's"
        # vertex path = reference results
        det.process_host(xyz)
        def exact_steps(f):
            st, status = det.steps(f)
            return [(float(hh).hex(), np.asarray(q, np.float64).tobytes()) for hh, q in st], status

        ref = [(det.labels(f), det.histogram(f), det.line(f), exact_steps(f)) for f in range(n)]
        for f in range(n):
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            assert not H.compare_results(o, gpu_result(S, det, f), tol=TOL), f
        for run in ("host", "device", "device-unfused", "host-unfused"):
            monkeypatch.setenv("SSD_GPU_DEPTH_UNFUSED", "1" if run.endswith("unfused") else "0")
            if run.startswith("host"):
                det.process_depth_host(depth, k)
            else:
                det.process_depth_device(d_depth, k, n)
            for f in range(n):
                assert np.array_equal(det.labels(f), ref[f][0]), (run, f)
                assert np.array_equal(det.histogram(f), ref[f][1]), (run, f)
                assert det.line(f) == ref[f][2], (run, f)
                assert exact_steps(f) == ref[f][3], (run, f)  # same vertices, same arithmetic: bit-identical doubles
        det.free(d_depth)
        det.free(d_xyz)


def test_hires_extended_range(S, oracle):
    cfg = S.default_config(4096, 3072, y_max=3.7, z_max=2.3)
    sc = S.default_scene(4096, 3072, n_steps=12, riser=0.17, tread=0.26, cam_height=3.2, cam_pitch_deg=48.0,
                         first_riser_y=0.5, **NOISY)
    run_frames(S, oracle, cfg, [sc])


def test_depth_input_edge_cases(S):
    """Depth frames that are not scenes -- all zero (every pixel invalid), all 65535, white noise, a constant plane -- and a
    batch that is not a multiple of the host chunk (33 frames, chunk 32): the fused depth kernels must give exactly what
    the vertex path gives on the host-deprojected vertices, frame by frame."""
    w, h = 320, 240
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    xf = S.scene_transform(base)
    k = S.scene_intrinsics(base)
    rng = np.random.default_rng(5)
    frames = [np.zeros((h, w), np.uint16), np.full((h, w), 65535, np.uint16), rng.integers(0, 65536, (h, w), dtype=np.uint16),
              np.full((h, w), 4000, np.uint16)]
    frames += [S.synth_depth_host(S.randomize_scene(base, 9, i, 3, 6)).reshape(h, w) for i in range(29)]
    depth = np.stack(frames).reshape(len(frames), -1)
    xyz = np.stack([S.deproject_host(base, d) for d in depth])
    n = len(frames)
    assert n == 33
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.process_host(xyz)
        ref = [(det.labels(f), det.histogram(f), det.line(f), det.steps(f)[1]) for f in range(n)]
        assert ref[0][2] == '["stairs",["stairSteps",0]]' and (ref[0][0] == 255).all()
        det.process_depth_host(depth, k)
        for f in range(n):
            assert np.array_equal(det.labels(f), ref[f][0]) and np.array_equal(det.histogram(f), ref[f][1]), f
            assert det.line(f) == ref[f][2] and det.steps(f)[1] == ref[f][3], f
        assert sum(len(det.steps(f)[0]) > 0 for f in range(n)) >= 20


def test_hires_depth_input_equals_vertex_input(S):
    """4096x3072 z16 frame through the fused depth kernels (row / column of a pixel by the 2^40 magic multiply, 12.6 M
    pixels per frame) against the same frame as packed vertices: labels, histogram and steps identical."""
    w, h = 4096, 3072
    cfg = S.default_config(w, h, y_max=3.7, z_max=2.3)
    sc = S.default_scene(w, h, n_steps=12, riser=0.17, tread=0.26, cam_height=3.2, cam_pitch_deg=48.0, first_riser_y=0.5, **NOISY)
    xf = S.scene_transform(sc)
    depth = S.synth_depth_host(sc)
    xyz = S.deproject_host(sc, depth)
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.process_host(xyz[None])
        ref = (det.labels(0), det.histogram(0), det.line(0))
        assert len(det.steps(0)[0]) >= 5
        det.process_depth_host(depth[None], S.scene_intrinsics(sc))
        assert np.array_equal(det.labels(0), ref[0]) and np.array_equal(det.histogram(0), ref[1]) and det.line(0) == ref[2]


def test_overlay_projection_golden(S, oracle):
    """drawStairStep (pointcloud.cpp:583-597) on the GPU against what the compiled reference handed to drawQuadrilateral
    (tests/golden/overlay.json). The corners' x, y agree with the reference to ~1e-12 m, the step's mean z to ~1e-8 m
    (k_quad_reduce sums z in fixed point; the bar on heights is 0.1 mm), so a pixel can differ in its last f32 bits:
    the bar here is 2e-3 px (the consumer, drawQuadrilateral, rounds to whole pixels) and most values are bit-identical."""
    import json
    import os
    from test_oracle_golden import GOLDEN, load_case, load_overlay_golden
    gold = load_overlay_golden()
    n_val = n_exact = 0
    for path in GOLDEN:
        z, meta, sc, xf = load_case(path)
        g = gold[meta["name"]]
        cfg = S.default_config(meta["width"], meta["height"])
        fx, fy, ppx, ppy = g["intrinsics"]
        intr = A.Intrinsics(fx=fx, fy=fy, ppx=ppx, ppy=ppy)
        xyz = H.deproject_np(sc, z["depth"])
        with S.Detector(cfg, xf, max_frames=1) as det:
            with pytest.raises(S.SsdError):
                det.process_host(xyz[None])
                det.overlay(0)  # not enabled yet
            det.set_overlay(S.inverse3(xf.a), intr)
            det.process_host(xyz[None])
            ov = det.overlay(0)
            want = np.array(g["px_bits"], np.uint32).reshape(-1, 4, 2).view(np.float32)
            assert ov.shape == want.shape, meta["name"]
            assert len(ov) == len(det.steps(0)[0])
            if len(ov):
                assert np.abs(ov - want).max() < 0.01, meta["name"]
                n_val += ov.size
                n_exact += int((ov.view(np.uint32) == want.view(np.uint32)).sum())
            det.set_overlay(None, None)
            det.process_host(xyz[None])
            with pytest.raises(S.SsdError):
                det.overlay(0)
    assert n_val >= 6 * 4 * 8 and n_exact >= 0.5 * n_val, (n_exact, n_val)


def test_overlay_projection_batch(S, oracle):
    """the same on a batch of random scenes, vertex and z16 depth input, against the oracle (itself bit-identical to the
    compiled reference, tests/test_oracle_vs_ref.py::test_overlay_projection); a_inv as the reference's triangle ctor holds it"""
    w, h = 1024, 768
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    scenes = [S.randomize_scene(base, 31337, i, 3, 8) for i in range(12)]
    scenes[5].rotate180, scenes[5].n_occluders = 1, 2
    xf, a_inv = S.scene_transform_ex(scenes[0])
    assert np.abs(a_inv.reshape(3, 3) - np.array(xf.a[:]).reshape(3, 3).T).max() == 0  # rotation: _a = transposed(_aInv)
    intr = S.scene_intrinsics(scenes[0])
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    with S.Detector(cfg, xf, max_frames=len(scenes)) as det:
        det.set_overlay(a_inv, intr)
        det.process_host(xyz)
        got_v = [det.overlay(f) for f in range(len(scenes))]
        det.process_depth_host(depth, intr)
        got_d = [det.overlay(f) for f in range(len(scenes))]
    n_val = n_exact = 0
    for f in range(len(scenes)):
        H.oracle_process(oracle, cfg, xf, xyz[f])
        want = H.oracle_overlay(oracle, xf, a_inv, intr)
        assert got_v[f].shape == want.shape, f
        assert np.array_equal(got_v[f].view(np.uint32), got_d[f].view(np.uint32)), f  # depth input: identical results
        if len(want):
            assert np.abs(got_v[f] - want).max() < 2e-3, f
            n_val += want.size
            n_exact += int((got_v[f].view(np.uint32) == want.view(np.uint32)).sum())
    assert n_val >= 12 * 3 * 8 and n_exact >= 0.5 * n_val, (n_exact, n_val)


def test_camera_to_world_exact(S, oracle):
    cfg = S.default_config(320, 240)
    sc = S.default_scene(320, 240, cam_roll_deg=3.0, cam_yaw_deg=-7.0)
    xf = S.scene_transform(sc)
    rng = np.random.default_rng(7)
    pts = rng.normal(0, 1.5, (200000, 3)).astype(np.float32)
    with S.Detector(cfg, xf) as det:
        g = det.camera_to_world(pts)
    o = np.empty_like(g)
    oracle.ssd_oracle_camera_to_world(C.byref(xf), H.ptr(pts), len(pts), H.ptr(o))
    assert np.array_equal(g.view(np.uint64), o.view(np.uint64))


def random_quads(rng, n):
    for _ in range(n):
        c = rng.uniform(-0.3, 0.3, 2)
        w, d = rng.uniform(0.2, 0.6), rng.uniform(0.1, 0.5)
        q = np.array([[-w, -d], [w, -d], [-w, d], [w, d]]) * 0.5
        th = rng.uniform(-0.4, 0.4)
        R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        yield q @ R.T + c + rng.normal(0, 0.02, (4, 2))


def test_points_in_quad_exact(S, oracle):
    cfg = S.default_config(320, 240)
    xf = S.scene_transform(S.default_scene(320, 240))
    rng = np.random.default_rng(3)
    with S.Detector(cfg, xf) as det:
        quads = list(random_quads(rng, 40))
        quads.append(np.array([[0, 0], [1, 0], [0, 1], [1, 1.0]]))       # axis aligned
        quads.append(np.array([[0, 0], [1, 0], [1, 1], [0, 1.0]]))       # bow-tie: ctor throws
        quads.append(np.array([[0, 0], [1, 0], [0, 0], [1, 0.0]]))       # no y extent
        for q in quads:
            xy = rng.uniform(-0.8, 0.8, (50000, 2))
            xy[:8] = np.repeat(q, 2, axis=0)  # the vertices themselves
            g, gs = det.points_in_quad(q, xy)
            o = np.empty(len(xy), np.uint8)
            st = C.c_int()
            qq = (C.c_double * 8)(*q.ravel())
            oracle.ssd_oracle_points_in_quad(qq, H.ptr(xy), len(xy), H.ptr(o), C.byref(st))
            assert gs == st.value
            assert np.array_equal(g, o)


def blob_image(rng, w, h, kind):
    """binary BEV-like test images: filled quadrilaterals with ragged edges, holes and speckle"""
    yy, xx = np.mgrid[0:h, 0:w]
    cx, cy = w * rng.uniform(0.4, 0.6), h * rng.uniform(0.3, 0.8)
    hw, hh = w * rng.uniform(0.15, 0.45), h * rng.uniform(0.08, 0.3)
    th = rng.uniform(-0.15, 0.15)
    u = (xx - cx) * np.cos(th) + (yy - cy) * np.sin(th)
    v = -(xx - cx) * np.sin(th) + (yy - cy) * np.cos(th)
    img = ((np.abs(u) < hw) & (np.abs(v) < hh)).astype(np.uint8) * 255
    if kind >= 1:
        img[rng.random((h, w)) < 0.25] = 0           # dropouts (the close fills most)
    if kind >= 2:
        img[rng.random((h, w)) < 0.002] = 255        # speckle
    if kind == 3:
        img[:, : w // 2 - 30] = 0                    # cut: few scan columns on the left
    return img


@pytest.mark.parametrize("w,h", [(320, 240), (1024, 768), (2560, 1920)])  # the last: > 12 "smallest distances" per line fit
def test_outline_and_front_edge_images(S, oracle, w, h):
    cfg = S.default_config(w, h)
    xf = S.scene_transform(S.default_scene(w, h))
    rng = np.random.default_rng(11)
    der = H.Derived()
    oracle.ssd_oracle_derive(C.byref(cfg), C.byref(der))
    n_valid = 0
    with S.Detector(cfg, xf) as det:
        for i in range(24 if w <= 1024 else 12):
            img = blob_image(rng, w, h, i % 4)
            gq, gv = det.detect_outline(img, der.min_img_y_extent, der.xy_ratio)
            oq = (C.c_double * 8)()
            ov = C.c_int()
            oracle.ssd_oracle_detect_outline(H.ptr(img), w, h, der.min_img_y_extent, der.xy_ratio, oq, C.byref(ov))
            assert gv == ov.value, i
            assert np.allclose(gq, np.array(oq[:]).reshape(4, 2), rtol=0, atol=1e-7), i
            n_valid += gv
            gl, gr, gfv = det.detect_front_edge(img)
            ol = (C.c_double * 2)()
            orr = (C.c_double * 2)()
            ofv = C.c_int()
            oracle.ssd_oracle_detect_front_edge(H.ptr(img), w, h, ol, orr, C.byref(ofv))
            assert gfv == ofv.value, i
            assert np.allclose(gl, ol[:], rtol=0, atol=1e-7) and np.allclose(gr, orr[:], rtol=0, atol=1e-7), i
    assert n_valid >= 6


def test_device_input_and_determinism(S, oracle):
    """device-resident input (synthetic frames generated in HBM) gives the same results as host input,
    and two runs are bit-identical (fixed-point z accumulation)."""
    cfg = S.default_config(1024, 768)
    base = S.default_scene(1024, 768, **NOISY)
    xf = S.scene_transform(base)
    nF, N = 6, 1024 * 768
    with S.Detector(cfg, xf, max_frames=nF) as det:
        d_xyz = det.malloc(nF * N * 12)
        det.synth_frames(base, 99, 0, nF, 3, 8, d_xyz)
        xyz = np.empty((nF, N, 3), np.float32)
        det.d2h(xyz, d_xyz)
        det.process_device(d_xyz, nF)
        first = [(det.steps(f), det.labels(f).copy()) for f in range(nF)]
        det.process_device(d_xyz, nF)
        for f in range(nF):
            (s, st), lab = first[f]
            (s2, st2) = det.steps(f)
            assert st == st2 and len(s) == len(s2)
            for (h1, q1), (h2, q2) in zip(s, s2):
                assert h1 == h2 and np.array_equal(q1, q2)
            assert np.array_equal(lab, det.labels(f))
            g = gpu_result(S, det, f)
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            assert not H.compare_results(o, g, tol=TOL), f
        det.free(d_xyz)


@pytest.mark.parametrize("nF", [63, 64, 71])
def test_small_device_batch_split_over_streams(S, monkeypatch, nF):
    """a device-resident batch that fits one chunk is split over the two streams when each part keeps >= 32 frames
    (64 -> 2 x 32, 71 -> 36 + 35; 63 stays one chain): results, labels and result lines are identical to the unsplit
    run (SSD_GPU_NO_SPLIT_SMALL=1) and to the single-stream run"""
    w, h = 320, 240
    N = w * h
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    xf = S.scene_transform(base)
    with S.Detector(cfg, xf, max_frames=nF) as det:
        d_xyz = det.malloc(nF * N * 12)
        det.synth_frames(base, 5150, 0, nF, 3, 8, d_xyz)
        det.process_device(d_xyz, nF)
        split = [(det.line(f), det.labels(f).copy()) for f in range(nF)]
        monkeypatch.setenv("SSD_GPU_NO_SPLIT_SMALL", "1")
        det.process_device(d_xyz, nF)
        whole = [(det.line(f), det.labels(f).copy()) for f in range(nF)]
        monkeypatch.delenv("SSD_GPU_NO_SPLIT_SMALL")
        det.process_device(d_xyz, nF, flags=A.FLAG_SINGLE_STREAM)
        single = [(det.line(f), det.labels(f).copy()) for f in range(nF)]
        det.free(d_xyz)
    assert sum(l.count("height") for l, _ in split) > nF  # the frames do hold stairs
    for f in range(nF):
        assert split[f][0] == whole[f][0] == single[f][0], f
        assert np.array_equal(split[f][1], whole[f][1]) and np.array_equal(split[f][1], single[f][1]), f


def _all_lines(det, n):
    return [det.line(f) for f in range(n)]


def test_batch_properties_at_scale(S, oracle, monkeypatch):
    """Size-independent properties on a batch the oracle cannot afford (config 3 shape: 600 device-generated 1024x768
    frames, several chunks and streams): the result of a frame does not depend on the batch it travels in -- chunk
    size, stream count and batch position change nothing, bit for bit; label counts equal the plateau sizes;
    spot frames agree with the oracle."""
    W, Hh = 1024, 768
    N = W * Hh
    cfg = S.default_config(W, Hh)
    base = S.default_scene(W, Hh, **NOISY)
    xf = S.scene_transform(base)
    nF = 600
    ref_lines = None
    keep = {}
    for chunk, streams in ((256, 3), (37, 2), (600, 1)):
        monkeypatch.setenv("SSD_GPU_CHUNK_FRAMES", str(chunk))
        monkeypatch.setenv("SSD_GPU_STREAMS", str(streams))
        with S.Detector(cfg, xf, max_frames=nF) as det:
            d_xyz = det.malloc(nF * N * 12)
            det.synth_frames(base, 4242, 0, nF, 3, 8, d_xyz)
            det.process_device(d_xyz, nF)
            lines = _all_lines(det, nF)
            if ref_lines is None:
                ref_lines = lines
                assert sum(l.count("height") for l in lines) > 3 * nF  # stairs were found nearly everywhere
                for f in (0, 255, 256, 511, 599):
                    lab = det.labels(f)
                    hist = det.histogram(f)
                    info = det.frame_info(f)
                    plats, K = det.plateaus(f)
                    keep[f] = lab.copy()
                    # label counts == plateau sizes (sums of their histogram bands); invalid / out-of-range / remainder counts
                    in_plateaus = 0
                    for k in range(K):
                        assert int((lab == k).sum()) == plats[k].n_points, (f, k)
                        in_plateaus += plats[k].n_points
                    assert int((lab == 253).sum()) == info.n_in_range - in_plateaus
                    assert int((lab == 255).sum()) == N - info.n_nonzero
                    assert int((lab == 254).sum()) == info.n_nonzero - info.n_in_range
                    assert int(hist.sum()) == info.n_in_range
                    xyz = np.empty((N, 3), np.float32)
                    det.d2h(xyz, C.c_void_p(d_xyz.value + f * N * 12))
                    o = H.oracle_process(oracle, cfg, xf, xyz)
                    assert not H.compare_results(o, gpu_result(S, det, f), tol=TOL), f
                # a frame alone == the same frame inside the batch
                det.process_device(C.c_void_p(d_xyz.value + 300 * N * 12), 1)
                assert det.line(0) == ref_lines[300]
            else:
                assert lines == ref_lines, (chunk, streams)
                for f, lab in keep.items():
                    assert np.array_equal(det.labels(f), lab), (chunk, streams, f)
            det.free(d_xyz)


def test_descending_batch(S, oracle):
    """config 4 shape: upside-down camera (image rotated 180 degrees), occluders, a batch of frames; every frame against
    the oracle."""
    cfg = S.default_config(1024, 768)
    base = S.default_scene(1024, 768, rotate180=1, n_occluders=2, **NOISY)
    scenes = [S.randomize_scene(base, 515, i, 3, 8) for i in range(12)]
    res = run_frames(S, oracle, cfg, scenes)
    assert sum(g.info["n_steps"] for g, _ in res) > 12 * 2


def test_cpp_host_classes_main_loop(S, oracle, tmp_path):
    """the reference's main loop on the kept class surface (examples/detect_stairs_synthetic.cpp): same lines
    as the oracle for the same synthetic frames"""
    import json
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "detect_stairs_synthetic")
    libdir = os.path.join(root, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(root, "examples", "detect_stairs_synthetic.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h, n = 640, 480, 3
    run = subprocess.run([exe, str(w), str(h), str(n), "overlay"], capture_output=True, text=True, check=True)
    out = run.stdout.strip().splitlines()
    assert len(out) == n
    drawn = [[float(v) for v in l.split()[1:]] for l in run.stderr.splitlines() if l.startswith("overlay ")]
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    xf, a_inv = S.scene_transform_ex(base)
    intr = S.scene_intrinsics(base)
    for f in range(n):
        sc = S.randomize_scene(base, 2026, f, 3, 8)
        o = H.oracle_process(oracle, cfg, xf, S.deproject_host(sc, S.synth_depth_host(sc)))
        # Pointcloud::overlay(): the quadrilaterals drawStairStep projects into the camera image (printed with 6 digits)
        want = H.oracle_overlay(oracle, xf, a_inv, intr)
        mine = np.array([d[1:] for d in drawn if d[0] == f]).reshape(-1, 4, 2)
        assert mine.shape == want.shape and len(want) == len(o.steps)
        assert np.abs(mine - want).max() < 2e-3
        # Pointcloud::verticalFaces(): one line per riser (printed with 6 digits)
        ris = [[float(v) for v in l.split()[1:]] for l in run.stderr.splitlines() if l.startswith("riser ")]
        want_r = H.oracle_vertical_faces(oracle, cfg, xf, S.deproject_host(sc, S.synth_depth_host(sc)).reshape(-1, 3))
        mine_r = [r for r in ris if r[0] == f]
        assert len(mine_r) == len(want_r)
        for m, r in zip(mine_r, want_r):
            assert m[1] == r["lower_plateau"] and m[2] == r["n_points"] and abs(m[3] - r["y_mean"]) < 1e-4 * max(1.0, abs(r["y_mean"]))
        got = json.loads(out[f])
        assert got[0] == "stairs" and got[1] == ["stairSteps", len(o.steps)]
        for s, g in zip(o.steps, got[2] if len(o.steps) else []):
            assert abs(g[0][1] - s["height"]) < 1.1e-3
            assert np.abs(np.array(g[1][1:]) - s["quad"]).max() < 1.1e-3
