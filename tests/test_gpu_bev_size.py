"""A BEV size of its own (ssd_gpu_create_bev, include/ssd_gpu.h): the frame size addresses the input, the labels and the depth
deprojection; the BEV size is the bird's-eye image the detector works in. A frame's results are defined by its points packed in
pixel order into k = ceil(N_frame / N_bev) BEV-size frames, the rest invalid (0,0,0): the oracle on that packing (one frame:
ssd_oracle_process, more: the group restatement tests/native/oracle_group.c) and the existing GPU path on it (the plain call, or a
one-camera group call) are the references."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

gpu = pytest.mark.gpu
TOL = 1e-4       # metres, as tests/test_gpu_parity.py
OVL_TOL = 2e-3   # pixels, as tests/test_gpu_distortion.py
ATOL = 1e-7      # BEV pixels, as tests/test_gpu_outline_fits.py
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)


# ---- the packing and its references ----
def bev_config(S, cfg, bev):
    """the configuration whose image (frame and BEV) is the BEV size, every other field cfg's"""
    c = S.default_config(*bev)
    for f, _ in A.Config._fields_:
        if f not in ("width", "height"):
            setattr(c, f, getattr(cfg, f))
    return c


def pack(xyz, bev):
    """one frame's points (N, 3) in pixel order -> (k, N_bev, 3), the rest invalid (0,0,0)"""
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    nb = bev[0] * bev[1]
    k = -(-len(xyz) // nb)
    out = np.zeros((k, nb, 3), np.float32)
    out.reshape(-1, 3)[:len(xyz)] = xyz
    return out


def oracle_of_packing(S, oracle, cfg_b, xf, packed):
    """the oracle's result of a packing: (FrameResult with the packing's labels flattened, status)"""
    if len(packed) == 1:
        return H.oracle_process(oracle, cfg_b, xf, packed[0])
    import test_gpu_groups as G
    g = G.oracle_group(cfg_b, [xf] * len(packed), packed)
    g.rec.labels = g.rec.labels.reshape(-1)
    return g.rec


def check_oracle(got, want, n, what):
    bad = H.compare_results(want, got, tol=TOL, check_labels=False)
    assert not bad, (what, bad)
    assert np.array_equal(got.labels, want.labels[:n]), what
    assert got.info["status"] == want.info["status"], what


def packed_gpu(S, cfg_b, cam, packed, options=None):
    """the existing GPU path on a packing: the plain call for one frame, else one group of one camera. Returns the result records
    with the labels (and step labels) of the members concatenated, the stats, and the detector's other per-frame results."""
    k = len(packed)
    with S.Detector(cfg_b, cam.xf, max_frames=k) as det:
        (options or (lambda d: None))(det)
        if k == 1:
            det.process_host(packed)
        else:
            det.set_cameras([cam])
            det.process_groups_host(packed, np.zeros(k, np.int32), [k])
        return collect(det, range(k))


def collect(det, frames):
    """everything of the record of frames[0] (the record every frame of a group shares), labels and step labels concatenated
    over frames"""
    frames = list(frames)
    r = H.gpu_result(det, frames[0])
    r.labels = np.concatenate([det.labels(f) for f in frames])
    st = det.stats()
    out = dict(rec=r, stats={k: getattr(st, k) for k in ("n_exact_fallback", "n_quad_fast", "n_quad_exact", "n_bev_exact")},
               n_points=st.n_points)
    if det._l.ssd_gpu_get_overlay(det._h, frames[0], None, 0, None) == 0:
        out["overlay"] = det.overlay(frames[0])
    if det._l.ssd_gpu_get_vertical_faces(det._h, frames[0], None, 0, None) == 0:
        out["risers"] = det.vertical_faces(frames[0])
    if det._l.ssd_gpu_get_step_surfaces(det._h, frames[0], None, 0, None) == 0:
        out["surfaces"] = det.step_surfaces(frames[0])
        out["step_labels"] = np.concatenate([det.step_labels(f) for f in frames])
    return out


def same_as_packed(got, want, n, what):
    """records exact, labels and step labels the packing's first n, stats equal except n_points"""
    a, b = got["rec"], want["rec"]
    b = H.FrameResult(b.labels[:n], b.hist, b.info, b.plateaus, b.steps, b.line)
    assert H.exact(a) == H.exact(b), what
    if "stats" in got:
        assert got["stats"] == want["stats"], what
    for k in ("risers", "surfaces"):
        assert (k in got) == (k in want) and got.get(k) == want.get(k), (what, k)
    if "step_labels" in want:
        assert np.array_equal(got["step_labels"], want["step_labels"][:n]), what
    if "overlay" in want:
        g, w = got["overlay"], want["overlay"]
        assert g.shape == w.shape and (g.size == 0 or np.abs(g - w).max() < OVL_TOL), what


def scene_frame(S, w, h, seed, lens=None, **kw):
    """one randomized noisy frame at w x h: (scene, z16 depth (h, w), vertices (h, w, 3) by the host deprojection)"""
    import test_gpu_distortion as D
    base = D.lens_scene(S, w, h, lens, **dict(NOISY, **kw))
    sc = S.randomize_scene(base, seed, 0, 3, 8)
    sc.distortion_model = base.distortion_model
    for i in range(5):
        sc.coeffs[i] = base.coeffs[i]
    d = S.synth_depth_host(sc)
    return sc, d, S.deproject_host(sc, d)


# ---- binding (no GPU) ----
def test_create_bev_is_declared_and_bound(S):
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    assert "int ssd_gpu_create_bev(const ssd_gpu_config *cfg, int32_t bev_width, int32_t bev_height" in hdr
    assert getattr(S.lib(), "ssd_gpu_create_bev").argtypes == A.PROTOTYPES["ssd_gpu_create_bev"][1]


def test_packing(S):
    xyz = np.arange(1024 * 768 * 3, dtype=np.float32).reshape(768, 1024, 3) + 1
    p = pack(xyz, (640, 480))
    assert p.shape == (3, 640 * 480, 3)
    assert np.array_equal(p.reshape(-1, 3)[:1024 * 768], xyz.reshape(-1, 3)) and not p.reshape(-1, 3)[1024 * 768:].any()
    assert pack(xyz[:240, :424], (640, 480)).shape == (1, 640 * 480, 3)


# ---- 1. the default is unchanged ----
def _run_everything(S, det, calls):
    out = []
    for name, call, n in calls:
        call()
        frames = []
        for f in range(n):
            r = H.gpu_result(det, f)
            frames.append((H.exact(r), det.overlay(f).tobytes(), det.vertical_faces(f), det.step_labels(f).tobytes(), det.step_surfaces(f)))
        st = det.stats()
        out.append((name, frames, bytes(st)))
    return out


@gpu
def test_create_bev_with_the_frame_size_is_create(S):
    import test_gpu_distortion as D
    w, h = 640, 480
    cfg = S.default_config(w, h)
    bases = [S.default_scene(w, h, **NOISY), S.default_scene(w, h, cam_pitch_deg=34.0, **NOISY)]
    lensed = D.lens_scene(S, w, h, D.BC, **NOISY)
    cams = [S.scene_camera(b) for b in bases + [lensed]]
    dist = [S.scene_distortion(b) for b in bases + [lensed]]
    scenes = [S.randomize_scene(bases[i % 2], 5, i, 3, 8) for i in range(4)]
    depth = np.stack([S.synth_depth_host(s) for s in scenes])
    xyz = np.stack([S.deproject_host(s, d) for s, d in zip(scenes, depth)])
    f32 = depth.astype(np.float32)
    intr = S.scene_intrinsics(bases[0])
    idx = np.array([0, 1, 2, 0], np.int32)
    results = []
    for make in ("create", "create_bev"):
        with S.Detector(cfg, cams[0].xf, max_frames=4, bev=None if make == "create" else (w, h)) as det:
            det.set_cameras(cams, dist)
            det.set_overlay(np.array(cams[0].a_inv[:]), cams[0].intr)
            det.set_vertical_faces(True)
            det.set_step_labels(True)
            det.set_step_surfaces(True)
            calls = [("vertices", lambda: det.process_host(xyz), 4),
                     ("z16", lambda: det.process_depth_host(depth, intr), 4),
                     ("float", lambda: det.process_depth_f32_host(f32, intr), 4),
                     ("cameras/z16", lambda: det.process_depth_cameras_host(depth, idx), 4),
                     ("groups/vertices", lambda: det.process_groups_host(xyz, idx, [1, 3]), 4),
                     ("groups/float", lambda: det.process_depth_f32_groups_host(f32, idx, [2, 2]), 4),
                     ("lens/z16", lambda: (det.set_distortion(S.scene_distortion(lensed)),
                                           det.process_depth_host(depth, S.scene_intrinsics(lensed))), 4)]
            results.append(_run_everything(S, det, calls))
            results[-1].append(det.chunk_frames)
    assert results[0] == results[1]


# ---- 2. the pixel layout of vertex input does not matter ----
@gpu
def test_pixel_layout_does_not_matter_for_vertex_input(S):
    w, h = 640, 480
    sc, _, xyz = scene_frame(S, w, h, 11)
    xf = S.scene_transform(sc)
    want = None
    for fw, fh in ((640, 480), (307200, 1), (19200, 16)):
        with S.Detector(S.default_config(fw, fh), xf, bev=(w, h)) as det:
            det.process_host(xyz.reshape(1, -1, 3))
            got = H.exact(H.gpu_result(det, 0))
        want = want or got
        assert got == want, (fw, fh)
    assert want[0]["info"]["n_steps"] >= 3


# ---- 3./4. frames larger and smaller than the BEV, against the oracle and the packed GPU path ----
SIZES = [((1280, 720), (640, 480)), ((1024, 768), (640, 480)), ((4096, 3072), (1024, 768)), ((424, 240), (640, 480)),
         ((640, 480), (2048, 1536))]


@gpu
@pytest.mark.parametrize("frame,bev", SIZES, ids=["%dx%d-bev%dx%d" % (f + b) for f, b in SIZES])
def test_frame_and_bev_sizes(S, oracle, frame, bev):
    w, h = frame
    sc, depth, xyz = scene_frame(S, w, h, 23 + w)
    xf = S.scene_transform(sc)
    cam = S.scene_camera(sc)
    cfg = S.default_config(w, h)
    cfg_b = bev_config(S, cfg, bev)
    n = w * h
    packed = pack(xyz, bev)
    want_o = oracle_of_packing(S, oracle, cfg_b, xf, packed)
    want_g = packed_gpu(S, cfg_b, cam, packed)
    assert want_g["n_points"] == len(packed) * bev[0] * bev[1]
    with S.Detector(cfg, xf, max_frames=2, bev=bev) as det:
        f32 = depth.astype(np.float32)
        intr = S.scene_intrinsics(sc)
        d_z16 = H.to_device(det, depth)
        for what, call in (("vertices/host", lambda: det.process_host(xyz[None])),
                           ("z16/host", lambda: det.process_depth_host(depth[None], intr)),
                           ("z16/device", lambda: det.process_depth_device(d_z16, intr, 1)),
                           ("float/host", lambda: det.process_depth_f32_host(f32[None], intr))):
            call()
            got = collect(det, [0])
            assert got["n_points"] == n
            check_oracle(got["rec"], want_o, n, what)
            same_as_packed(got, want_g, n, what)
        det.free(d_z16)
    assert any(p["outlined"] for p in want_o.plateaus), want_o.info
    if bev[0] * bev[1] <= 2 * n:  # (a 640x480 frame is too sparse on a 2048x1536 BEV for an outline to hold: no steps there)
        assert want_o.info["n_steps"] >= 2, want_o.info


@gpu
def test_lens_frame_larger_than_the_bev(S, oracle):
    """z16 through a Brown-Conrady lens: the reference packs the numpy restatement of the lens deprojection"""
    import test_gpu_distortion as D
    w, h, bev = 1280, 720, (640, 480)
    sc, depth, _ = scene_frame(S, w, h, 41, lens=D.BC)
    xyz = D.np_deproject(sc, depth, D.BC).astype(np.float32)
    cam = S.scene_camera(sc)
    cfg = S.default_config(w, h)
    cfg_b = bev_config(S, cfg, bev)
    packed = pack(xyz, bev)
    want_o = oracle_of_packing(S, oracle, cfg_b, cam.xf, packed)
    want_g = packed_gpu(S, cfg_b, cam, packed)
    with S.Detector(cfg, cam.xf, bev=bev) as det:
        det.set_distortion(S.scene_distortion(sc))
        det.process_depth_host(depth[None], S.scene_intrinsics(sc))
        got = collect(det, [0])
    check_oracle(got["rec"], want_o, w * h, "lens")
    same_as_packed(got, want_g, w * h, "lens")


# ---- 5. options, camera tables and groups under a BEV override ----
def _options(a_inv, intr):
    def apply(det):
        det.set_overlay(a_inv, intr)
        det.set_vertical_faces(True)
        det.set_step_labels(True)
        det.set_step_surfaces(True)
    return apply


def packed_group(S, cfg_b, cams, opts, xyz, cam_of_frame, bev):
    """the existing path on frames xyz (M, N, 3) of cameras cam_of_frame as one group: every frame packed to BEV-size frames, all
    packings one group of the camera table cams. Labels and step labels: each frame's packing's first N, frame after frame."""
    n, nb = xyz.shape[1], bev[0] * bev[1]
    packs = [pack(x, bev) for x in xyz]
    ks = [len(p) for p in packs]
    with S.Detector(cfg_b, cams[0].xf, max_frames=sum(ks)) as ref:
        ref.set_cameras(cams)
        opts(ref)
        ref.process_groups_host(np.concatenate(packs), np.repeat(np.asarray(cam_of_frame, np.int32), ks), [sum(ks)])
        want = collect(ref, range(sum(ks)))
    first = np.concatenate([[0], np.cumsum(ks)[:-1]])
    for key, arr in (("labels", want["rec"].labels), ("step_labels", want["step_labels"])):
        a = arr.reshape(sum(ks), nb)
        per = np.concatenate([a[f0:f0 + k].reshape(-1)[:n] for f0, k in zip(first, ks)])
        if key == "labels":
            want["rec"].labels = per
        else:
            want["step_labels"] = per
    return want


@gpu
@pytest.mark.parametrize("kind", ["vertices", "depth"])
def test_options_cameras_and_groups_under_a_bev_override(S, kind):
    """overlay, risers, step labels and surfaces through a camera call and a group call of 1280x720 frames on a 640x480 BEV, with
    two cameras of different poses and intrinsics: each frame (group) equals the packed groups of its camera(s) on the existing
    path, built from the frames' host deprojection. kind "depth": the camera call takes z16 frames and the group call float frames,
    so every frame is deprojected on the device with its own camera's tables (frame-size strides in the camera table)."""
    w, h, bev = 1280, 720, (640, 480)
    cfg = S.default_config(w, h)
    cfg_b = bev_config(S, cfg, bev)
    bases = [S.default_scene(w, h, **NOISY), S.default_scene(w, h, cam_pitch_deg=34.0, cam_height=0.9, **NOISY)]
    bases[1].fx, bases[1].fy = bases[1].fx * 1.07, bases[1].fy * 1.07
    bases[1].ppx, bases[1].ppy = bases[1].ppx + 23.0, bases[1].ppy - 11.0
    cams = [S.scene_camera(b) for b in bases]
    idx = np.array([1, 0, 1], np.int32)
    depth, xyz = [], []
    for i, c in enumerate(idx):
        sc = S.randomize_scene(bases[c], 77, i, 3, 8)
        assert bytes(S.scene_intrinsics(sc)) == bytes(cams[c].intr)  # each frame is its camera's
        depth.append(S.synth_depth_host(sc))
        xyz.append(S.deproject_host(sc, depth[-1]))
    depth, xyz = np.stack(depth), np.stack(xyz).reshape(len(idx), -1, 3)
    n = w * h
    opts = _options(np.array(cams[0].a_inv[:]), cams[0].intr)
    with S.Detector(cfg, cams[0].xf, max_frames=3, bev=bev) as det:
        det.set_cameras(cams)
        opts(det)
        # camera call: frame f against the packed one-camera group of its camera, the overlay through that camera
        if kind == "depth":
            det.process_depth_cameras_host(depth, idx)
        else:
            det.process_cameras_host(xyz, idx)
        got = [collect(det, [f]) for f in range(3)]
        # group call: frame 0 alone, frames 1 and 2 (two cameras) as one group
        if kind == "depth":
            det.process_depth_f32_groups_host(depth.astype(np.float32), idx, [1, 2])
        else:
            det.process_groups_host(xyz, idx, [1, 2])
        got_g0 = collect(det, [0])
        got_g = collect(det, [1, 2])
    # the stats count a whole call: each call's are the sum of its records' packed references
    call_stats = {"cameras": got[0]["stats"], "groups": got_g["stats"]}
    for r in got + [got_g, got_g0]:
        del r["stats"]
    want = [packed_group(S, cfg_b, cams, opts, xyz[f:f + 1], idx[f:f + 1], bev) for f in range(3)]
    for f in range(3):
        same_as_packed(got[f], want[f], n, (kind, "camera call", f))
    same_as_packed(got_g0, want[0], n, (kind, "group of one"))
    want_g = packed_group(S, cfg_b, cams, opts, xyz[1:], idx[1:], bev)
    same_as_packed(got_g, want_g, 2 * n, (kind, "group of two"))
    ref_stats = {"cameras": [r["stats"] for r in want], "groups": [want[0]["stats"], want_g["stats"]]}
    for call, st in call_stats.items():
        assert st == {k: sum(r[k] for r in ref_stats[call]) for k in st}, (kind, call)
    assert all(r["rec"].info["n_steps"] >= 2 for r in got + [got_g]), kind


# ---- 6. refusals ----
@gpu
def test_refusals(S):
    xf = S.scene_transform(S.default_scene(640, 480))
    h = C.c_void_p()

    def create(cfg, bw, bh):
        rc = S.lib().ssd_gpu_create_bev(C.byref(cfg), bw, bh, C.byref(xf), 0, 1, C.byref(h))
        if rc == 0:
            S.lib().ssd_gpu_destroy(h)
        return rc

    cfg = S.default_config(640, 480)
    assert create(cfg, 9349, 5109) == A.OK
    for bw, bh in ((9350, 480), (640, 5110), (12000, 6000)):
        assert create(cfg, bw, bh) == A.E_RANGE, (bw, bh)
    for bw, bh in ((0, 480), (640, 0), (-640, 480), (640, -1)):
        assert create(cfg, bw, bh) == A.E_INVALID_ARG, (bw, bh)
    assert create(S.default_config(641, 481), 640, 480) == A.E_INVALID_ARG          # N % 16 != 0
    assert create(S.default_config(9348 * 5108 + 16, 1), 640, 480) == A.E_RANGE    # above the largest frame
    assert create(S.default_config(9348 * 5108, 1), 640, 480) == A.OK
    assert create(S.default_config(1 << 20, 1 << 14), 640, 480) == A.E_RANGE        # int overflow of width * height is refused
    # depth input: W % 4 and N * W < 2^40 are refused, the previous results stay readable
    sc, _, xyz = scene_frame(S, 640, 480, 3)
    intr = S.scene_intrinsics(sc)
    for fw, fh in ((642, 480), (1 << 18, 16)):  # W % 4 == 2; N * W == 2^40
        with S.Detector(S.default_config(fw, fh), S.scene_transform(sc), bev=(640, 480)) as det:
            pts = np.zeros((fw * fh, 3), np.float32)
            pts[:640 * 480] = xyz.reshape(-1, 3)
            det.process_host(pts[None])
            before = H.exact(H.gpu_result(det, 0))
            assert before[0]["info"]["n_steps"] >= 3
            z = np.zeros(fw * fh, np.uint16)
            with pytest.raises(S.SsdError, match=r"\(-1\)"):
                det.process_depth_host(z[None], intr)
            with pytest.raises(S.SsdError, match=r"\(-1\)"):
                det.process_depth_f32_host(z[None].astype(np.float32), intr)
            assert H.exact(H.gpu_result(det, 0)) == before
    # (1 << 18) x 15 is below the bound: accepted
    with S.Detector(S.default_config(1 << 18, 15), S.scene_transform(sc), bev=(640, 480)) as det:
        det.process_depth_host(np.zeros((1, 15, 1 << 18), np.uint16), intr)
        assert det.frame_info(0).n_nonzero == 0


# ---- 7. the single-stage entry points take BEV images ----
@gpu
def test_single_stage_entry_points_take_bev_images(S):
    import outline_frames as O
    sc = S.default_scene(640, 480)
    for bev in ((640, 480), (1024, 768), (2048, 1536)):
        # a tread seen in perspective: a trapezoid, wider at the front (bottom) edge
        img = np.zeros((bev[1], bev[0]), np.uint8)
        y0, y1 = bev[1] // 5, bev[1] // 2
        for y in range(y0, y1):
            half = bev[0] // 5 + (y - y0) * bev[0] // (8 * (y1 - y0))
            img[y, bev[0] // 2 - half:bev[0] // 2 + half] = 1
        with S.Detector(S.default_config(4096, 3072), S.scene_transform(sc), bev=bev) as det:
            gq, gv = det.detect_outline(img, O.MIN_EXT, 1.0)
            oq, ov = O.run_outline(img, O.MIN_EXT, 1.0)
            assert gv == ov and np.allclose(gq, oq, rtol=0, atol=ATOL), (bev, gq, oq)
            gl, gr, gv = det.detect_front_edge(img)
            ol, orr, ov = O.run_front_edge(img)
            assert gv == ov and np.allclose(gl, ol, rtol=0, atol=ATOL) and np.allclose(gr, orr, rtol=0, atol=ATOL), bev


# ---- 8. the C++ host classes ----
@gpu
def test_cpp_configuration_binary_image(S, tmp_path):
    """tests/native/bev_size_check.cpp: a Pointcloud whose Configuration sets binaryImage prints the line of Detector(bev=...)"""
    exe = str(tmp_path / "bev_size_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "bev_size_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h, bw, bh = 1280, 720, 640, 480
    out = subprocess.run([exe, str(w), str(h), str(bw), str(bh)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    sc = S.default_scene(w, h, noise_sigma=0.0025)
    depth = S.synth_depth_host(sc)
    lines = []
    for bev in ((bw, bh), None):
        with S.Detector(S.default_config(w, h), S.scene_transform(sc), bev=bev) as det:
            det.process_depth_host(depth[None], S.scene_intrinsics(sc))
            lines.append(det.line(0))
    assert out == lines + ["refused", "refused"]
    assert lines[0].count("height") >= 2
