"""Depth frames of cameras with Brown-Conrady lenses (ssd_gpu_set_distortion / ssd_gpu_set_cameras_ex, include/ssd_gpu.h).

The lenses used throughout (coefficients k1, k2, p1, p2, k3 of the size real depth and colour streams report):
  BC  (SSD_DISTORTION_BROWN_CONRADY, 4):          [ 0.12, -0.08,  0.002,  -0.0015,  0.03]
  IBC (SSD_DISTORTION_INVERSE_BROWN_CONRADY, 2):  [-0.11,  0.06, -0.0012,  0.0018, -0.02]
The synthetic scene casts pixel (u, v) along its deprojected ray, so the frames of a distorted scene are what such a camera
delivers. z16 input with the lens declared must equal vertex input from the host deprojection of the same frames bit for bit."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

gpu = pytest.mark.gpu
TOL = 1e-4  # metres, as tests/test_gpu_parity.py
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
BC = (A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
IBC = (A.DISTORTION_INVERSE_BROWN_CONRADY, (-0.11, 0.06, -0.0012, 0.0018, -0.02))
LENSES = {"BC": BC, "IBC": IBC}
f32 = np.float32


def lens_scene(S, w, h, lens, **kw):
    sc = S.default_scene(w, h, **kw)
    if lens is not None:
        sc.distortion_model = lens[0]
        for i, c in enumerate(lens[1]):
            sc.coeffs[i] = c
    return sc


# ---- numpy restatement of the definition in include/ssd_gpu.h (float32 throughout, left to right) ----
def np_P(k, x, y):
    k1, k2, p1, p2, k3 = (f32(v) for v in k)
    two, one = f32(2), f32(1)
    r2 = x * x + y * y
    f = one + k1 * r2 + k2 * r2 * r2 + k3 * r2 * r2 * r2
    return x * f + two * p1 * x * y + p2 * (r2 + two * x * x), y * f + two * p2 * x * y + p1 * (r2 + two * y * y)


def np_Pinv(k, x0, y0):
    k1, k2, p1, p2, k3 = (f32(v) for v in k)
    two, one = f32(2), f32(1)
    x, y = x0, y0
    with np.errstate(all="ignore"):
        for _ in range(10):
            r2 = x * x + y * y
            icd = one / (one + ((k3 * r2 + k2) * r2 + k1) * r2)
            dx = two * p1 * x * y + p2 * (r2 + two * x * x)
            dy = two * p2 * x * y + p1 * (r2 + two * y * y)
            x, y = (x0 - dx) * icd, (y0 - dy) * icd
    return x, y


def np_deproject(sc, depth, lens):
    Hh, W = depth.shape
    u = np.broadcast_to(np.arange(W, dtype=f32)[None, :], (Hh, W))
    v = np.broadcast_to(np.arange(Hh, dtype=f32)[:, None], (Hh, W))
    x0 = (u - f32(sc.ppx)) / f32(sc.fx)
    y0 = (v - f32(sc.ppy)) / f32(sc.fy)
    if lens is None or lens[0] == A.DISTORTION_NONE or not any(lens[1]):
        x, y = x0, y0
    elif lens[0] == A.DISTORTION_INVERSE_BROWN_CONRADY:
        x, y = np_P(lens[1], x0, y0)
    else:
        x, y = np_Pinv(lens[1], x0, y0)
    z = depth.astype(f32) * f32(sc.depth_unit)
    return np.stack([z * x, z * y, z], -1)


def np_project(lens, X, Y, Z, intr):
    """drawStairStep's projection of camera point (X, Y, Z) through the lens (None: the pin-hole)"""
    x, y = X / Z, Y / Z
    if lens is None or lens[0] == A.DISTORTION_NONE:
        pass
    elif lens[0] == A.DISTORTION_INVERSE_BROWN_CONRADY:
        x, y = np_Pinv(lens[1], x, y)
    else:
        x, y = np_P(lens[1], x, y)
    return x * f32(intr.fx) + f32(intr.ppx), y * f32(intr.fy) + f32(intr.ppy)


def overlay_reference(oracle, cfg, xf, a_inv, intr, lens, xyz):
    """The overlay of one frame through the lens, restated in numpy: the oracle's steps mapped back from ToExternalWorld to the
    world frame in double precision (ext_a of these transforms is a rotation, so the round trip moves a corner by ~1e-16 m),
    WorldToCamera as the oracle evaluates it (a_inv * (p - b), left to right, narrowed to f32), then np_project.
    Returns (n_steps, 4, 2) float32."""
    o = H.oracle_process(oracle, cfg, xf, xyz)
    ea, eb = np.array(xf.ext_a[:]).reshape(2, 2), np.array(xf.ext_b[:])
    a, b = np.asarray(a_inv, np.float64).reshape(3, 3), np.array(xf.b[:])
    out = np.zeros((len(o.steps), 4, 2), np.float32)
    for s, st in enumerate(o.steps):
        z = st["height"] - xf.ext_z
        for c in range(4):
            x, y = np.linalg.solve(ea, st["quad"][c] - eb)
            d = (x - b[0], y - b[1], z - b[2])
            X, Y, Z = (f32((a[r, 0] * d[0] + a[r, 1] * d[1]) + a[r, 2] * d[2]) for r in range(3))
            with np.errstate(all="ignore"):
                out[s, c] = np_project(lens, X, Y, Z, intr)
    return out


# ---- host only ----
@pytest.mark.parametrize("size", [(640, 480), (1024, 768)])
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_host_deprojection_equals_numpy_and_overlay_reference(S, oracle, name, size):
    w, h = size
    lens = LENSES[name]
    sc = lens_scene(S, w, h, lens, **NOISY)
    depth = S.synth_depth_host(sc)
    # every pixel of the grid deprojects to a finite ray (depth set to 1 everywhere) ...
    ones = np.ones((h, w), np.uint16)
    grid = S.deproject_host(sc, ones)
    want = np_deproject(sc, ones, lens)
    assert np.isfinite(want).all() and grid.tobytes() == want.tobytes()
    # ... and the scene's own frame
    xyz = S.deproject_host(sc, depth)
    assert xyz.tobytes() == np_deproject(sc, depth, lens).tobytes()
    # the overlay reference of the GPU tests: without the lens it is the oracle's own overlay (the steps' round trip through
    # ToExternalWorld moves no projected corner by more than f32 rounding), with the lens it moves the corners by pixels
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(sc)
    intr = S.scene_intrinsics(sc)
    pin = overlay_reference(oracle, cfg, xf, a_inv, intr, None, xyz)
    oracle_pin = H.oracle_overlay(oracle, xf, a_inv, intr)
    assert len(pin) >= 3 and pin.shape == oracle_pin.shape and np.abs(pin - oracle_pin).max() < 1e-3
    assert np.abs(overlay_reference(oracle, cfg, xf, a_inv, intr, lens, xyz) - pin).max() > 0.5


@pytest.mark.parametrize("model", [A.DISTORTION_BROWN_CONRADY, A.DISTORTION_INVERSE_BROWN_CONRADY])
def test_zero_coefficients_are_the_pinhole(S, oracle, model):
    w, h = 640, 480
    pin = S.default_scene(w, h, **NOISY)
    zero = lens_scene(S, w, h, (model, (0.0,) * 5), **NOISY)
    d = S.synth_depth_host(zero)
    assert d.tobytes() == S.synth_depth_host(pin).tobytes()
    assert S.deproject_host(zero, d).tobytes() == S.deproject_host(pin, d).tobytes()
    # with zero coefficients P and P^-1 are the identity in f32 over the image (the definition's claim, both directions)
    u, v = np.meshgrid(np.arange(w, dtype=f32), np.arange(h, dtype=f32))
    x, y = (u - f32(pin.ppx)) / f32(pin.fx), (v - f32(pin.ppy)) / f32(pin.fy)
    for fn in (np_P, np_Pinv):
        px, py = fn((0.0,) * 5, x, y)
        assert px.tobytes() == x.tobytes() and py.tobytes() == y.tobytes()
    xf, a_inv = S.scene_transform_ex(pin)
    xyz = S.deproject_host(pin, d)
    cfg, intr = S.default_config(w, h), S.scene_intrinsics(pin)
    assert (overlay_reference(oracle, cfg, xf, a_inv, intr, (model, (0.0,) * 5), xyz).tobytes() ==
            overlay_reference(oracle, cfg, xf, a_inv, intr, None, xyz).tobytes())


@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_P_inverts_P_inverse_over_the_image(S, name):
    """P(P^-1(q)) == q within 1e-5 over every pixel of a 1024 x 768 L515-like frame (normalised radius up to 0.87): the ten
    fixed-point iterations converge geometrically at these coefficients. Worst case observed: BC 2.4e-7, IBC 1.8e-7 (about two
    float32 ulps of the coordinates)."""
    k = LENSES[name][1]
    sc = S.default_scene(1024, 768)
    u, v = np.meshgrid(np.arange(1024, dtype=f32), np.arange(768, dtype=f32))
    qx, qy = (u - f32(sc.ppx)) / f32(sc.fx), (v - f32(sc.ppy)) / f32(sc.fy)
    px, py = np_Pinv(k, qx, qy)
    rx, ry = np_P(k, px, py)
    worst = float(max(np.abs(rx - qx).max(), np.abs(ry - qy).max()))
    print(f"{name}: worst |P(P^-1(q)) - q| = {worst:.3g}")
    assert worst < 1e-5


def test_distortion_symbols_layout_and_values(S):
    assert C.sizeof(A.Distortion) == 24 and A.Distortion.coeffs.offset == 4
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    for name, val in (("NONE", 0), ("MODIFIED_BROWN_CONRADY", 1), ("INVERSE_BROWN_CONRADY", 2), ("FTHETA", 3), ("BROWN_CONRADY", 4),
                      ("KANNALA_BRANDT4", 5)):
        assert re.search(r"#define SSD_DISTORTION_%s %d\b" % (name, val), hdr), name
        assert getattr(A, "DISTORTION_" + name) == val
    for name in ("ssd_gpu_set_distortion", "ssd_gpu_set_cameras_ex", "ssd_gpu_n_ray_tables"):
        assert re.search(r"\b%s\(" % name, hdr) and name in A.PROTOTYPES, name
        assert getattr(S.lib(), name).argtypes == A.PROTOTYPES[name][1]
    d = S.scene_distortion(lens_scene(S, 64, 48, IBC))
    assert d.model == 2 and np.array_equal(np.array(d.coeffs[:], np.float32), np.array(IBC[1], np.float32))
    with pytest.raises(ValueError):
        S.make_distortion(4, (0.1,))


@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_scene_distortion_is_real(S, name):
    """A flat floor (no steps) seen through the lens: deprojected with the lens, every floor point lies on the floor plane within
    2 mm (depth quantisation 0.25 mm per count at up to ~3.5 m range, and the calibration's own float rounding); deprojected as
    pin-hole, the same depth puts image-edge points more than 1 cm off the plane."""
    w, h = 640, 480
    sc = lens_scene(S, w, h, LENSES[name], n_steps=0)
    d = S.synth_depth_host(sc)
    xf = S.scene_transform(sc)
    a, b = np.array(xf.a[:]).reshape(3, 3), np.array(xf.b[:])
    ok = d > 0
    assert ok.mean() > 0.5

    def off_plane(xyz):
        p = xyz[ok].astype(np.float64)
        return np.abs((p @ a.T + b)[:, 2] - sc.ground_z)

    with_lens = off_plane(S.deproject_host(sc, d))
    pin = S.default_scene(w, h, n_steps=0)
    as_pinhole = off_plane(S.deproject_host(pin, d))
    assert with_lens.max() < 2e-3, with_lens.max()
    assert as_pinhole.max() > 1e-2, as_pinhole.max()


# ---- GPU ----
def gpu_result(S, det, f):
    from test_gpu_parity import gpu_result as g
    return g(S, det, f)


def exact(r):
    return H.frame_record(r, 0xffffffff), r.line


def to_device(det, a):
    p = det.malloc(a.nbytes)
    det.h2d(p, a)
    return p


def lens_frames(S, w, h, lens, n, seed, cfg_kw=None, **kw):
    base = lens_scene(S, w, h, lens, **dict(NOISY, **kw))
    scenes = [S.randomize_scene(base, seed, i, 3, 8) for i in range(n)]
    depth = np.stack([S.synth_depth_host(s) for s in scenes])
    xyz = np.stack([S.deproject_host(s, dd) for s, dd in zip(scenes, depth)])
    return base, depth, xyz


@gpu
@pytest.mark.parametrize("size", [(640, 480), (1024, 768)])
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_lens_z16_equals_vertex_input(S, oracle, name, size):
    """z16 frames with the lens declared == the host deprojection as vertex input, bit for bit (labels, histograms, plateaus,
    steps, status, risers): plain and camera calls, host and device input. The vertex run agrees with the oracle."""
    w, h = size
    n = 4
    base, depth, xyz = lens_frames(S, w, h, LENSES[name], n, 31 + w)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(base)
    intr, dist = S.scene_intrinsics(base), S.scene_distortion(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_vertical_faces(True)
        det.process_host(xyz)
        want = [exact(gpu_result(S, det, f)) for f in range(n)]
        want_r = [det.vertical_faces(f) for f in range(n)]
        for f in range(n):
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            assert not H.compare_results(o, gpu_result(S, det, f), tol=TOL), f
            assert want_r[f] == H.oracle_vertical_faces(oracle, cfg, xf, xyz[f])
        assert sum(len(H.oracle_process(oracle, cfg, xf, xyz[f]).steps) for f in range(n)) >= 2 * n
        det.set_distortion(dist)
        d_z16 = to_device(det, depth)
        det.set_cameras([S.scene_camera(base)], [dist])
        runs = {"plain/host": lambda: det.process_depth_host(depth, intr),
                "plain/device": lambda: det.process_depth_device(d_z16, intr, n),
                "camera/host": lambda: det.process_depth_cameras_host(depth, np.zeros(n, np.int32)),
                "camera/device": lambda: det.process_depth_cameras_device(d_z16, np.zeros(n, np.int32), n)}
        for kind, run in runs.items():
            run()
            for f in range(n):
                assert exact(gpu_result(S, det, f)) == want[f], (kind, f)
                assert det.vertical_faces(f) == want_r[f], (kind, f)
        det.free(d_z16)


@gpu
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_lens_z16_4096x3072(S, name):
    w, h, n = 4096, 3072, 2
    base, depth, xyz = lens_frames(S, w, h, LENSES[name], n, 77, noise_sigma=0.0025, dropout=0.0, n_holes=0)
    cfg = S.default_config(w, h, y_max=3.7, z_max=2.3)
    xf = S.scene_transform(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.process_host(xyz)
        want = [exact(gpu_result(S, det, f)) for f in range(n)]
        det.set_distortion(S.scene_distortion(base))
        det.process_depth_host(depth, S.scene_intrinsics(base))
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want
        assert det.n_ray_tables == 1


@gpu
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_deproject_device_and_unfused_route(S, name, monkeypatch):
    w, h, n = 640, 480, 3
    base, depth, xyz = lens_frames(S, w, h, LENSES[name], n, 5)
    cfg = S.default_config(w, h)
    xf = S.scene_transform(base)
    intr, dist = S.scene_intrinsics(base), S.scene_distortion(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_distortion(dist)
        d_z16 = to_device(det, depth)
        d_xyz = det.malloc(xyz.nbytes)
        det.deproject_device(d_z16, intr, n, d_xyz)
        got = np.empty_like(xyz)
        det.d2h(got, d_xyz)
        assert got.tobytes() == xyz.tobytes()
        det.process_host(xyz)
        want = [exact(gpu_result(S, det, f)) for f in range(n)]
        det.free(d_z16)
        det.free(d_xyz)
    monkeypatch.setenv("SSD_GPU_DEPTH_UNFUSED", "1")
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_distortion(dist)
        det.process_depth_host(depth, intr)
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want


@gpu
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_overlay_through_the_lens(S, oracle, name):
    """the overlay with a lens agrees with overlay_reference (the oracle's steps through the numpy restatement of the lens) within
    2e-3 px (tests/test_gpu_parity.py's bar), plain and camera mode"""
    w, h, n = 640, 480, 4
    base, depth, xyz = lens_frames(S, w, h, LENSES[name], n, 11)
    cfg = S.default_config(w, h)
    xf, a_inv = S.scene_transform_ex(base)
    intr, dist = S.scene_intrinsics(base), S.scene_distortion(base)
    want = []
    for f in range(n):
        want.append(overlay_reference(oracle, cfg, xf, a_inv, intr, LENSES[name], xyz[f]))
    assert sum(len(q) for q in want) >= 2 * n
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_overlay(a_inv, intr)
        det.set_distortion(dist)
        for run in (lambda: det.process_host(xyz), lambda: det.process_depth_host(depth, intr)):
            run()
            for f in range(n):
                got = det.overlay(f)
                assert got.shape == want[f].shape and np.abs(got - want[f]).max() < 2e-3, f
        det.set_distortion(None)
        det.set_cameras([S.scene_camera(S.default_scene(w, h)), S.scene_camera(base)], [S.make_distortion(0), dist])
        det.process_depth_cameras_host(depth, np.ones(n, np.int32))
        for f in range(n):
            got = det.overlay(f)
            assert got.shape == want[f].shape and np.abs(got - want[f]).max() < 2e-3, f


@gpu
def test_mixed_lens_table_in_one_call(S):
    """one call over pin-hole, BC and IBC cameras, two of them sharing a lens: every frame equals a context of its own camera,
    and the pin-hole frames equal the plain call bit for bit although they ran through the lens kernels"""
    w, h = 1024, 768
    d = S.default_scene(w, h)
    other = dict(cam_pitch_deg=d.cam_pitch_deg + 4.0, cam_height=d.cam_height * 1.05)
    bases = [lens_scene(S, w, h, None, **NOISY),                       # 0 pin-hole
             lens_scene(S, w, h, BC, **NOISY),                         # 1 BC
             lens_scene(S, w, h, IBC, rotate180=1, **NOISY),           # 2 IBC, upside down
             lens_scene(S, w, h, BC, **dict(NOISY, **other)),          # 3 BC, camera 1's lens, another pose
             lens_scene(S, w, h, None, **dict(NOISY, **other))]        # 4 pin-hole, camera 0's intrinsics, another pose
    cams = [S.scene_camera(b) for b in bases]
    dists = [S.scene_distortion(b) for b in bases]
    order = np.array([0, 1, 2, 3, 4, 2, 1, 0, 4, 3], np.int32)
    scenes = []
    for i, c in enumerate(order):
        sc = S.randomize_scene(bases[c], 900, i, 3, 8)
        sc.rotate180 = bases[c].rotate180
        scenes.append(sc)
    depth = np.stack([S.synth_depth_host(s) for s in scenes])
    cfg = S.default_config(w, h)
    n = len(order)
    with S.Detector(cfg, cams[0].xf, max_frames=n) as det:
        det.set_cameras(cams, dists)
        assert det.n_ray_tables == 3  # pin-hole (cameras 0, 4), BC (1, 3), IBC (2)
        det.process_depth_cameras_host(depth, order)
        got = [exact(gpu_result(S, det, f)) for f in range(n)]
    for f, c in enumerate(order):
        with S.Detector(cfg, cams[c].xf, max_frames=1) as one:
            one.set_distortion(dists[c])
            one.process_depth_host(depth[f:f + 1], cams[c].intr)
            assert exact(gpu_result(S, one, 0)) == got[f], f
            if c in (0, 4):
                assert one.n_ray_tables == 0  # the plain pin-hole call: the existing kernels


@gpu
@pytest.mark.parametrize("model", [A.DISTORTION_BROWN_CONRADY, A.DISTORTION_INVERSE_BROWN_CONRADY])
def test_zero_coefficient_lens_runs_the_pinhole_kernels(S, model):
    w, h, n = 640, 480, 3
    base, depth, xyz = lens_frames(S, w, h, None, n, 3)
    cfg = S.default_config(w, h)
    xf = S.scene_transform(base)
    intr = S.scene_intrinsics(base)
    zero = S.make_distortion(model)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.process_depth_host(depth, intr)
        want = [exact(gpu_result(S, det, f)) for f in range(n)]
        launches = det.timing().n_launches
        det.set_distortion(zero)
        det.process_depth_host(depth, intr)
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want
        assert det.n_ray_tables == 0 and det.timing().n_launches == launches  # no ray table exists: the z16 kernels ran
        det.set_cameras([S.scene_camera(base)], [zero])
        det.process_depth_cameras_host(depth, np.zeros(n, np.int32))
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want
        assert det.n_ray_tables == 0


@gpu
def test_geometry_through_the_lens(S):
    """One staircase, one pose, no noise, through a pin-hole camera and a BC camera with the same fx, fy, ppx, ppy (1024 x 768).
    Bounds, derived before running: a step height is the mean z of thousands of tread points, each quantised to 0.25 mm of depth,
    and both renderings see the same planar treads, so heights agree to well under a millimetre: 2 mm. Corners come from the
    outlines of the BEV images, whose pixels are 1.2 m / 1024 = 1.2 mm by 1.2 m / 768 = 1.6 mm; the lens samples the edges at other
    points, which may move an outline by a few pixels: 1 cm (6 pixels). Not compared: the two front corners of the ground step.
    They lie on the near edge of the visible floor, which is the footprint of the image border and so depends on the lens's field
    of view, not on the scene. Declared pin-hole, the BC frame's points away from the image centre are misplaced by centimetres
    (test_scene_distortion_is_real), which must break at least one bound. Observed on a B200: with the lens, heights within
    0.3 mm and corners within 1.6 mm; declared pin-hole, heights off by up to 8.8 mm and corners by up to 10.5 mm."""
    w, h = 1024, 768
    pin = lens_scene(S, w, h, None, n_steps=4)
    bc = lens_scene(S, w, h, BC, n_steps=4)
    cfg = S.default_config(w, h)
    xf = S.scene_transform(pin)
    intr = S.scene_intrinsics(pin)
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.process_depth_host(S.synth_depth_host(pin)[None], intr)
        ref, _ = det.steps(0)
        d_bc = S.synth_depth_host(bc)[None]
        det.set_distortion(S.scene_distortion(bc))
        det.process_depth_host(d_bc, intr)
        lens, _ = det.steps(0)
        det.set_distortion(None)
        det.process_depth_host(d_bc, intr)
        naive, _ = det.steps(0)
    assert len(ref) >= 4

    def deltas(a):
        """(height difference, largest corner difference) per step; step 0 is the ground step"""
        return [(abs(x[0] - y[0]), float(np.abs((x[1] - y[1])[2 if i == 0 else 0:]).max())) for i, (x, y) in enumerate(zip(a, ref))]

    def within(a):
        return len(a) == len(ref) and all(dh < 2e-3 and dq < 1e-2 for dh, dq in deltas(a))

    print("lens", deltas(lens), "declared pin-hole", deltas(naive))
    assert within(lens), deltas(lens)
    assert not within(naive), deltas(naive)


@gpu
def test_errors_leave_results_and_table_in_place(S):
    w, h, n = 640, 480, 2
    base, depth, xyz = lens_frames(S, w, h, BC, n, 21)
    cfg = S.default_config(w, h)
    xf = S.scene_transform(base)
    intr, dist = S.scene_intrinsics(base), S.scene_distortion(base)
    # a lens whose P^-1 diverges at the image edge (large tangential terms): non-finite rays
    diverging = (A.DISTORTION_BROWN_CONRADY, (0.0, 0.0, 50.0, 50.0, 0.0))
    assert not np.isfinite(np_deproject(base, np.ones((h, w), np.uint16), diverging)).all()
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_cameras([S.scene_camera(base)], [dist])
        det.process_depth_cameras_host(depth, np.zeros(n, np.int32))
        want = [exact(gpu_result(S, det, f)) for f in range(n)]

        def unchanged():
            assert [exact(gpu_result(S, det, f)) for f in range(n)] == want
            assert det.n_cameras == 1 and det.n_ray_tables == 1

        for model in (1, 3, 5, 7):
            bad = S.make_distortion(model, (0.1, 0, 0, 0, 0))
            with pytest.raises(S.SsdError, match="model %d" % model):
                det.set_distortion(bad)
            with pytest.raises(S.SsdError, match="model %d" % model):
                det.set_cameras([S.scene_camera(base)], [bad])
            unchanged()
        with pytest.raises(S.SsdError, match="MODIFIED_BROWN_CONRADY"):
            det.set_distortion(S.make_distortion(1, (0.1, 0, 0, 0, 0)))
        nan = S.make_distortion(4, (0.1, float("nan"), 0, 0, 0))
        with pytest.raises(S.SsdError, match="not finite"):
            det.set_distortion(nan)
        with pytest.raises(S.SsdError, match="not finite"):
            det.set_cameras([S.scene_camera(base)], [nan])
        unchanged()
        div = S.make_distortion(*diverging)
        with pytest.raises(S.SsdError, match="diverges"):
            det.set_cameras([S.scene_camera(base)], [div])
        unchanged()
        det.set_distortion(div)  # the plain lens is checked against the intrinsics of the depth call
        with pytest.raises(S.SsdError, match="diverges"):
            det.process_depth_host(depth, intr)
        unchanged()
        # the camera table still works after the rejections
        det.process_depth_cameras_host(depth, np.zeros(n, np.int32))
        unchanged()


@gpu
def test_experimental_chain_rejects_a_distorted_depth_call(S, monkeypatch):
    w, h, n = 640, 480, 2
    base, depth, xyz = lens_frames(S, w, h, BC, n, 23)
    cfg = S.default_config(w, h)
    xf = S.scene_transform(base)
    intr = S.scene_intrinsics(base)
    monkeypatch.setenv("SSD_GPU_PATH", "records")
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.process_host(xyz)
        want = [exact(gpu_result(S, det, f)) for f in range(n)]
        det.set_distortion(S.scene_distortion(base))
        with pytest.raises(S.SsdError, match=r"\(-5\)"):
            det.process_depth_host(depth, intr)
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want
        det.process_host(xyz)  # vertex input without overlay does not use the lens
        assert [exact(gpu_result(S, det, f)) for f in range(n)] == want


@gpu
def test_cpp_host_classes_with_lenses(S, tmp_path):
    """tests/native/distortion_check.cpp: DepthFrame(z16, intrinsics, distortion, w, h) and addCamera(..., distortion) print the
    lines the Python binding gives for the same frames"""
    exe = str(tmp_path / "distortion_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "distortion_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h = 640, 480
    out = subprocess.run([exe, str(w), str(h)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == 6
    bases = [lens_scene(S, w, h, BC, noise_sigma=0.0025), lens_scene(S, w, h, IBC, noise_sigma=0.0025)]
    bases[1].cam_pitch_deg = float(f32(bases[1].cam_pitch_deg) + f32(4.0))
    bases[1].fx = float(f32(bases[1].fx) * f32(1.05))
    depth = np.stack([S.synth_depth_host(S.randomize_scene(bases[f % 2], 99, f, 3, 8)) for f in range(4)])
    cfg = S.default_config(w, h)
    lines = []
    for c in range(2):
        with S.Detector(cfg, S.scene_transform(bases[c]), max_frames=1) as det:
            det.set_distortion(S.scene_distortion(bases[c]))
            det.process_depth_host(depth[c:c + 1], S.scene_intrinsics(bases[c]))
            lines.append(det.line(0))
    with S.Detector(cfg, S.scene_transform(bases[0]), max_frames=4) as det:
        det.set_cameras([S.scene_camera(b) for b in bases], [S.scene_distortion(b) for b in bases])
        det.process_depth_cameras_host(depth, np.array([0, 1, 0, 1], np.int32))
        lines += [det.line(f) for f in range(4)]
    assert out == lines
    assert all(l.count("height") >= 2 for l in lines)
