"""GPU: directed tests of the reference's degenerate behaviours that parity requires reproducing (SURVEY.md 5 / 8(a) notes):
hand-built vertex frames that force each SSD_STATUS_* bit, GPU (fused and seven-launch chain) against the C oracle and -- where it
survives the input -- the compiled reference (oracle/_ref). Every test asserts that the bit is actually set.

The frames are built in WORLD coordinates and pushed through an affine camera-to-world map that is the identity (or a pure
scale where the exact double value of a world coordinate matters), so that the world position of every point is known."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

pytestmark = pytest.mark.gpu
TOL = 1e-4
W, HH = 320, 240
N = W * HH


def identity_xf(sx=1.0):
    xf = A.Transform()
    for i, v in enumerate((sx, 0, 0, 0, 1, 0, 0, 0, 1)):
        xf.a[i] = float(v)
    xf.ext_a[0] = xf.ext_a[3] = 1.0
    return xf


def slab(rng, n, x0, x1, y0, y1, z, dz=0.0015):
    """n points of a horizontal surface at height z (inside one 1 cm bin)"""
    p = np.empty((n, 3), np.float32)
    p[:, 0] = rng.uniform(x0, x1, n)
    p[:, 1] = rng.uniform(y0, y1, n)
    p[:, 2] = z + rng.uniform(-dz, dz, n)
    return p


def frame_of(parts):
    """N x 3 frame: the parts, then invalid (0,0,0) vertices; a world z <= 0 would be dropped by the z > 0 filter, so the frame
    lives in a camera frame shifted by +1 m in z (b_z = -1)"""
    pts = np.concatenate(parts).astype(np.float32)
    assert len(pts) <= N, len(pts)
    out = np.zeros((N, 3), np.float32)
    out[:len(pts)] = pts
    out[:len(pts), 2] += 1.0
    return out


def shifted(xf):
    xf.b[2] = -1.0
    return xf


def run_paths(S, cfg, xf, xyz):
    """the frame through both forms of the chain: a one-frame host call takes the fused small-batch form (the peaks in
    k_transform_bin, the frame logic in k_outline); stage timing selects the seven-launch form with k_peaks and k_frame_logic
    at any batch size"""
    import test_gpu_parity as T
    res = {}
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.process_host(xyz[None])
        assert det.timing().n_launches == 5
        res["fused"] = H.gpu_result(det, 0)
        d = det.malloc(xyz.nbytes)
        try:
            det.h2d(d, xyz)
            det.process_device(d, 1, A.FLAG_STAGE_TIMING)
            assert det.timing().n_launches == 7
            res["seven-launch"] = H.gpu_result(det, 0)
        finally:
            det.free(d)
    return res


def check(S, oracle, cfg, xf, xyz, bit, ref_too=True, ref_mask=0):
    o = H.oracle_process(oracle, cfg, xf, xyz)
    assert o.info["status"] & bit, hex(o.info["status"])
    for path, g in run_paths(S, cfg, xf, xyz).items():
        assert g.info["status"] == o.info["status"], (path, hex(g.info["status"]), hex(o.info["status"]))
        bad = H.compare_results(o, g, tol=TOL)
        assert not bad, (path, bad)
    if ref_too and H.ref_available():
        ref = H.load_ref(cfg)
        r = H.ref_process(ref, cfg, xf, xyz)
        bad = H.compare_results(r, o, tol=1e-9)
        assert not bad, bad
        assert (r.info["status"] | ref_mask) == (o.info["status"] | ref_mask)
    return o


def test_hmin_wrap_empties_every_plateau(S, oracle):
    """SSD_STATUS_HMIN_WRAP: a peak at bin 1 with hist[0] > hist[2] -- heightMin - 1 wraps as uint16 (pointcloud.cpp:324), every
    remaining point falls into the remainder and that plateau and all later ones come out empty."""
    rng = np.random.default_rng(11)
    cfg = S.default_config(W, HH)
    parts = [slab(rng, 1500, -0.4, 0.4, 0.2, 0.6, -0.095), slab(rng, 4000, -0.4, 0.4, 0.2, 0.6, -0.085),  # bins 0 and 1
             slab(rng, 6000, -0.4, 0.4, 0.7, 1.1, 0.305)]                                               # a regular plateau above
    xyz = frame_of(parts)
    o = check(S, oracle, cfg, shifted(identity_xf()), xyz, A.STATUS_HMIN_WRAP, ref_mask=A.STATUS_HMIN_WRAP)
    assert o.info["n_plateaus"] == 2 and all(p["n_points"] == 0 for p in o.plateaus)
    assert not (o.labels < 32).any()


def test_more_peaks_than_plateau_slots(S, oracle):
    """SSD_STATUS_TOO_MANY_PLATEAUS: 35 histogram peaks; the ABI keeps the first 32 (the reference has no limit: not compared)."""
    rng = np.random.default_rng(12)
    cfg = S.default_config(W, HH)
    parts = [slab(rng, 2100, -0.5, 0.5, 0.2, 1.2, -0.1 + (1 + 3 * k + 0.5) * 0.01) for k in range(35)]
    xyz = frame_of(parts)
    o = check(S, oracle, cfg, shifted(identity_xf()), xyz, A.STATUS_TOO_MANY_PLATEAUS, ref_too=False)
    assert o.info["n_plateaus"] == 32


def test_ground_without_points_in_its_quadrilateral(S, oracle):
    """SSD_STATUS_INVALID_FRONT_EDGE: the ground plateau exists, but none of its points lies between y_min and the first step's
    front edge: calcGround finds no front edge and returns the all-zero quadrilateral, which is still emitted as a step
    (pointcloud.cpp:546, 442)."""
    rng = np.random.default_rng(13)
    cfg = S.default_config(W, HH)
    parts = [slab(rng, 9000, -0.45, 0.45, 1.0, 1.25, 0.004),   # ground only BEHIND the step
             slab(rng, 30000, -0.45, 0.45, 0.45, 0.75, 0.185)]  # one step
    xyz = frame_of(parts)
    o = check(S, oracle, cfg, shifted(identity_xf()), xyz, A.STATUS_INVALID_FRONT_EDGE, ref_mask=A.STATUS_INVALID_FRONT_EDGE)
    assert o.info["n_steps"] == 2 and o.steps[0]["height"] == 0.0 and not o.steps[0]["quad"].any()


def test_bev_pixel_past_the_image(S, oracle):
    """SSD_STATUS_BEV_OOB: Projection2D::worldToImage has no bounds check (pointcloud.cpp:81, 468). A world y one double-ulp
    above y_min is inside the measuring range, but (y_max - y) * yToImage rounds up to H: the reference writes past the end of
    the image (undefined behaviour there: not run); the ABI drops the pixel and raises the bit. World y = a11 * y_camera with
    y_camera = 0.5 and a11 = 2 * (that y), exact in binary."""
    rng = np.random.default_rng(14)
    cfg = S.default_config(W, HH)
    y2i = HH / (cfg.y_max - cfg.y_min)
    wy = cfg.y_min
    for _ in range(16):
        wy = float(np.nextafter(wy, 1.0))
        if int((cfg.y_max - wy) * y2i) == HH:
            break
    else:
        pytest.skip("no double above y_min whose pixel row rounds to H at this size")
    a11 = 2.0 * wy
    xf = shifted(identity_xf())
    xf.a[4] = a11
    step = slab(rng, 30000, -0.45, 0.45, 0.45 / a11, 0.75 / a11, 0.185)
    ground = slab(rng, 12000, -0.45, 0.45, 0.12 / a11, 0.44 / a11, 0.004)
    edge = np.array([[0.1, 0.5, 0.185], [-0.2, 0.5, 0.185]], np.float32)  # two points of the step's band on that y
    xyz = frame_of([step, ground, edge])
    o = H.oracle_process(oracle, cfg, xf, xyz)
    assert o.info["status"] & A.STATUS_BEV_OOB, hex(o.info["status"])
    assert o.info["n_steps"] >= 2
    for path, g in run_paths(S, cfg, xf, xyz).items():
        assert g.info["status"] == o.info["status"], (path, hex(g.info["status"]), hex(o.info["status"]))
        assert not H.compare_results(o, g, tol=TOL), path


def test_two_contexts_of_different_sizes_alternate(S, oracle):
    """ADVICE r1: the dynamic shared-memory attribute of k_outline / k_finalize is per function and process-wide; a context
    of a smaller frame size created later must not lower it for a live context of a larger one."""
    big_cfg, small_cfg = S.default_config(640, 480), S.default_config(320, 240)
    big_sc, small_sc = S.default_scene(640, 480, noise_sigma=0.0025), S.default_scene(320, 240, noise_sigma=0.0025)
    big_xf, small_xf = S.scene_transform(big_sc), S.scene_transform(small_sc)
    big_xyz = S.deproject_host(big_sc, S.synth_depth_host(big_sc))
    small_xyz = S.deproject_host(small_sc, S.synth_depth_host(small_sc))
    import test_gpu_parity as T
    with S.Detector(big_cfg, big_xf, max_frames=1) as big:
        with S.Detector(small_cfg, small_xf, max_frames=1) as small:
            for _ in range(2):
                small.process_host(small_xyz[None])
                big.process_host(big_xyz[None])
                assert not H.compare_results(H.oracle_process(oracle, big_cfg, big_xf, big_xyz), H.gpu_result(big, 0), tol=TOL)
                assert not H.compare_results(H.oracle_process(oracle, small_cfg, small_xf, small_xyz), H.gpu_result(small, 0), tol=TOL)


def test_misaligned_device_input_is_refused(S):
    cfg = S.default_config(320, 240)
    xf = S.scene_transform(S.default_scene(320, 240))
    with S.Detector(cfg, xf, max_frames=1) as det:
        d = det.malloc(N * 12 + 64)
        with pytest.raises(S.SsdError, match="aligned"):
            det.process_device(C.c_void_p(d.value + 4), 1)
        det.free(d)


def test_registered_host_buffer(S, oracle):
    """ssd_gpu_register_host: a caller-owned (pageable) frame buffer, page-locked in place, gives the same results"""
    cfg = S.default_config(640, 480)
    sc = S.default_scene(640, 480, noise_sigma=0.0025, dropout=0.03, n_holes=2)
    xf = S.scene_transform(sc)
    intr = S.scene_intrinsics(sc)
    depth = np.ascontiguousarray(S.synth_depth_host(sc)[None])
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.process_depth_host(depth, intr)
        a = det.steps(0)
        S.register_host(depth)
        try:
            det.process_depth_host(depth, intr)
            b = det.steps(0)
        finally:
            S.unregister_host(depth)
        assert a[1] == b[1] and len(a[0]) == len(b[0]) >= 3
        for (h0, q0), (h1, q1) in zip(a[0], b[0]):
            assert h0 == h1 and np.array_equal(q0, q1)
    with pytest.raises(S.SsdError):
        S.unregister_host(depth)  # not registered any more
