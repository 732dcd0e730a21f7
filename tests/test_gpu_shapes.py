"""Frame sizes and configurations outside the ones the rest of the suite runs: RealSense D400 depth modes whose BEV rows end in a
partial 32-bit word (848x480: 26.5 words per row, 424x240: 13.25), frames on either side of the k_outline size-class boundary
(W / 50 + 6 <= 32 and H / 10 + 2 <= 112: 1348x1108 fills both fixed line-point lists exactly, 1352x1108 and 1348x1112 are the
first hi-res frames), narrow frames with one or two words per BEV row, a width that is not a multiple of 4 (vertex input only),
and configurations whose derived constants (n_bins, min_height, min_img_y_extent, the filter bounds) differ from the defaults.

Every size runs vertex, z16 host and z16 device input, a Brown-Conrady lens, a two-camera table, the fused and the seven-launch
chain, the overlay and the risers; every result is compared with the oracle (oracle/ssd_oracle.c) or, for inputs that
deproject to the same vertices, with the vertex run bit for bit."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

TOL = 1e-4  # metres, as tests/test_gpu_parity.py
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
BC = (A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
gpu = pytest.mark.gpu

# width, height, configuration overrides, whether the oracle finds steps in the default scene
SIZES = {
    "848x480": (848, 480, {}, True),
    "424x240": (424, 240, {}, True),
    "1280x720": (1280, 720, {}, True),
    "1348x1108": (1348, 1108, {}, True),   # largest small-class frame: W / 50 + 6 == 32, H / 10 + 2 == 112
    "1352x1108": (1352, 1108, {}, True),   # hi-res class by width
    "1348x1112": (1348, 1112, {}, True),   # hi-res class by height
    "64x128": (64, 128, dict(x_min=-0.4, x_max=0.4, min_peak_points=40), True),  # two words per BEV row
    "32x64": (32, 64, dict(x_min=-0.4, x_max=0.4, min_peak_points=40), False),   # one word per BEV row: no valid outline
    "322x240": (322, 240, {}, True),       # W % 4 != 0: vertex input only
}


def size_case(S, key, n):
    w, h, kw, _ = SIZES[key]
    cfg = S.default_config(w, h, **kw)
    base = S.default_scene(w, h, **NOISY)
    scenes = [S.randomize_scene(base, 1000 + w + h, i, 3, 8) for i in range(n)]
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    return cfg, base, depth, xyz


def test_size_class_boundaries_are_where_the_sizes_claim():
    """the sizes sit where their comments put them: partial last BEV word, the k_outline size-class boundary. This restates
    ssd_gpu.cu's outline_small condition to document the choice of sizes; which class the library picks is not observable
    through the ABI, and the GPU tests at these sizes check the results of either class"""
    for key in ("848x480", "424x240", "322x240"):
        assert SIZES[key][0] % 32 != 0, key
    small = lambda w, h: w // 25 + 4 <= 64 and w // 50 + 6 <= 32 and h // 10 + 2 <= 112  # ssd_gpu.cu: outline_small
    assert small(1348, 1108) and 1348 // 50 + 6 == 32 and 1108 // 10 + 2 == 112
    assert not small(1352, 1108) and not small(1348, 1112)
    assert (SIZES["64x128"][0] + 31) // 32 == 2 and (SIZES["32x64"][0] + 31) // 32 == 1


@pytest.mark.parametrize("key", list(SIZES))
def test_oracle_finds_the_steps(S, oracle, key):
    """the default scene at each size: the oracle finds ground + 3 steps where the size allows an outline"""
    w, h, kw, steps = SIZES[key]
    cfg = S.default_config(w, h, **kw)
    sc = S.default_scene(w, h)
    o = H.oracle_process(oracle, cfg, S.scene_transform(sc), S.deproject_host(sc, S.synth_depth_host(sc)))
    assert (o.info["n_steps"] == 4) if steps else (o.info["n_steps"] == 0), o.info


@gpu
@pytest.mark.parametrize("key", list(SIZES))
def test_sizes_every_input_kind(S, oracle, key):
    """a batch of randomized scenes: vertex input against the oracle (results, overlay, risers); the fused chain (one call of
    at most 16 frames) against the seven-launch chain (stage timing); z16 host / device input and a two-camera table call
    against the vertex run, bit for bit; widths that are not a multiple of 4 refuse depth input"""
    w, h, _, steps = SIZES[key]
    n = 4 if w * h <= 1400 * 1120 else 2
    cfg, base, depth, xyz = size_case(S, key, n)
    xf, a_inv = S.scene_transform_ex(base)
    intr = S.scene_intrinsics(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_overlay(a_inv, intr)
        det.set_vertical_faces(True)

        def everything():
            return [(H.exact(H.gpu_result(det, f)), det.overlay(f).tobytes(), det.vertical_faces(f)) for f in range(n)]

        det.process_host(xyz)
        fused = det.timing().n_launches  # five, plus the overlay's k_finalize
        want = everything()
        n_steps = 0
        for f in range(n):
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            g = H.gpu_result(det, f)
            assert not H.compare_results(o, g, tol=TOL), (f, H.compare_results(o, g, tol=TOL))
            assert g.info["status"] == o.info["status"], f
            ov = H.oracle_overlay(oracle, xf, a_inv, intr)
            got = det.overlay(f)
            assert got.shape == ov.shape, f
            if len(ov):
                assert np.abs(got - ov).max() < 2e-3, f
            assert det.vertical_faces(f) == H.oracle_vertical_faces(oracle, cfg, xf, xyz[f].reshape(-1, 3)), f
            n_steps += o.info["n_steps"]
        if steps:
            assert n_steps >= 3 * n
        d_xyz = H.to_device(det, xyz)
        det.process_device(d_xyz, n, A.FLAG_STAGE_TIMING)
        assert det.timing().n_launches == fused + 2  # k_peaks and k_frame_logic as launches of their own
        assert everything() == want, "seven-launch chain"
        # camera 1 of the table is this context's own; the even frames go through camera 0, another mounting, and are
        # compared with the oracle run with its transform
        other, _ = S.scene_transform_ex(S.default_scene(w, h, cam_height=base.cam_height * 1.1, cam_pitch_deg=base.cam_pitch_deg + 3))
        det.set_cameras([S.make_camera(other), S.scene_camera(base)])
        cof = (np.arange(n) % 2).astype(np.int32)
        det.process_cameras_device(d_xyz, cof, n)
        for f in range(n):
            if cof[f]:
                assert H.exact(H.gpu_result(det, f)) == want[f][0], ("camera table, own camera", f)
            else:
                o = H.oracle_process(oracle, cfg, other, xyz[f])
                g = H.gpu_result(det, f)
                assert not H.compare_results(o, g, tol=TOL) and g.info["status"] == o.info["status"], ("camera table, camera 0", f)
        det.free(d_xyz)
        if w % 4:
            for call in (lambda: det.process_depth_host(depth, intr), lambda: det.process_depth_cameras_host(depth, np.ones(n))):
                with pytest.raises(S.SsdError, match=r"\(-1\).*multiple of 4"):
                    call()
            return
        d_z16 = H.to_device(det, depth)
        for kind, run in (("z16 host", lambda: det.process_depth_host(depth, intr)),
                          ("z16 device", lambda: det.process_depth_device(d_z16, intr, n)),
                          ("z16 camera table", lambda: det.process_depth_cameras_device(d_z16, np.ones(n, np.int32), n))):
            run()
            assert everything() == want, kind
        det.free(d_z16)


@gpu
@pytest.mark.parametrize("key", [k for k in SIZES if SIZES[k][0] % 4 == 0])
def test_sizes_lens_frame(S, oracle, key):
    """one Brown-Conrady frame per size: z16 with the lens declared equals the host deprojection as vertex input, which
    equals the oracle"""
    w, h, kw, _ = SIZES[key]
    cfg = S.default_config(w, h, **kw)
    base = S.default_scene(w, h, **NOISY)
    base.distortion_model = BC[0]
    for i, c in enumerate(BC[1]):
        base.coeffs[i] = c
    depth = S.synth_depth_host(base)[None]
    xyz = S.deproject_host(base, depth[0])[None]
    xf = S.scene_transform(base)
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.set_vertical_faces(True)
        det.process_host(xyz)
        want = (H.exact(H.gpu_result(det, 0)), det.vertical_faces(0))
        o = H.oracle_process(oracle, cfg, xf, xyz[0])
        assert not H.compare_results(o, H.gpu_result(det, 0), tol=TOL)
        det.set_distortion(S.scene_distortion(base))
        det.process_depth_host(depth, S.scene_intrinsics(base))
        assert (H.exact(H.gpu_result(det, 0)), det.vertical_faces(0)) == want


# ---- configurations (640x480) ----
CONFIGS = {
    "interval_0.005": (dict(height_interval=0.005), {}, True),
    "interval_0.02": (dict(height_interval=0.02), {}, True),
    "interval_0.007": (dict(height_interval=0.007), {}, True),                # 1 / 0.007 is not exact
    "n_bins_253": (dict(z_min=-0.1, z_max=2.425), {}, True),  # (z_max - z_min) / 0.01 + 1 = 253, the cap
    "n_bins_3": (dict(z_min=-0.1, z_max=-0.075), {}, False),
    "asymmetric_xy": (dict(x_min=-0.35, x_max=0.8, y_min=0.25, y_max=1.45), dict(x_center=0.2, first_riser_y=0.55), True),
    "z_min_0": (dict(z_min=0.0), dict(ground_z=0.004), True),
    "z_min_-0.35": (dict(z_min=-0.35), {}, True),
    "min_height_0": (dict(min_height_above_ground=0.0), {}, True),
    "min_height_0.2": (dict(min_height_above_ground=0.2), {}, True),
    "min_step_depth_0.05": (dict(min_step_depth=0.05), {}, True),
    "min_step_depth_0.25": (dict(min_step_depth=0.25), {}, True),
    "min_peak_points_20": (dict(min_peak_points=20), {}, True),
    "min_peak_points_20000": (dict(min_peak_points=20000), {}, True),
}


def config_case(S, key, n=4):
    ckw, skw, _ = CONFIGS[key]
    w, h = 640, 480
    cfg = S.default_config(w, h, **ckw)
    base = S.default_scene(w, h, **dict(NOISY, **skw))
    scenes = [S.randomize_scene(base, 4000 + len(key), i, 3, 6) for i in range(n)]
    for sc in scenes:  # randomize_scene draws the stairs' placement: keep the overrides that put them in range
        for k, v in skw.items():
            setattr(sc, k, v)
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    return cfg, base, depth, xyz


def test_config_derived_constants(S, oracle):
    """the configurations reach what their names claim (n_bins at the cap and at the minimum)"""
    for key, want in (("n_bins_253", 253), ("n_bins_3", 3)):
        der = H.Derived()
        assert oracle.ssd_oracle_derive(C.byref(S.default_config(640, 480, **CONFIGS[key][0])), C.byref(der)) == 0, key
        assert der.n_bins == want, (key, der.n_bins)


@pytest.mark.parametrize("key", list(CONFIGS))
def test_config_oracle_finds_steps(S, oracle, key):
    cfg, base, depth, xyz = config_case(S, key)
    xf = S.scene_transform(base)
    n = sum(H.oracle_process(oracle, cfg, xf, x).info["n_steps"] for x in xyz)
    if CONFIGS[key][2]:
        assert n >= 2 * len(xyz), (key, n)
    else:
        assert n == 0, (key, n)


@gpu
@pytest.mark.parametrize("key", list(CONFIGS))
def test_configurations(S, oracle, key):
    """vertex input against the oracle, z16 input against the vertex run; fused and seven-launch chains"""
    cfg, base, depth, xyz = config_case(S, key)
    n = len(xyz)
    xf = S.scene_transform(base)
    intr = S.scene_intrinsics(base)
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.set_vertical_faces(True)
        det.process_host(xyz)
        want = [(H.exact(H.gpu_result(det, f)), det.vertical_faces(f)) for f in range(n)]
        for f in range(n):
            o = H.oracle_process(oracle, cfg, xf, xyz[f])
            g = H.gpu_result(det, f)
            assert not H.compare_results(o, g, tol=TOL), (f, H.compare_results(o, g, tol=TOL))
            assert g.info["status"] == o.info["status"], f
            assert want[f][1] == H.oracle_vertical_faces(oracle, cfg, xf, xyz[f].reshape(-1, 3)), f
        d_z16 = H.to_device(det, depth)
        for kind, run in (("z16 host", lambda: det.process_depth_host(depth, intr)),
                          ("z16 device", lambda: det.process_depth_device(d_z16, intr, n))):
            run()
            assert [(H.exact(H.gpu_result(det, f)), det.vertical_faces(f)) for f in range(n)] == want, kind
        det.free(d_z16)
