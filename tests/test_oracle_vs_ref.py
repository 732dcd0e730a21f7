"""CPU: the oracle against the reference's own code. Where the compiled reference is available (oracle/_ref, built by path
from the original project's sources named by SSD_REFERENCE_DIR) each test runs it live; otherwise it compares with what the
reference produced for the same seeded inputs, stored in tests/golden/reference_runs.json (make_reference_runs.py)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
# status bits the harness around the compiled reference does not raise (it reports only NO_STEPS / DEGENERATE_QUAD; the quirks
# themselves -- all-zero ground step, NaN mean, wrap -- are in the compared RESULTS)
QUIRKS = A.STATUS_BEV_OOB | A.STATUS_INVALID_FRONT_EDGE | A.STATUS_EMPTY_MEAN | A.STATUS_HMIN_WRAP | A.STATUS_TOO_MANY_PLATEAUS
RUNS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json")


def stored(key):
    """the reference's results for the seeded inputs of one test case"""
    with open(RUNS) as f:
        return json.load(f)["runs"][key]


class RefSource:
    """the reference's side of each comparison, from the compiled reference itself"""

    def __init__(self, S):
        self.S = S

    def lib(self, cfg):
        return H.load_ref(cfg)

    def frame(self, cfg, xf, xyz):
        return H.ref_process(self.lib(cfg), cfg, xf, xyz)

    def overlay(self, cfg, xf, xyz, intr):
        """intr None: the harness' default intrinsics"""
        ref = self.lib(cfg)
        ref.ssd_ref_set_intrinsics(C.byref(intr) if intr is not None else None)
        try:
            r = H.ref_process(ref, cfg, xf, xyz)
            px, label, z = H.ref_overlay(ref)
            a_inv = H.ref_a_inv(ref, xf)
        finally:
            ref.ssd_ref_set_intrinsics(None)
        ns = r.info["n_steps"]
        for k in range(ns):  # second pass labels: external-world corners and height (pointcloud.cpp:388-392)
            assert np.array_equal(label[ns + k], r.steps[k]["quad"][:2]) and z[ns + k] == r.steps[k]["height"]
        return dict(a_inv=[H.hexf(v) for v in a_inv], n_steps=ns, n_calls=len(px), px_bits=[int(v) for v in px.view(np.uint32).ravel()])

    def derived(self, cfg, px):
        ref = self.lib(cfg)
        mh, my, nb = C.c_int(), C.c_int(), C.c_int()
        xr, hir = C.c_double(), C.c_double()
        ref.ssd_ref_derived(C.byref(mh), C.byref(my), C.byref(xr), C.byref(hir), C.byref(nb))
        out = np.empty_like(px)
        ref.ssd_ref_image_to_world(H.ptr(px), len(px), H.ptr(out))
        return dict(min_height=mh.value, min_img_y_extent=my.value, n_bins=nb.value, xy_ratio=H.hexf(xr.value),
                    height_interval_reciprocal=H.hexf(hir.value), image_to_world_sha256=H.digest(out))

    def outline(self, img, w, h):
        ref = self.lib(self.S.default_config(w, h))
        q, l, r = (C.c_double * 8)(), (C.c_double * 2)(), (C.c_double * 2)()
        v, fv = C.c_int(), C.c_int()
        assert ref.ssd_ref_detect_outline(H.ptr(img), w, h, 20, 4 / 3, q, C.byref(v)) == 0, ref.ssd_ref_last_error()
        assert ref.ssd_ref_detect_front_edge(H.ptr(img), w, h, l, r, C.byref(fv)) == 0
        return dict(valid=v.value, quad=[H.hexf(x) for x in q], front_valid=fv.value, left=[H.hexf(x) for x in l], right=[H.hexf(x) for x in r])

    def points_in_quad(self, q, xy):
        ref = self.lib(self.S.default_config(320, 240))
        inside, st = np.empty(len(xy), np.uint8), C.c_int()
        ref.ssd_ref_points_in_quad((C.c_double * 8)(*q.ravel()), H.ptr(xy), len(xy), H.ptr(inside), C.byref(st))
        return dict(status=st.value, inside_sha256=H.digest(inside))


def source(S):
    """RefSource when the compiled reference can be loaded, else None (the tests then read the stored runs)"""
    return RefSource(S) if H.load_ref(S.default_config(320, 240)) is not None else None


def frames_random_scenes_inputs(S, w, h, n):
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, randomize_camera=1, **NOISY)
    for i in range(n):
        sc = S.randomize_scene(base, 99, i, 3, 8)
        if i % 3 == 2:
            sc.rotate180, sc.n_occluders = 1, 2
        yield cfg, S.scene_transform(sc), S.deproject_host(sc, S.synth_depth_host(sc))


@pytest.mark.parametrize("w,h,n", [(320, 240, 10), (640, 480, 6), (1024, 768, 3)])
def test_frames_random_scenes(S, oracle, w, h, n):
    src = source(S)
    want = None if src else stored(f"frames_random_scenes/{w}x{h}")
    for i, (cfg, xf, xyz) in enumerate(frames_random_scenes_inputs(S, w, h, n)):
        o = H.oracle_process(oracle, cfg, xf, xyz)
        r = H.frame_record(src.frame(cfg, xf, xyz), ~QUIRKS & 0xffffffff) if src else want[i]
        assert not H.compare_with_record(r, o, tol=1e-12), i
        assert (o.info["status"] & ~QUIRKS) == r["info"]["status"]
    assert oracle.ssd_oracle_sort_ties() == 0  # no rank tie that the reference's unstable sort could resolve differently


HIRES = dict(n_steps=12, riser=0.17, tread=0.26, cam_height=3.2, cam_pitch_deg=48.0, first_riser_y=0.5)
HIRES_CASES = [(2560, 1920, {}, {}, 2), (4096, 3072, dict(y_max=3.7, z_max=2.3), HIRES, 2)]


def frames_hires_inputs(S, w, h, ck, sk, n):
    cfg = S.default_config(w, h, **ck)
    base = S.default_scene(w, h, **sk, **NOISY)
    for i in range(n):
        sc = S.randomize_scene(base, 4141, i, sk.get("n_steps", 3), sk.get("n_steps", 8))
        yield cfg, S.scene_transform(base), S.deproject_host(sc, S.synth_depth_host(sc))


@pytest.mark.parametrize("w,h,ck,sk,n", HIRES_CASES)
def test_frames_hires(S, oracle, w, h, ck, sk, n):
    """BASELINE.json configs[4] (4096x3072, extended range: 241 height bins, ~83 points per BestLine list) and 2560x1920
    (more than 12 'smallest distances' per line fit): the restatement against the compiled reference, as pinned as the
    small sizes."""
    src = source(S)
    want = None if src else stored(f"frames_hires/{w}x{h}")
    for i, (cfg, xf, xyz) in enumerate(frames_hires_inputs(S, w, h, ck, sk, n)):
        o = H.oracle_process(oracle, cfg, xf, xyz)
        r = H.frame_record(src.frame(cfg, xf, xyz), ~QUIRKS & 0xffffffff) if src else want[i]
        assert not H.compare_with_record(r, o, tol=1e-12), i
        assert (o.info["status"] & ~QUIRKS) == r["info"]["status"]
        assert o.info["n_plateaus"] >= 3
    assert oracle.ssd_oracle_sort_ties() == 0


def overlay_inputs(S, w, h, n):
    """odd frames: the scene's intrinsics, even frames: None (the harness default, fx = fy = w at the image centre)"""
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, randomize_camera=1, **NOISY)
    for i in range(n):
        sc = S.randomize_scene(base, 777, i, 3, 8)
        if i % 3 == 2:
            sc.rotate180, sc.n_occluders = 1, 2
        yield cfg, S.scene_transform(sc), S.deproject_host(sc, S.synth_depth_host(sc)), S.scene_intrinsics(sc) if i % 2 else None


@pytest.mark.parametrize("w,h,n", [(320, 240, 6), (640, 480, 4), (1024, 768, 2)])
def test_overlay_projection(S, oracle, w, h, n):
    """drawStairStep (pointcloud.cpp:583-597): the quadrilaterals the reference hands to drawQuadrilateral, recorded by
    the harness' stub, against the oracle's restatement -- bit-exact f32 pixels; every step is drawn twice (depth and
    infrared viewport) with the same corners; labelling arguments as detectStairs passes them (checked live)."""
    src = source(S)
    want = None if src else stored(f"overlay_projection/{w}x{h}")
    for i, (cfg, xf, xyz, intr) in enumerate(overlay_inputs(S, w, h, n)):
        r = src.overlay(cfg, xf, xyz, intr) if src else want[i]
        if intr is None:
            intr = A.Intrinsics(fx=w, fy=w, ppx=w * 0.5, ppy=h * 0.5)
        o = H.oracle_process(oracle, cfg, xf, xyz)
        a_inv = np.empty(9)
        assert oracle.ssd_oracle_inverse3(xf.a, a_inv.ctypes.data_as(C.POINTER(C.c_double))) == 0
        assert np.array_equal(a_inv, H.unhexf(r["a_inv"]))
        assert np.array_equal(a_inv, S.inverse3(xf.a))  # host library: same inverse
        ov = H.oracle_overlay(oracle, xf, a_inv, intr)
        ns = r["n_steps"]
        assert ns == o.info["n_steps"] and ns > 0 and r["n_calls"] == 2 * ns and len(ov) == ns
        px = np.array(r["px_bits"], np.uint32).reshape(-1, 4, 2)
        assert np.array_equal(px[:ns], ov.view(np.uint32)), i
        assert np.array_equal(px[ns:], ov.view(np.uint32)), i
        assert np.isfinite(ov).all()


def derived_px(w):
    return np.random.default_rng(0).uniform(0, w, (1000, 2))


def test_derived_constants(S, oracle):
    src = source(S)
    for (w, h) in ((320, 240), (640, 480), (1024, 768)):
        cfg = S.default_config(w, h)
        px = derived_px(w)
        r = src.derived(cfg, px) if src else stored(f"derived_constants/{w}x{h}")
        d = H.Derived()
        assert oracle.ssd_oracle_derive(C.byref(cfg), C.byref(d)) == 0
        assert (d.min_height, d.min_img_y_extent, d.n_bins) == (r["min_height"], r["min_img_y_extent"], r["n_bins"])
        assert (d.xy_ratio, d.height_interval_reciprocal) == (H.unhexf(r["xy_ratio"]), H.unhexf(r["height_interval_reciprocal"]))
        assert d.min_height == 15 and d.n_bins == 121
        # Projection2D round trips through the reference
        exp = np.stack([cfg.x_min + px[:, 0] * d.x_to_world, cfg.y_max - px[:, 1] * d.y_to_world], 1)
        assert H.digest(exp) == r["image_to_world_sha256"]


def blob(rng, w, h, kind):
    yy, xx = np.mgrid[0:h, 0:w]
    cx, cy = w * rng.uniform(0.4, 0.6), h * rng.uniform(0.3, 0.8)
    hw, hh = w * rng.uniform(0.15, 0.45), h * rng.uniform(0.08, 0.3)
    th = rng.uniform(-0.15, 0.15)
    u = (xx - cx) * np.cos(th) + (yy - cy) * np.sin(th)
    v = -(xx - cx) * np.sin(th) + (yy - cy) * np.cos(th)
    img = ((np.abs(u) < hw) & (np.abs(v) < hh)).astype(np.uint8) * 255
    if kind >= 1:
        img[rng.random((h, w)) < 0.25] = 0
    if kind >= 2:
        img[rng.random((h, w)) < 0.002] = 255
    if kind == 3:
        img[:, : w // 2 - 30] = 0
    return img


def outline_inputs(w, h):
    rng = np.random.default_rng(5)
    for i in range(60):
        yield blob(rng, w, h, i % 4)


def test_outline_front_edge_fuzz(S, oracle):
    w, h = 320, 240
    src = source(S)
    want = None if src else stored("outline_front_edge_fuzz")
    nvalid = 0
    for i, img in enumerate(outline_inputs(w, h)):
        r = src.outline(img, w, h) if src else want[i]
        q1, v1 = (C.c_double * 8)(), C.c_int()
        assert oracle.ssd_oracle_detect_outline(H.ptr(img), w, h, 20, 4 / 3, q1, C.byref(v1)) == 0
        assert v1.value == r["valid"] and np.array_equal(np.array(q1[:]), H.unhexf(r["quad"])), i
        nvalid += v1.value
        l1, r1 = (C.c_double * 2)(), (C.c_double * 2)()
        assert oracle.ssd_oracle_detect_front_edge(H.ptr(img), w, h, l1, r1, C.byref(v1)) == 0
        assert v1.value == r["front_valid"], i
        assert np.array_equal(np.array(l1[:]), H.unhexf(r["left"])) and np.array_equal(np.array(r1[:]), H.unhexf(r["right"])), i
    assert nvalid > 10


def points_in_quad_inputs():
    rng = np.random.default_rng(9)
    quads = []
    for _ in range(200):
        c = rng.uniform(-0.3, 0.3, 2)
        wq, d = rng.uniform(0.2, 0.6), rng.uniform(0.1, 0.5)
        q = np.array([[-wq, -d], [wq, -d], [-wq, d], [wq, d]]) * 0.5
        th = rng.uniform(-0.8, 0.8)
        R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        quads.append(q @ R.T + c + rng.normal(0, 0.03, (4, 2)))
    quads += [np.array([[0, 0], [1, 0], [0, 1], [1, 1.0]]), np.array([[0, 0], [1, 0], [1, 1], [0, 1.0]]),
              np.array([[0, 0], [1, 0], [0, 0], [1, 0.0]]), np.array([[0, 0], [0, 0], [0, 1], [0, 1.0]])]
    for q in quads:
        xy = rng.uniform(-0.8, 0.8, (4000, 2))
        xy[:8] = np.repeat(q, 2, axis=0)
        yield q, xy


def test_points_in_quad_fuzz(S, oracle):
    src = source(S)
    want = None if src else stored("points_in_quad_fuzz")
    thrown = 0
    for i, (q, xy) in enumerate(points_in_quad_inputs()):
        r = src.points_in_quad(q, xy) if src else want[i]
        a, sa = np.empty(len(xy), np.uint8), C.c_int()
        oracle.ssd_oracle_points_in_quad((C.c_double * 8)(*q.ravel()), H.ptr(xy), len(xy), H.ptr(a), C.byref(sa))
        assert sa.value == r["status"]
        assert H.digest(a) == r["inside_sha256"]
        thrown += sa.value
    assert thrown >= 3


def test_close_matches_opencv(S, oracle):
    """the 3x3 MORPH_CLOSE restatements (oracle and the reference-build shim) against opencv-python"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2)
    ref = H.load_ref(S.default_config(320, 240))
    for (w, h) in ((320, 240), (37, 19), (64, 5), (3, 3)):
        for dens in (0.02, 0.3, 0.7):
            img = (rng.random((h, w)) < dens).astype(np.uint8) * 255
            exp = cv2.morphologyEx(img, cv2.MORPH_CLOSE, None)
            a = img.copy()
            assert oracle.ssd_oracle_close(H.ptr(a), w, h) == 0
            assert np.array_equal(a, exp)
            if ref is not None:
                b = img.copy()
                assert ref.ssd_ref_close(H.ptr(b), w, h) == 0
                assert np.array_equal(b, exp)
