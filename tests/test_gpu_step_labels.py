"""Step labels (ssd_gpu_set_step_labels, include/ssd_gpu.h): per pixel the step whose height its point is averaged into -- the set
StairsDetector::getPointsInQuadrilateral returns for the step (pointcloud.cpp:560-572) -- or SSD_STEP_LABEL_NONE.

The reference map is built from pinned oracle primitives: the oracle's labels, frame info and plateaus, then for every emitted
step's plateau its pixels through ssd_oracle_camera_to_world and ssd_oracle_points_in_quad(quad_world). Without a GPU the map is
checked against the oracle's and the compiled reference's n_in_quad; on the GPU every map is compared with it pixel for pixel."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

gpu = pytest.mark.gpu
NONE = A.STEP_LABEL_NONE
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)


# ---- the reference map ----
def step_plateaus(info, plats):
    """plateau index of each emitted step (k_finalize / detectStairSteps order): the ground, when it is a step with a usable
    quadrilateral, then the valid plateaus with a usable quadrilateral, ascending"""
    get = (lambda p, k: p[k]) if isinstance(plats[0] if len(plats) else {}, dict) else getattr
    K, g, fv = info["n_plateaus"], info["ground_index"], info["first_valid_index"]
    out = []
    if fv < 0:
        return out
    if g >= 0 and get(plats[g], "quad_status") == 0:
        out.append(g)
    out += [l for l in range(fv, K) if get(plats[l], "valid") and get(plats[l], "quad_status") == 0]
    return out


def reference_map(oracle, xfs, xyz, labels, info, plats):
    """step labels of the member frames (M, N): xfs / xyz (M, N, 3) / labels (M, N) per member, info / plats of the record"""
    M = len(xfs)
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(M, -1, 3)
    labels = np.asarray(labels).reshape(M, -1)
    out = np.full(labels.shape, NONE, np.uint8)
    for s, l in enumerate(step_plateaus(info, plats)):
        q = np.ascontiguousarray(np.asarray(plats[l]["quad_world"], np.float64).ravel())
        for m in range(M):
            idx = np.flatnonzero(labels[m] == l)
            if not len(idx):
                continue
            pts = np.ascontiguousarray(xyz[m][idx])
            world = np.empty((len(idx), 3), np.float64)
            assert oracle.ssd_oracle_camera_to_world(C.byref(xfs[m]), H.ptr(pts), len(idx), H.ptr(world)) == 0
            xy = np.ascontiguousarray(world[:, :2])
            inside = np.empty(len(idx), np.uint8)
            st = C.c_int()
            assert oracle.ssd_oracle_points_in_quad((C.c_double * 8)(*q), H.ptr(xy), len(idx), H.ptr(inside), C.byref(st)) == 0
            assert st.value == 0, (s, l)
            out[m][idx[inside != 0]] = s
    return out


def oracle_map(oracle, cfg, xf, xyz):
    o = H.oracle_process(oracle, cfg, xf, xyz)
    return o, reference_map(oracle, [xf], xyz, o.labels, o.info, o.plateaus)[0]


def check_invariants(o, m, what=""):
    """count == n_in_quad of the step's plateau, step pixels within that plateau, nothing else labelled"""
    plats = step_plateaus(o.info, o.plateaus)
    for s, l in enumerate(plats):
        sel = m == s
        assert int(sel.sum()) == o.plateaus[l]["n_in_quad"], (what, s, l)
        assert (o.labels[sel] == l).all(), (what, s, l)
    assert ((m == NONE) | (m < len(plats))).all(), what
    return plats


# ---- without a GPU ----
def test_step_label_symbols_are_declared_and_bound(S):
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    assert re.search(r"#define SSD_STEP_LABEL_NONE 255u\b", hdr) and NONE == 255
    assert re.search(r"#define SSD_GPU_ABI_VERSION 3\b", hdr)
    lib = S.lib()
    for name in ("ssd_gpu_set_step_labels", "ssd_gpu_get_step_labels", "ssd_gpu_step_labels_device_ptr"):
        assert re.search(r"\bint " + name + r"\(", hdr), name
        assert name in A.PROTOTYPES, name
        assert getattr(lib, name).restype is C.c_int, name


GOLDEN = sorted(__import__("glob").glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_reference_map_counts_on_the_golden_scenes(S, oracle, path):
    import test_oracle_golden as G
    z, meta, sc, xf = G.load_case(path)
    cfg = S.default_config(meta["width"], meta["height"])
    o, m = oracle_map(oracle, cfg, xf, H.deproject_np(sc, z["depth"]))
    plats = check_invariants(o, m, path)
    for l in plats:
        assert o.plateaus[l]["n_in_quad"] == meta["plateaus"][l]["n_in_quad"], l  # the compiled reference's count
    if meta["info"]["n_steps"] == 0:
        assert (m == NONE).all()


@pytest.mark.parametrize("key", ["frames_random_scenes/320x240", "frames_random_scenes/640x480", "frames_random_scenes/1024x768",
                                 "frames_hires/2560x1920", "frames_hires/4096x3072"])
def test_reference_map_counts_on_the_reference_runs(S, oracle, key):
    import test_oracle_vs_ref as R
    kind, size = key.split("/")
    w, h = (int(v) for v in size.split("x"))
    if kind == "frames_hires":
        _, _, ck, sk, n = next(c for c in R.HIRES_CASES if c[:2] == (w, h))
        inputs = R.frames_hires_inputs(S, w, h, ck, sk, n)
    else:
        inputs = R.frames_random_scenes_inputs(S, w, h, {320: 10, 640: 6, 1024: 3}[w])
    want = R.stored(key)
    n_steps = 0
    for i, (cfg, xf, xyz) in enumerate(inputs):
        o, m = oracle_map(oracle, cfg, xf, xyz)
        plats = check_invariants(o, m, (key, i))
        for l in plats:
            assert o.plateaus[l]["n_in_quad"] == want[i]["plateaus"][l]["n_in_quad"], (key, i, l)
        n_steps += len(plats)
    assert n_steps > 0


# ---- on the GPU ----
def assert_maps(det, want, what, f0=0):
    for f, m in enumerate(want):
        got = det.step_labels(f0 + f)
        bad = np.flatnonzero(got != m)
        assert not len(bad), (what, f, len(bad), bad[:8], got[bad[:8]], m[bad[:8]])


def scenes_of(S, w, h, seed, n, **kw):
    base = S.default_scene(w, h, **dict(NOISY, **kw))
    return base, [S.randomize_scene(base, seed, i, 3, 8) for i in range(n)]


@gpu
@pytest.mark.parametrize("w,h", [(320, 240), (640, 480), (1024, 768)])
def test_random_scenes_fused_and_seven_launch(S, oracle, w, h):
    """vertex and z16 input (host and device), fused calls (<= 16 frames) and seven-launch calls (stage timing, and a batch of
    more than 16 frames), upright and rotated / occluded scenes"""
    cfg = S.default_config(w, h)
    for kw, seed, n in ((dict(), 11, 4), (dict(rotate180=1, n_occluders=2), 12, 18)):
        base, sc = scenes_of(S, w, h, seed, n, **kw)
        xf = S.scene_transform(base)
        depth = np.stack([S.synth_depth_host(s) for s in sc])
        xyz = np.stack([S.deproject_host(s, d) for s, d in zip(sc, depth)])
        want = [oracle_map(oracle, cfg, xf, x)[1] for x in xyz]
        assert sum(int((m != NONE).any()) for m in want) >= n // 2
        intr = S.scene_intrinsics(base)
        with S.Detector(cfg, xf, max_frames=n) as det:
            det.set_step_labels(True)
            det.process_host(xyz[:1])
            assert det.timing().n_launches == 5
            assert_maps(det, want[:1], "vertices/host one frame (fused)")
            det.process_host(xyz)
            assert_maps(det, want, ("vertices/host", n))
            d = H.to_device(det, xyz)
            det.process_device(d, n, A.FLAG_STAGE_TIMING)
            assert det.timing().n_launches == 7 * det.stage_times()["transform_bin"][1]
            assert_maps(det, want, "vertices/device seven-launch")
            det.free(d)
            det.process_depth_host(depth, intr)
            assert_maps(det, want, "z16/host")
            d = H.to_device(det, depth)
            det.process_depth_device(d, intr, n)
            assert_maps(det, want, "z16/device")
            det.free(d)


@gpu
def test_hires_frame(S, oracle):
    """one 4096x3072 frame: pixel indices of the write sites up to 12.6 M"""
    import test_oracle_vs_ref as R
    _, _, ck, sk, _ = next(c for c in R.HIRES_CASES if c[:2] == (4096, 3072))
    cfg, xf, xyz = next(R.frames_hires_inputs(S, 4096, 3072, ck, sk, 1))
    o, want = oracle_map(oracle, cfg, xf, xyz)
    assert (want != NONE).sum() > 0
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.set_step_labels(True)
        det.process_host(xyz[None])
        assert_maps(det, [want], "4096x3072 fused")
        d = H.to_device(det, np.ascontiguousarray(xyz[None]))
        det.process_device(d, 1, A.FLAG_STAGE_TIMING)
        assert_maps(det, [want], "4096x3072 seven-launch")
        det.free(d)


@gpu
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_brown_conrady_lenses(S, oracle, name):
    import test_gpu_distortion as D
    w, h = 640, 480
    cfg = S.default_config(w, h)
    base, depth, xyz = D.lens_frames(S, w, h, D.LENSES[name], 5, 61)
    xf = S.scene_transform(base)
    want = [oracle_map(oracle, cfg, xf, x)[1] for x in xyz]
    with S.Detector(cfg, xf, max_frames=5) as det:
        det.set_distortion(S.scene_distortion(base))
        det.set_step_labels(True)
        det.process_depth_host(depth, S.scene_intrinsics(base))
        assert_maps(det, want, (name, "z16/host"))
        d = H.to_device(det, depth)
        det.process_depth_device(d, S.scene_intrinsics(base), 5)
        assert_maps(det, want, (name, "z16/device"))
        det.free(d)


@gpu
def test_camera_table_with_mixed_lenses(S, oracle):
    import test_gpu_distortion as D
    import test_gpu_groups as G
    w, h = 640, 480
    cfg = S.default_config(w, h)
    bases = [G.camera_scenes(S, w, h)[0], D.lens_scene(S, w, h, D.BC, **NOISY), D.lens_scene(S, w, h, D.IBC, rotate180=1, **NOISY)]
    cams = [S.scene_camera(b) for b in bases]
    idx = np.array([0, 1, 2, 2, 1, 0], np.int32)
    depth, xyz = G.frames_of(S, bases, idx, 47)
    want = [oracle_map(oracle, cfg, cams[c].xf, xyz[f])[1] for f, c in enumerate(idx)]
    with S.Detector(cfg, cams[0].xf, max_frames=len(idx)) as det:
        det.set_cameras(cams, [S.scene_distortion(b) for b in bases])
        det.set_step_labels(True)
        det.process_depth_cameras_host(depth, idx)
        assert_maps(det, want, "camera table z16")
        det.process_cameras_host(xyz, idx)
        assert_maps(det, want, "camera table vertices")


@gpu
def test_groups_of_1_3_and_8(S):
    """each member's map indexes its group's steps, its pixels tested through its own camera"""
    import test_gpu_groups as G
    w, h = 320, 240
    cfg = S.default_config(w, h)
    bases = G.camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    sizes = [1, 3, 8]
    idx = np.random.default_rng(9).integers(0, 3, sum(sizes)).astype(np.int32)
    depth, xyz = G.frames_of(S, bases, idx, 31)
    orc = G.group_oracle()
    for fn in ("ssd_oracle_camera_to_world", "ssd_oracle_points_in_quad"):
        getattr(orc, fn).argtypes = getattr(H.load_oracle(), fn).argtypes
    want = []
    for s, k in zip(G.starts(sizes), sizes):
        xfs = [cams[c].xf for c in idx[s:s + k]]
        g = G.oracle_group(cfg, xfs, xyz[s:s + k])
        want += list(reference_map(orc, xfs, xyz[s:s + k], g.rec.labels, g.rec.info, g.rec.plateaus))
    assert sum(int((m != NONE).any()) for m in want) >= len(want) // 2
    with S.Detector(cfg, cams[0].xf, max_frames=len(idx)) as det:
        det.set_cameras(cams)
        det.set_step_labels(True)
        det.process_groups_host(xyz, idx, sizes)
        assert_maps(det, want, "groups vertices/host")
        d = H.to_device(det, depth)
        det.process_depth_groups_device(d, idx, sizes)
        assert_maps(det, want, "groups z16/device")
        det.free(d)


@gpu
def test_quadrilateral_threshold_constructions(S, oracle):
    """tests/threshold_frames.py quad_edges: points inside the f32 bound of every step's quadrilateral, so the exact pass and the
    filtered test decide many of them"""
    import test_gpu_thresholds as T
    for name in ("scene", "sheared", "singular"):
        cfg, xf, f, pts, B = T.cached(S, oracle, name, "quad")
        o, want = oracle_map(oracle, cfg, xf, f)
        with S.Detector(cfg, xf, max_frames=1) as det:
            det.set_step_labels(True)
            det.process_host(f[None])
            assert det.stats().n_quad_exact > 0, name
            assert_maps(det, [want], (name, "fused"))
            d = H.to_device(det, np.ascontiguousarray(f[None]))
            det.process_device(d, 1, A.FLAG_STAGE_TIMING)
            assert det.stats().n_quad_exact > 0, name
            assert_maps(det, [want], (name, "seven-launch"))
            det.free(d)


def _edge_map(S, oracle, cfg, xf, xyz, bit):
    o, want = oracle_map(oracle, cfg, xf, xyz)
    assert o.info["status"] & bit, hex(o.info["status"])
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.set_step_labels(True)
        det.process_host(xyz[None])
        assert_maps(det, [want], ("fused", bit))
        d = H.to_device(det, np.ascontiguousarray(xyz[None]))
        det.process_device(d, 1, A.FLAG_STAGE_TIMING)
        assert_maps(det, [want], ("seven-launch", bit))
        det.free(d)
    return o, want


def unseen_front_edge_frame(E):
    """SSD_STATUS_INVALID_FRONT_EDGE with ground points inside the ground quadrilateral: the ground lies between y_min and the
    step's front edge, but only in two strips of BEV columns that Segmentation::detectFrontEdge does not probe (BottomScanner looks
    at columns W/2 + 50 j, two columns either side after the close; at 320 px over 1.2 m those are x = -0.6 + (160 + 50 j) / 266.7).
    calcGround finds no front edge and emits the all-zero step, and getPointsInQuadrilateral still returns the ground's points."""
    rng = np.random.default_rng(21)
    return E.frame_of([E.slab(rng, 6000, -0.15, -0.05, 0.15, 0.40, 0.004), E.slab(rng, 6000, 0.05, 0.15, 0.15, 0.40, 0.004),
                       E.slab(rng, 30000, -0.45, 0.45, 0.45, 0.75, 0.185)])


def test_unseen_front_edge_frame_has_ground_pixels(S, oracle):
    """the construction (no GPU): the status bit is set, the ground step is the all-zero one, and its pixels are present"""
    import test_gpu_edge_cases as E
    cfg = S.default_config(E.W, E.HH)
    o, m = oracle_map(oracle, cfg, E.shifted(E.identity_xf()), unseen_front_edge_frame(E))
    assert o.info["status"] == A.STATUS_INVALID_FRONT_EDGE, hex(o.info["status"])
    assert o.info["n_steps"] == 2 and not o.steps[0]["quad"].any() and o.steps[0]["height"] == 0.0
    check_invariants(o, m)
    assert int((m == 0).sum()) == o.plateaus[o.info["ground_index"]]["n_in_quad"] > 0


@gpu
def test_edge_statuses(S, oracle):
    """Directed frames, each with its status bit asserted set. Two statuses are not among them: no frame that reaches
    SSD_STATUS_DEGENERATE_QUAD or SSD_STATUS_EMPTY_MEAN through the chain is known (DESIGN.md section 6, Step labels). A ground
    step with an empty mean cannot occur: its front edge is found in the BEV image of the very points that are counted, so no
    counted point means an invalid front edge instead. A plateau's quadrilateral is fitted to its own BEV image, and the outlines
    found have vertical sides, which QuadrilateralTest accepts; the random scenes the tests build are not known to raise either
    bit. So these two statuses have no directed frame; the quad_amask rule that would leave such a plateau without pixels is
    the one every other frame exercises."""
    import test_gpu_edge_cases as E
    cfg = S.default_config(E.W, E.HH)
    xf = E.shifted(E.identity_xf())
    # invalid ground front edge with ground points in the quadrilateral: step 0 is all zero, its pixels are marked
    o, m = _edge_map(S, oracle, cfg, xf, unseen_front_edge_frame(E), A.STATUS_INVALID_FRONT_EDGE)
    assert int((m == 0).sum()) == o.plateaus[o.info["ground_index"]]["n_in_quad"] > 0
    assert int((m == 1).sum()) == o.plateaus[o.info["first_valid_index"]]["n_in_quad"] > 0
    # ... and the frame of test_gpu_edge_cases, whose ground lies only behind the step: no ground point in the quadrilateral
    rng = np.random.default_rng(13)
    xyz = E.frame_of([E.slab(rng, 9000, -0.45, 0.45, 1.0, 1.25, 0.004), E.slab(rng, 30000, -0.45, 0.45, 0.45, 0.75, 0.185)])
    o, m = _edge_map(S, oracle, cfg, xf, xyz, A.STATUS_INVALID_FRONT_EDGE)
    assert o.plateaus[o.info["ground_index"]]["n_in_quad"] == 0 and not (m == 0).any()
    assert int((m == 1).sum()) == o.plateaus[o.info["first_valid_index"]]["n_in_quad"] > 0
    # HMIN_WRAP: every plateau empty, no step pixels
    rng = np.random.default_rng(11)
    xyz = E.frame_of([E.slab(rng, 1500, -0.4, 0.4, 0.2, 0.6, -0.095), E.slab(rng, 4000, -0.4, 0.4, 0.2, 0.6, -0.085),
                      E.slab(rng, 6000, -0.4, 0.4, 0.7, 1.1, 0.305)])
    o, m = _edge_map(S, oracle, cfg, xf, xyz, A.STATUS_HMIN_WRAP)
    assert (m == NONE).all()
    # no steps: an empty frame and a flat floor
    for xyz in (np.zeros((E.N, 3), np.float32), E.frame_of([E.slab(rng, 20000, -0.45, 0.45, 0.2, 1.2, 0.004)])):
        o, m = _edge_map(S, oracle, cfg, xf, xyz, A.STATUS_NO_STEPS)
        assert (m == NONE).all()


@gpu
def test_invariants_at_scale(S, oracle):
    """Scale: 600 device-generated 1024x768 frames over several chunks and streams. In every frame the count and subset
    invariants hold against the GPU's own plateaus, and spot frames equal the reference map."""
    W, Hh = 1024, 768
    N = W * Hh
    cfg = S.default_config(W, Hh)
    base = S.default_scene(W, Hh, **NOISY)
    xf = S.scene_transform(base)
    nF = 600
    with S.Detector(cfg, xf, max_frames=nF) as det:
        d_xyz = det.malloc(nF * N * 12)
        det.synth_frames(base, 4242, 0, nF, 3, 8, d_xyz)
        det.set_step_labels(True)
        det.process_device(d_xyz, nF)
        allm = np.empty(nF * N, np.uint8)
        det.d2h(allm, C.c_void_p(det.step_labels_device_ptr()), nF * N)
        n_steps = 0
        for f in range(nF):
            m = allm[f * N:(f + 1) * N]
            info = det.frame_info(f)
            plats, K = det.plateaus(f)
            pl = [dict(valid=p.valid, quad_status=p.quad_status, n_in_quad=p.n_in_quad) for p in plats[:K]]
            I = {k: getattr(info, k) for k, _ in A.FrameInfo._fields_}
            o = H.FrameResult(det.labels(f), None, I, pl, None)
            sp = check_invariants(o, m, f)
            assert len(sp) == info.n_steps, f
            n_steps += len(sp)
            if f in (0, 299, 599):
                assert np.array_equal(det.step_labels(f), m)
                xyz = np.empty((N, 3), np.float32)
                det.d2h(xyz, C.c_void_p(d_xyz.value + f * N * 12))
                assert np.array_equal(oracle_map(oracle, cfg, xf, xyz)[1], m), f
        assert n_steps > 3 * nF
        det.free(d_xyz)


def _everything(S, det, n):
    out = []
    for f in range(n):
        r = H.gpu_result(det, f)
        out.append((H.frame_record(r, 0xffffffff), r.line, H.digest(r.labels), det.overlay(f).tobytes(), det.vertical_faces(f)))
    return out


@gpu
def test_nothing_else_changes(S):
    """the same input with the option on and off: steps, plateaus, frame info, labels, histogram, overlay and risers
    byte-identical; n_launches unchanged"""
    w, h = 640, 480
    cfg = S.default_config(w, h)
    base, sc = scenes_of(S, w, h, 71, 20)
    xf = S.scene_transform(base)
    xyz = np.stack([S.deproject_host(s, S.synth_depth_host(s)) for s in sc])
    xfe = S.scene_transform_ex(base)
    with S.Detector(cfg, xf, max_frames=20) as det:
        det.set_overlay(xfe[1], S.scene_intrinsics(base))
        det.set_vertical_faces(True)
        res = {}
        for on in (False, True, False):
            det.set_step_labels(on)
            for n in (1, 20):
                det.process_host(xyz[:n])
                res.setdefault((on, n), []).append((_everything(S, det, n), det.timing().n_launches))
        for n in (1, 20):
            off, on = res[(False, n)][0], res[(True, n)][0]
            assert off == res[(False, n)][1]
            assert on[0] == off[0], n
            assert on[1] == off[1], n


@gpu
def test_getter_errors(S):
    w, h = 320, 240
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h)
    xf = S.scene_transform(base)
    xyz = S.deproject_host(base, S.synth_depth_host(base))[None]
    with S.Detector(cfg, xf, max_frames=2) as det:
        def rc(fn, *a):
            return getattr(det._l, fn)(det._h, *a)
        out = np.empty(w * h, np.uint8)
        p = C.c_void_p()
        det.process_host(xyz)
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.E_STATE  # not enabled
        assert rc("ssd_gpu_step_labels_device_ptr", C.byref(p)) == A.E_STATE
        det.set_step_labels(True)
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.E_STATE  # the last call ran without it
        det.process_host(xyz)
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.OK and (out != NONE).any()
        assert rc("ssd_gpu_step_labels_device_ptr", C.byref(p)) == A.OK and p.value
        assert rc("ssd_gpu_get_step_labels", 1, H.ptr(out)) == A.E_RANGE  # frame outside the last call
        assert rc("ssd_gpu_get_step_labels", -1, H.ptr(out)) == A.E_RANGE
        kept = out.copy()
        # a rejected call leaves the step labels readable
        assert det._l.ssd_gpu_process_host(det._h, H.ptr(np.ascontiguousarray(np.repeat(xyz, 3, 0))), 3) == A.E_RANGE
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.OK and np.array_equal(out, kept)
        # a call that invalidates the last call's results (a single-stage entry point reuses the per-frame records; a failed call
        # does the same) takes the step labels with them, the device pointer included
        det.detect_front_edge(np.zeros((h, w), np.uint8))
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.E_STATE
        assert rc("ssd_gpu_step_labels_device_ptr", C.byref(p)) == A.E_STATE
        det.process_host(xyz)
        assert rc("ssd_gpu_step_labels_device_ptr", C.byref(p)) == A.OK
        det.set_step_labels(True)  # enabling again keeps the map of the last call
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.OK and np.array_equal(out, kept)
        det.set_step_labels(False)  # disabled after a call
        assert rc("ssd_gpu_get_step_labels", 0, H.ptr(out)) == A.E_STATE
        assert rc("ssd_gpu_step_labels_device_ptr", C.byref(p)) == A.E_STATE
        with pytest.raises(S.SsdError):
            det.step_labels(0)


@gpu
def test_cpp_step_labels(S, tmp_path):
    """tests/native/step_labels_check.cpp: Pointcloud::enableStepLabels / stepLabels on one frame; the map equals the C ABI's"""
    exe = str(tmp_path / "step_labels_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "step_labels_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h = 640, 480
    mp = tmp_path / "map.u8"
    out = subprocess.run([exe, str(w), str(h), str(mp)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    got = np.fromfile(str(mp), np.uint8)
    base = S.default_scene(w, h, noise_sigma=0.0025)
    depth = S.synth_depth_host(base)
    with S.Detector(S.default_config(w, h), S.scene_transform(base), max_frames=1) as det:
        det.set_step_labels(True)
        det.process_depth_host(depth[None], S.scene_intrinsics(base))
        want = det.step_labels(0)
        assert out[0] == det.line(0)
    assert np.array_equal(got, want)
    assert len(set(np.unique(got)) - {NONE}) >= 3
