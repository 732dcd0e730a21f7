"""Frame groups (ssd_gpu_process_groups_* / ssd_gpu_process_depth_groups_*, include/ssd_gpu.h): one stair detection from the union
of the world points of several frames, each member through its own camera. The reference for the union is the group restatement of
the oracle (tests/native/oracle_group.c, which compiles oracle/ssd_oracle.c into the same translation unit): a group of one frame is
ssd_oracle_process bit for bit, and a group of one frame on the GPU is the camera call bit for bit."""
import atexit
import ctypes as C
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

gpu = pytest.mark.gpu
TOL = 1e-4       # metres, as tests/test_gpu_parity.py
OVL_TOL = 2e-3   # pixels, as tests/test_gpu_distortion.py
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
_vp, _P = C.c_void_p, C.POINTER


# ---- the group oracle ----
_ORACLE = {}


def group_oracle():
    """tests/native/oracle_group.c compiled with oracle/Makefile's flags into a temporary directory"""
    if "lib" not in _ORACLE:
        tmp = tempfile.mkdtemp(prefix="ssd_oracle_group_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libssd_oracle_group.so")
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                        os.path.join(H.ROOT, "tests", "native", "oracle_group.c"), "-lm"], check=True)
        lib = C.CDLL(out)
        lib.ssd_oracle_process.argtypes = [_P(A.Config), _P(A.Transform), _vp, _vp, _vp, C.c_int, _P(A.FrameInfo), _P(A.Plateau), _P(A.Step)]
        lib.ssd_oracle_process_group.argtypes = [_P(A.Config), _P(A.Transform), _vp, C.c_int, _vp, _vp, C.c_int, _P(A.FrameInfo),
                                                 _P(A.Plateau), _P(A.Step)]
        lib.ssd_oracle_vertical_faces_group.argtypes = [_P(A.Config), _P(A.Transform), _vp, C.c_int, _vp, _P(A.Plateau), C.c_int,
                                                        _P(A.Riser), C.c_int, _P(C.c_int)]
        lib.ssd_oracle_last_overlay.argtypes = [_P(A.Transform), _P(C.c_double), _P(A.Intrinsics), _P(A.Overlay), C.c_int, _P(C.c_int)]
        _ORACLE["lib"] = lib
    return _ORACLE["lib"]


class Group:
    """the oracle's result of one group: rec (FrameResult of the group, labels (n_members, N)), risers, overlay(m) per member"""

    def __init__(self, cfg, xfs, xyz, cams=None, lenses=None):
        lib = group_oracle()
        self.xf0 = xfs[0]
        M, N = len(xfs), cfg.width * cfg.height
        xyz = np.ascontiguousarray(xyz, np.float32).reshape(M, N, 3)
        arr = (A.Transform * M)(*xfs)
        labels = np.empty((M, N), np.uint8)
        hist = np.zeros(A.MAX_BINS, np.uint32)
        info, plats, steps = A.FrameInfo(), (A.Plateau * A.MAX_PLATEAUS)(), (A.Step * A.MAX_STEPS)()
        assert lib.ssd_oracle_process_group(C.byref(cfg), arr, H.ptr(xyz), M, H.ptr(labels), H.ptr(hist), A.MAX_BINS, C.byref(info), plats,
                                            steps) == 0
        self.rec = H._collect(labels, hist, info, plats, steps)
        out, n = (A.Riser * A.MAX_PLATEAUS)(), C.c_int()
        assert lib.ssd_oracle_vertical_faces_group(C.byref(cfg), arr, H.ptr(xyz), M, H.ptr(labels), plats, info.n_plateaus, out,
                                                   A.MAX_PLATEAUS, C.byref(n)) == 0
        self.risers = [{f: getattr(r, f) for f, _ in A.Riser._fields_ if f != "pad"} for r in out[:n.value]]
        self.overlays = []
        for m in range(M if cams is not None else 0):
            if lenses is not None and lenses[m] is not None:
                import test_gpu_distortion as D
                self.overlays.append(self._lens_overlay(cams[m], lenses[m], D))
                continue
            o, k = (A.Overlay * A.MAX_STEPS)(), C.c_int()
            assert lib.ssd_oracle_last_overlay(C.byref(cams[m].xf), cams[m].a_inv, C.byref(cams[m].intr), o, A.MAX_STEPS, C.byref(k)) == 0
            self.overlays.append(np.array([[[q.px[c][0], q.px[c][1]] for c in range(4)] for q in o[:k.value]], np.float32).reshape(-1, 4, 2))

    def _lens_overlay(self, cam, lens, D):
        """the group's steps (before ToExternalWorld of the first member) through a member's lens, as test_gpu_distortion restates it"""
        xf0 = self.xf0
        ea, eb = np.array(xf0.ext_a[:]).reshape(2, 2), np.array(xf0.ext_b[:])
        a, b = np.array(cam.a_inv[:]).reshape(3, 3), np.array(cam.xf.b[:])
        out = np.zeros((len(self.rec.steps), 4, 2), np.float32)
        for s, st in enumerate(self.rec.steps):
            z = st["height"] - xf0.ext_z
            for c in range(4):
                x, y = np.linalg.solve(ea, st["quad"][c] - eb)
                d = (x - b[0], y - b[1], z - b[2])
                X, Y, Z = (np.float32((a[r, 0] * d[0] + a[r, 1] * d[1]) + a[r, 2] * d[2]) for r in range(3))
                with np.errstate(all="ignore"):
                    out[s, c] = D.np_project(lens, X, Y, Z, cam.intr)
        return out


oracle_group = Group


def camera_scenes(S, w, h):
    from test_gpu_cameras import camera_scenes as cs
    return cs(S, w, h)


def frames_of(S, bases, cam_index, seed, lens_of=None):
    """one randomized frame per entry of cam_index, of that camera's mounting: depth (n, N), xyz (n, N, 3)"""
    depth, xyz = [], []
    for i, c in enumerate(cam_index):
        sc = S.randomize_scene(bases[c], seed, i, 3, 8)
        sc.rotate180, sc.n_occluders = bases[c].rotate180, bases[c].n_occluders
        sc.distortion_model = bases[c].distortion_model
        for k in range(5):
            sc.coeffs[k] = bases[c].coeffs[k]
        d = S.synth_depth_host(sc)
        depth.append(d)
        xyz.append(S.deproject_host(sc, d))
    return np.stack(depth), np.stack(xyz)


def starts(sizes):
    return np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(int)


# ---- declaration and binding (no GPU) ----
def test_group_entry_points_are_declared_and_bound(S):
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    assert re.search(r"#define SSD_GPU_MAX_GROUP_FRAMES 32\b", hdr) and A.MAX_GROUP_FRAMES == 32
    assert re.search(r"#define SSD_GPU_ABI_VERSION 3\b", hdr)
    for name, nargs in (("ssd_gpu_process_groups_host", 5), ("ssd_gpu_process_groups_device", 6), ("ssd_gpu_process_depth_groups_host", 5),
                        ("ssd_gpu_process_depth_groups_device", 6)):
        assert re.search(r"\b%s\(" % name, hdr) and name in A.PROTOTYPES, name
        assert len(A.PROTOTYPES[name][1]) == nargs and A.PROTOTYPES[name][1][-1] == C.c_int, name
        assert getattr(S.lib(), name).argtypes == A.PROTOTYPES[name][1]


# ---- the group oracle (no GPU) ----
def _oracle_one(lib, cfg, xf, xyz):
    N = cfg.width * cfg.height
    labels, hist = np.empty(N, np.uint8), np.zeros(A.MAX_BINS, np.uint32)
    info, plats, steps = A.FrameInfo(), (A.Plateau * A.MAX_PLATEAUS)(), (A.Step * A.MAX_STEPS)()
    xyz = np.ascontiguousarray(xyz, np.float32)
    assert lib.ssd_oracle_process(C.byref(cfg), C.byref(xf), H.ptr(xyz), H.ptr(labels), H.ptr(hist), A.MAX_BINS, C.byref(info), plats, steps) == 0
    return labels, hist, bytes(info), bytes(plats), bytes(steps)


def _group_one(cfg, xf, xyz):
    lib = group_oracle()
    N = cfg.width * cfg.height
    labels, hist = np.empty(N, np.uint8), np.zeros(A.MAX_BINS, np.uint32)
    info, plats, steps = A.FrameInfo(), (A.Plateau * A.MAX_PLATEAUS)(), (A.Step * A.MAX_STEPS)()
    xyz = np.ascontiguousarray(xyz, np.float32)
    assert lib.ssd_oracle_process_group(C.byref(cfg), (A.Transform * 1)(xf), H.ptr(xyz), 1, H.ptr(labels), H.ptr(hist), A.MAX_BINS,
                                        C.byref(info), plats, steps) == 0
    return labels, hist, bytes(info), bytes(plats), bytes(steps)


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def test_oracle_group_of_one_is_the_oracle(S, oracle):
    w, h = 640, 480
    cfg = S.default_config(w, h)
    for sc in camera_scenes(S, w, h):
        xf = S.scene_transform(sc)
        xyz = S.deproject_host(sc, S.synth_depth_host(sc))
        assert _same(_group_one(cfg, xf, xyz), _oracle_one(oracle, cfg, xf, xyz))
    import test_oracle_vs_ref as R
    for cfg, xf, xyz in R.frames_random_scenes_inputs(S, 320, 240, 4):
        assert _same(_group_one(cfg, xf, xyz), _oracle_one(oracle, cfg, xf, xyz))


def test_oracle_group_histogram_and_label_classes(S, oracle):
    """the group histogram is the sum of the members' histograms; every member pixel keeps its single-frame class
    (invalid, out of range, in range)"""
    w, h = 320, 240
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    idx = [0, 1, 2, 0, 2]
    _, xyz = frames_of(S, bases, idx, 91)
    g = oracle_group(cfg, [cams[c].xf for c in idx], xyz)
    singles = [_oracle_one(oracle, cfg, cams[c].xf, xyz[m]) for m, c in enumerate(idx)]
    assert np.array_equal(g.rec.hist, np.sum([s[1][:g.rec.info["n_bins"]] for s in singles], axis=0))
    cls = lambda l: np.where(l >= A.LABEL_OUT_OF_RANGE, l, 0)
    for m, s in enumerate(singles):
        assert np.array_equal(cls(g.rec.labels[m]), cls(s[0])), m
    assert g.rec.info["n_nonzero"] == sum(int((s[0] != A.LABEL_INVALID).sum()) for s in singles)


# ---- 1. groups of one frame equal the camera call ----
def _everything(S, det, n):
    return [(H.exact(H.gpu_result(det, f)), det.overlay(f).tobytes(), det.vertical_faces(f)) for f in range(n)]


def _stats(det):
    st = det.stats()
    return tuple(getattr(st, k) for k in ("n_points", "n_exact_fallback", "n_quad_fast", "n_quad_exact", "n_bev_exact", "filter_eps0", "filter_eps1"))


@gpu
@pytest.mark.parametrize("size", [(640, 480), (1024, 768)])
def test_groups_of_one_equal_the_camera_call(S, size):
    import test_gpu_distortion as D
    w, h = size
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    lensed = [D.lens_scene(S, w, h, D.BC, **NOISY), D.lens_scene(S, w, h, D.IBC, rotate180=1, **NOISY)]
    for table in ("pinhole", "lens"):
        bb = bases if table == "pinhole" else [bases[0]] + lensed
        cams = [S.scene_camera(b) for b in bb]
        dist = [S.scene_distortion(b) for b in bb]
        idx = np.array([0, 1, 2, 1, 0, 2, 2], np.int32)
        n = len(idx)
        depth, xyz = frames_of(S, bb, idx, 17 + w)
        ones = np.ones(n, np.int32)
        with S.Detector(cfg, cams[0].xf, max_frames=n) as det:
            det.set_cameras(cams, dist)
            det.set_overlay(np.array(cams[0].a_inv[:]), cams[0].intr)
            det.set_vertical_faces(True)
            d_xyz, d_z16 = H.to_device(det, xyz), H.to_device(det, depth)
            calls = [("vertices/host", lambda: det.process_cameras_host(xyz, idx), lambda: det.process_groups_host(xyz, idx, ones)),
                     ("vertices/device", lambda: det.process_cameras_device(d_xyz, idx, n), lambda: det.process_groups_device(d_xyz, idx, ones)),
                     ("vertices/device/timing", lambda: det.process_cameras_device(d_xyz, idx, n, A.FLAG_STAGE_TIMING),
                      lambda: det.process_groups_device(d_xyz, idx, ones, A.FLAG_STAGE_TIMING)),
                     ("z16/host", lambda: det.process_depth_cameras_host(depth, idx), lambda: det.process_depth_groups_host(depth, idx, ones)),
                     ("z16/device", lambda: det.process_depth_cameras_device(d_z16, idx, n),
                      lambda: det.process_depth_groups_device(d_z16, idx, ones)),
                     ("z16/device/timing", lambda: det.process_depth_cameras_device(d_z16, idx, n),
                      lambda: det.process_depth_groups_device(d_z16, idx, ones, A.FLAG_STAGE_TIMING))]
            for kind, cam_call, group_call in calls:
                cam_call()
                want, want_stats = _everything(S, det, n), _stats(det)
                group_call()
                assert _everything(S, det, n) == want, (table, kind)
                assert _stats(det) == want_stats, (table, kind)
            det.free(d_xyz)
            det.free(d_z16)


# ---- 2. mixed groups against the oracle group ----
def _check_group(S, det, cfg, f0, g, tag, risers=False):
    for m in range(len(g.rec.labels)):
        r = H.gpu_result(det, f0 + m)
        assert np.array_equal(r.labels, g.rec.labels[m]), (tag, m)
        bad = H.compare_results(g.rec, r, tol=TOL, check_labels=False)
        assert not bad, (tag, m, bad)
        assert r.info["status"] == g.rec.info["status"], (tag, m)
        if g.overlays:
            got, want = det.overlay(f0 + m), g.overlays[m]
            assert got.shape == want.shape and (got.size == 0 or np.abs(got - want).max() < OVL_TOL), (tag, m)
        if risers:
            assert det.vertical_faces(f0 + m) == g.risers, (tag, m)


@gpu
def test_mixed_groups_equal_the_oracle(S):
    w, h = 320, 240
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    sizes = [1, 2, 3, 5, 8, 32, 4, 3]
    rng = np.random.default_rng(5)
    idx = rng.integers(0, 3, sum(sizes)).astype(np.int32)
    # the last two groups: one camera's noisy frames of one scene with different seeds (a static camera accumulating frames)
    tail = sizes[-1] + sizes[-2]
    idx[-tail:] = 1
    depth, xyz = frames_of(S, bases, idx, 29)
    for m in range(sum(sizes) - tail, sum(sizes)):
        sc = S.default_scene(w, h, **dict(NOISY, seed=1000 + m))
        base = bases[1]
        for k in ("cam_height", "cam_pitch_deg", "cam_roll_deg", "cam_yaw_deg", "fx", "fy", "ppx", "ppy", "n_occluders"):
            setattr(sc, k, getattr(base, k))
        depth[m] = S.synth_depth_host(sc)
        xyz[m] = S.deproject_host(sc, depth[m])
    n = len(idx)
    want = [oracle_group(cfg, [cams[c].xf for c in idx[s:s + k]], xyz[s:s + k], [cams[c] for c in idx[s:s + k]])
            for s, k in zip(starts(sizes), sizes)]
    with S.Detector(cfg, cams[2].xf, max_frames=n) as det:
        det.set_cameras(cams)
        det.set_overlay(np.array(cams[0].a_inv[:]), cams[0].intr)
        det.set_vertical_faces(True)
        d_z16 = H.to_device(det, depth)
        for kind in ("vertices/host", "z16/device"):
            if kind == "vertices/host":
                det.process_groups_host(xyz, idx, sizes)
            else:
                det.process_depth_groups_device(d_z16, idx, sizes)
            for s, k, g in zip(starts(sizes), sizes, want):
                _check_group(S, det, cfg, s, g, (kind, k), risers=True)
        det.free(d_z16)
    assert sum(len(g.rec.steps) for g in want) >= 2 * len(sizes)


@gpu
def test_mixed_lens_groups_equal_the_oracle(S):
    import test_gpu_distortion as D
    w, h = 640, 480
    cfg = S.default_config(w, h)
    bases = [camera_scenes(S, w, h)[0], D.lens_scene(S, w, h, D.BC, **NOISY), D.lens_scene(S, w, h, D.IBC, rotate180=1, **NOISY)]
    cams = [S.scene_camera(b) for b in bases]
    lens = [None, D.BC, D.IBC]
    sizes = [3, 1, 2]
    idx = np.array([0, 1, 2, 2, 1, 0], np.int32)
    depth, xyz = frames_of(S, bases, idx, 43)
    want = [oracle_group(cfg, [cams[c].xf for c in idx[s:s + k]], xyz[s:s + k], [cams[c] for c in idx[s:s + k]],
                         [lens[c] for c in idx[s:s + k]]) for s, k in zip(starts(sizes), sizes)]
    with S.Detector(cfg, cams[0].xf, max_frames=len(idx)) as det:
        det.set_cameras(cams, [S.scene_distortion(b) for b in bases])
        det.set_overlay(np.array(cams[0].a_inv[:]), cams[0].intr)
        det.process_depth_groups_host(depth, idx, sizes)
        for s, k, g in zip(starts(sizes), sizes, want):
            _check_group(S, det, cfg, s, g, k)


# ---- 3. chunking does not matter ----
@gpu
def test_chunking_does_not_matter(S, monkeypatch):
    w, h = 320, 240
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    rng = np.random.default_rng(3)
    sizes = [int(v) for v in rng.choice([1, 2, 3, 5, 7, 11, 32], 40)]
    n = sum(sizes)
    idx = rng.integers(0, 3, n).astype(np.int32)
    depth, xyz = frames_of(S, bases, idx, 61)
    alone = []
    with S.Detector(cfg, cams[0].xf, max_frames=32) as det:
        det.set_cameras(cams)
        det.set_vertical_faces(True)
        for s, k in zip(starts(sizes), sizes):
            det.process_groups_host(xyz[s:s + k], idx[s:s + k], [k])
            alone.append([(H.exact(H.gpu_result(det, m)), det.vertical_faces(m)) for m in range(k)])
    # chunks of 7 frames (device input) and 5 frames (host input): the old boundaries would split most groups
    monkeypatch.setenv("SSD_GPU_CHUNK_FRAMES", "7")
    monkeypatch.setenv("SSD_GPU_HOST_CHUNK_FRAMES", "5")
    with S.Detector(cfg, cams[1].xf, max_frames=n) as det:
        assert det.chunk_frames == 7
        det.set_cameras(cams)
        det.set_vertical_faces(True)
        d_xyz = H.to_device(det, xyz)
        for run in range(3):
            [lambda: det.process_groups_host(xyz, idx, sizes), lambda: det.process_groups_device(d_xyz, idx, sizes),
             lambda: det.process_groups_device(d_xyz, idx, sizes, A.FLAG_SINGLE_STREAM | A.FLAG_STAGE_TIMING)][run]()
            for g, (s, k) in enumerate(zip(starts(sizes), sizes)):
                got = [(H.exact(H.gpu_result(det, s + m)), det.vertical_faces(s + m)) for m in range(k)]
                assert got == alone[g], (run, g, k)
        det.free(d_xyz)


# ---- 4. the capability: views that each miss a tread detect the whole flight together ----
def occluded_pair(S, oracle, w, h):
    """two frames of one static camera, each with a different tread's points dropped (as an occluder in front of it would)"""
    sc = S.default_scene(w, h, noise_sigma=0.002, dropout=0.0, n_holes=0)
    xf = S.scene_transform(sc)
    depth = S.synth_depth_host(sc)
    o = H.oracle_process(oracle, cfg := S.default_config(w, h), xf, S.deproject_host(sc, depth))
    valid = [k for k, p in enumerate(o.plateaus) if p["valid"]]
    assert len(valid) >= 4
    views = []
    for k in (valid[1], valid[2]):
        d = depth.copy().reshape(-1)
        d[o.labels == k] = 0
        views.append(d.reshape(depth.shape))
    return cfg, sc, np.stack(views)


@gpu
def test_views_missing_different_treads_detect_more_steps_together(S, oracle):
    w, h = 640, 480
    cfg, sc, depth = occluded_pair(S, oracle, w, h)
    cam = S.scene_camera(sc)
    xyz = np.stack([S.deproject_host(sc, d) for d in depth])
    single = [oracle_group(cfg, [cam.xf], xyz[m:m + 1]) for m in range(2)]
    fused = oracle_group(cfg, [cam.xf, cam.xf], xyz)
    n1, n2, nf = (len(g.rec.steps) for g in (single[0], single[1], fused))
    assert nf > max(n1, n2), (n1, n2, nf)
    with S.Detector(cfg, cam.xf, max_frames=2) as det:
        det.set_cameras([cam])
        det.process_depth_groups_host(depth, [0, 0], [1, 1])
        for m in range(2):
            _check_group(S, det, cfg, m, single[m], ("single", m))
        det.process_depth_groups_host(depth, [0, 0], [2])
        _check_group(S, det, cfg, 0, fused, "fused")
        assert len(det.steps(0)[0]) == nf


# ---- 6. errors ----
@gpu
def test_group_call_rejections(S):
    w, h = 320, 240
    cfg = S.default_config(w, h)
    bases = camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    idx = np.array([0, 1, 2, 0], np.int32)
    depth, xyz = frames_of(S, bases, idx, 7)
    L = S.lib()
    ptr = H.ptr
    with S.Detector(cfg, cams[0].xf, max_frames=4) as det:
        h_ = det._h
        sizes = np.array([2, 2], np.int32)
        # no camera table
        assert L.ssd_gpu_process_groups_host(h_, ptr(xyz), ptr(idx), ptr(sizes), 2) == A.E_STATE
        det.set_cameras(cams[:2] + [A.Camera()])  # camera 2 has no depth intrinsics
        det.process_groups_host(xyz, idx, sizes)
        want = [H.exact(H.gpu_result(det, f)) for f in range(4)]
        bad_idx = np.array([0, 1, 3, 0], np.int32)
        big = np.array([2, 3], np.int32)
        cases = [(L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(bad_idx), ptr(sizes), 2), A.E_RANGE),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(np.array([0, 1, 2, 0, 1], np.int32)), ptr(big), 2), A.E_RANGE),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(idx), ptr(sizes), 0), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_host, (None, ptr(idx), ptr(sizes), 2), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), None, ptr(sizes), 2), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(idx), None, 2), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(idx), ptr(np.array([4, 0], np.int32)), 2), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_host, (ptr(xyz), ptr(np.zeros(33, np.int32)), ptr(np.array([33], np.int32)), 1), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_depth_groups_host, (ptr(depth), ptr(idx), ptr(sizes), 2), A.E_INVALID_ARG),
                 (L.ssd_gpu_process_groups_device, (xyz.ctypes.data + 4, ptr(idx), ptr(sizes), 2, 0), A.E_INVALID_ARG)]
        for i, (fn, args, rc) in enumerate(cases):
            assert fn(h_, *args) == rc, i
            assert [H.exact(H.gpu_result(det, f)) for f in range(4)] == want, i
        det.process_groups_host(xyz, idx, sizes)
        assert [H.exact(H.gpu_result(det, f)) for f in range(4)] == want


# ---- 7. high resolution ----
@gpu
def test_group_of_two_4096x3072_depth_frames(S):
    w, h = 4096, 3072
    cfg = S.default_config(w, h, y_max=3.7, z_max=2.3)
    d = S.default_scene(w, h)
    bases = [S.default_scene(w, h, noise_sigma=0.0025, dropout=0.0, n_holes=0),
             S.default_scene(w, h, cam_height=d.cam_height * 1.1, cam_pitch_deg=d.cam_pitch_deg + 4.0, cam_yaw_deg=-3.0, fx=d.fx * 1.05,
                             noise_sigma=0.0025, dropout=0.0, n_holes=0)]
    cams = [S.scene_camera(b) for b in bases]
    depth, xyz = frames_of(S, bases, [0, 1], 3)
    g = oracle_group(cfg, [c.xf for c in cams], xyz)
    with S.Detector(cfg, cams[0].xf, max_frames=2) as det:
        det.set_cameras(cams)
        d_z16 = H.to_device(det, depth)
        det.process_depth_groups_device(d_z16, [0, 1], [2])
        _check_group(S, det, cfg, 0, g, "4096x3072")
        det.free(d_z16)
    assert len(g.rec.steps) >= 3


# ---- the C++ host classes ----
@gpu
def test_cpp_process_groups(S, tmp_path):
    """tests/native/groups_check.cpp: Pointcloud::processGroups prints the lines (and statuses) the Python binding gives for the
    same groups"""
    exe = str(tmp_path / "groups_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "groups_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h = 640, 480
    out = subprocess.run([exe, str(w), str(h)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == 3
    f32 = np.float32
    bases = [S.default_scene(w, h, noise_sigma=0.0025), S.default_scene(w, h, noise_sigma=0.0025)]
    bases[1].cam_pitch_deg = float(f32(bases[1].cam_pitch_deg) + f32(4.0))
    bases[1].fx = float(f32(bases[1].fx) * f32(1.05))
    depth = np.stack([S.synth_depth_host(S.randomize_scene(bases[f % 2], 99, f, 3, 8)) for f in range(4)])
    with S.Detector(S.default_config(w, h), S.scene_transform(bases[0]), max_frames=4) as det:
        det.set_cameras([S.scene_camera(b) for b in bases])
        det.process_depth_groups_host(depth, np.array([0, 1, 0, 1], np.int32), [1, 3])
        lines = [det.line(0), det.line(1)]
        status = [det.steps(0)[1], det.steps(1)[1]]
        assert det.line(1) == det.line(3)
    assert out[:2] == lines
    assert out[2] == "2 %d %d" % tuple(status)
    assert all(l.count("height") >= 2 for l in lines)


# ---- 5. the bound rule ----
@gpu
def test_group_filters_hold_for_every_member_camera(S):
    """tests/threshold_frames.py's points on the sides and thresholds of each step's quadrilateral, seen by a camera displaced by
    several metres (a large f32 bound epsc), in a group whose FIRST member is the scene pose's camera (a small epsc) with an empty
    frame: the union is the displaced camera's frame, so the construction holds, and the group's quadrilateral filters must use
    the larger bound of the two cameras"""
    import threshold_frames as T
    w, h = 640, 480
    cfg = S.default_config(w, h)
    tr = T.transforms(S)
    xf_s, xf_t = tr["scene"][0], tr["translated"][0]
    assert T.Bounds(cfg, xf_t).epsc > 2 * T.Bounds(cfg, xf_s).epsc
    o0 = H.oracle_process(H.load_oracle(), cfg, xf_t, T.base_frame(cfg, xf_t))
    quads = {s: o0.plateaus[s]["quad_world"] for s in (1, 2, 3)}
    f, pts, _ = T.quad_edges(cfg, xf_t, quads)
    xyz = np.stack([np.zeros_like(f), f]).astype(np.float32)
    g = oracle_group(cfg, [xf_s, xf_t], xyz)
    with S.Detector(cfg, xf_s, max_frames=2) as det:
        det.set_cameras([S.make_camera(xf_s), S.make_camera(xf_t)])
        for flags in (0, A.FLAG_STAGE_TIMING):
            d = H.to_device(det, xyz)
            det.process_groups_device(d, [0, 1], [2], flags)
            det.free(d)
            _check_group(S, det, cfg, 0, g, flags)
            r = H.gpu_result(det, 1)
            for s in (1, 2, 3):
                assert r.plateaus[s]["n_in_quad"] == g.rec.plateaus[s]["n_in_quad"], s
            assert det.stats().n_quad_exact >= len(pts) // 2, (det.stats().n_quad_exact, len(pts))
