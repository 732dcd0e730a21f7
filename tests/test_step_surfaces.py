"""Step surfaces (ssd_gpu_set_step_surfaces, include/ssd_gpu.h): least-squares plane, tilt, flatness and z extent of the points
each step is measured from -- the pixels its step labels mark.

Without a GPU: the oracle's restatement (ssd_oracle_step_surfaces, tests/native/oracle_step_surfaces.c) against an independent
evaluation of the definition here, with Python integers for the moments, field for field and bit for bit; known answers on flat
vertex staircases seen through a camera tilted by a known angle; invariants against the step records. On the GPU every field is compared with the oracle for equality."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
import test_gpu_step_labels as L
from stair_step_detector_b200 import _abi as A

gpu = pytest.mark.gpu
_P = C.POINTER
FIELDS = [f for f, _ in A.StepSurface._fields_]


_ORACLE = {}


def surfaces_oracle():
    """tests/native/oracle_step_surfaces.c compiled with oracle/Makefile's flags into a temporary directory"""
    if "lib" not in _ORACLE:
        import atexit
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="ssd_oracle_surfaces_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libssd_oracle_surfaces.so")
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                        os.path.join(H.ROOT, "tests", "native", "oracle_step_surfaces.c"), "-lm"], check=True)
        lib = C.CDLL(out)
        lib.ssd_oracle_step_surfaces.argtypes = [_P(A.Config), C.c_int, _P(A.Transform), C.c_void_p, C.c_void_p, C.c_int,
                                                 _P(A.Transform), _P(A.StepSurface)]
        _ORACLE["lib"] = lib
    return _ORACLE["lib"]


def as_dict(r):
    return {f: (tuple(getattr(r, f)) if f in ("centroid", "gradient") else getattr(r, f)) for f in FIELDS}


def oracle_surfaces(oracle, cfg, xfs, xyz, smap, n_steps, ext_xf):
    """ssd_oracle_step_surfaces (tests/native/oracle_step_surfaces.c) of the member frames xyz (M, N, 3) with their step labels
    smap (M, N)"""
    M = len(xfs)
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(M, -1, 3)
    smap = np.ascontiguousarray(smap, np.uint8).reshape(M, -1)
    out = (A.StepSurface * A.MAX_STEPS)()
    assert surfaces_oracle().ssd_oracle_step_surfaces(C.byref(cfg), M, (A.Transform * M)(*xfs), H.ptr(xyz), H.ptr(smap),
                                                      n_steps, C.byref(ext_xf), out) == 0
    return [as_dict(r) for r in out[:n_steps]]


# ---- the definition, evaluated independently ----
def _sum(v):
    """exact sum of non-negative integers below 2^64 (uint64) as a Python int"""
    v = np.asarray(v, np.uint64)
    return int(np.sum(v >> np.uint64(32))) * (1 << 32) + int(np.sum(v & np.uint64(0xffffffff)))


def python_surfaces(cfg, xfs, xyz, smap, n_steps, ext):
    M = len(xfs)
    xyz = np.asarray(xyz, np.float32).reshape(M, -1, 3).astype(np.float64)
    smap = np.asarray(smap, np.uint8).reshape(M, -1)
    fix = {k: [] for k in "XYZ"}
    for s in range(n_steps):
        for k in fix:
            fix[k].append([])
    for m, xf in enumerate(xfs):
        a, b = np.array(xf.a[:]).reshape(3, 3), np.array(xf.b[:])
        x, y, z = xyz[m, :, 0], xyz[m, :, 1], xyz[m, :, 2]
        w = [((a[i, 0] * x + a[i, 1] * y) + a[i, 2] * z) + b[i] for i in range(3)]  # CameraToWorld, left to right
        for s in range(n_steps):
            sel = smap[m] == s
            for k, wk, lo in zip("XYZ", w, (cfg.x_min, cfg.y_min, cfg.z_min)):
                fix[k][s].append(np.trunc((wk[sel] - lo) * 65536.0).astype(np.int64))
    out = []
    for s in range(n_steps):
        X, Y, Z = (np.concatenate(fix[k][s]).astype(np.uint64) for k in "XYZ")
        n = len(X)
        r = dict(n_points=n, fit_valid=0, centroid=(0.0, 0.0, 0.0), gradient=(0.0, 0.0), tilt_deg=0.0, rms_dz=0.0, z_lo=0.0, z_hi=0.0)
        if n:
            assert max(int(X.max()), int(Y.max()), int(Z.max())) < 1 << 32
            Sx, Sy, Sz = _sum(X), _sum(Y), _sum(Z)
            Sxx, Sxy, Syy, Sxz, Syz, Szz = (_sum(p * q) for p, q in ((X, X), (X, Y), (Y, Y), (X, Z), (Y, Z), (Z, Z)))
            cxx, cxy, cyy = float(n * Sxx - Sx * Sx), float(n * Sxy - Sx * Sy), float(n * Syy - Sy * Sy)
            cxz, cyz, czz = float(n * Sxz - Sx * Sz), float(n * Syz - Sy * Sz), float(n * Szz - Sz * Sz)
            det = cxx * cyy - cxy * cxy
            ga = gb = 0.0
            if n >= 3 and det > 0:
                ga = (cxz * cyy - cyz * cxy) / det
                gb = (cyz * cxx - cxz * cxy) / det
                res = czz - ga * cxz - gb * cyz
                r.update(fit_valid=1, rms_dz=math.sqrt(max(res, 0.0)) / float(n) / 65536.0,
                         tilt_deg=math.atan(math.sqrt(ga * ga + gb * gb)) * (180.0 / math.pi))
            xm, ym, zm = (lo + float(S_) / float(n) / 65536.0 for lo, S_ in ((cfg.x_min, Sx), (cfg.y_min, Sy), (cfg.z_min, Sz)))
            ea, eb = ext.ext_a, ext.ext_b
            r.update(centroid=((ea[0] * xm + ea[1] * ym) + eb[0], (ea[2] * xm + ea[3] * ym) + eb[1], ext.ext_z + zm),
                     gradient=(ea[0] * ga + ea[1] * gb, ea[2] * ga + ea[3] * gb),
                     z_lo=ext.ext_z + (cfg.z_min + float(int(Z.min())) / 65536.0), z_hi=ext.ext_z + (cfg.z_min + float(int(Z.max())) / 65536.0))
        out.append(r)
    return out


def check_invariants(o, surf, what=""):
    """n_points == n_in_quad of the step's plateau; z_lo <= centroid z <= z_hi; centroid z within 1e-4 m of the step's height"""
    plats = L.step_plateaus(o.info, o.plateaus)
    assert len(surf) == len(plats) == o.info["n_steps"], what
    for s, l in enumerate(plats):
        r = surf[s]
        assert r["n_points"] == o.plateaus[l]["n_in_quad"], (what, s)
        if r["n_points"]:
            assert r["z_lo"] <= r["centroid"][2] <= r["z_hi"], (what, s, r)
            if o.steps[s]["quad"].any():  # (the ground step with an invalid front edge has height 0)
                assert abs(r["centroid"][2] - o.steps[s]["height"]) < 1e-4, (what, s, r["centroid"][2], o.steps[s]["height"])


def frame_surfaces(oracle, cfg, xf, xyz):
    """oracle result, step labels and surfaces of one frame"""
    o, m = L.oracle_map(oracle, cfg, xf, xyz)
    return o, m, oracle_surfaces(oracle, cfg, [xf], xyz, m, o.info["n_steps"], xf)


# ---- without a GPU ----
def test_step_surface_symbols_are_declared_and_bound(S):
    hdr = open(os.path.join(H.ROOT, "include", "ssd_gpu.h")).read()
    assert re.search(r"#define SSD_GPU_ABI_VERSION 3\b", hdr)
    assert re.search(r"typedef struct ssd_gpu_step_surface\b", hdr)
    assert C.sizeof(A.StepSurface) == 80
    lib = S.lib()
    for name, nargs in (("ssd_gpu_set_step_surfaces", 2), ("ssd_gpu_get_step_surfaces", 5)):
        assert re.search(r"\bint " + name + r"\(", hdr), name
        assert len(A.PROTOTYPES[name][1]) == nargs, name
        assert getattr(lib, name).restype is C.c_int, name


GOLDEN = L.GOLDEN


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_equals_the_definition_on_the_golden_scenes(S, oracle, path):
    import test_oracle_golden as G
    z, meta, sc, xf = G.load_case(path)
    cfg = S.default_config(meta["width"], meta["height"])
    xyz = H.deproject_np(sc, z["depth"])
    o, m, got = frame_surfaces(oracle, cfg, xf, xyz)
    assert got == python_surfaces(cfg, [xf], xyz, m, o.info["n_steps"], xf)
    check_invariants(o, got, path)


@pytest.mark.parametrize("key", ["frames_random_scenes/320x240", "frames_random_scenes/640x480", "frames_random_scenes/1024x768",
                                 "frames_hires/4096x3072"])
def test_oracle_equals_the_definition_on_the_reference_runs(S, oracle, key):
    import test_oracle_vs_ref as R
    kind, size = key.split("/")
    w, h = (int(v) for v in size.split("x"))
    if kind == "frames_hires":
        _, _, ck, sk, n = next(c for c in R.HIRES_CASES if c[:2] == (w, h))
        inputs = R.frames_hires_inputs(S, w, h, ck, sk, n)
    else:
        inputs = R.frames_random_scenes_inputs(S, w, h, {320: 10, 640: 6, 1024: 3}[w])
    n_fits = 0
    for i, (cfg, xf, xyz) in enumerate(inputs):
        o, m, got = frame_surfaces(oracle, cfg, xf, xyz)
        assert got == python_surfaces(cfg, [xf], xyz, m, o.info["n_steps"], xf), (key, i)
        check_invariants(o, got, (key, i))
        n_fits += sum(r["fit_valid"] for r in got)
    assert n_fits > 0


def group_case(S, w, h, sizes, seed):
    """groups of the three-camera rig: per group the member transforms, frames, step labels (reference map of the group oracle)
    and step count; and the camera table, frames and camera index of the whole call"""
    import test_gpu_groups as G
    bases = G.camera_scenes(S, w, h)
    cams = [S.scene_camera(b) for b in bases]
    idx = np.random.default_rng(seed).integers(0, 3, sum(sizes)).astype(np.int32)
    depth, xyz = G.frames_of(S, bases, idx, seed)
    orc = G.group_oracle()
    for fn in ("ssd_oracle_camera_to_world", "ssd_oracle_points_in_quad"):
        getattr(orc, fn).argtypes = getattr(H.load_oracle(), fn).argtypes
    cfg = S.default_config(w, h)
    groups = []
    for s, k in zip(G.starts(sizes), sizes):
        xfs = [cams[c].xf for c in idx[s:s + k]]
        g = G.oracle_group(cfg, xfs, xyz[s:s + k])
        m = L.reference_map(orc, xfs, xyz[s:s + k], g.rec.labels, g.rec.info, g.rec.plateaus)
        groups.append((xfs, xyz[s:s + k], m, g.rec))
    return cfg, cams, idx, depth, xyz, groups


def test_oracle_equals_the_definition_on_a_group(S, oracle):
    cfg, _, _, _, _, groups = group_case(S, 320, 240, [3], 9)
    xfs, xyz, m, rec = groups[0]
    got = oracle_surfaces(oracle, cfg, xfs, xyz, m, rec.info["n_steps"], xfs[0])
    assert got == python_surfaces(cfg, xfs, xyz, m, rec.info["n_steps"], xfs[0])
    assert sum(r["fit_valid"] for r in got) >= 2
    check_invariants(rec, got, "group of 3")


# ---- known answers: a flat vertex staircase through a camera tilted by theta ----
def flat_staircase(seed):
    """ground and three treads, every point exactly at its tread's height (320x240, camera shifted as in test_gpu_edge_cases)"""
    import test_gpu_edge_cases as E
    rng = np.random.default_rng(seed)
    return E.frame_of([E.slab(rng, 20000, -0.45, 0.45, 0.15, 0.45, 0.004, 0), E.slab(rng, 20000, -0.45, 0.45, 0.45, 0.75, 0.185, 0),
                       E.slab(rng, 20000, -0.45, 0.45, 0.75, 1.05, 0.365, 0), E.slab(rng, 12000, -0.45, 0.45, 1.05, 1.25, 0.545, 0)])


def rotated(xf, axis, theta):
    """xf composed with a rotation by theta about the world x or y axis: a' = R a, b' = R b"""
    c, s = math.cos(theta), math.sin(theta)
    R = np.array([[1, 0, 0], [0, c, -s], [0, s, c]]) if axis == "x" else np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    out = A.Transform()
    C.memmove(C.byref(out), C.byref(xf), C.sizeof(out))
    a, b = R @ np.array(xf.a[:]).reshape(3, 3), R @ np.array(xf.b[:])
    for i in range(9):
        out.a[i] = a.flat[i]
    for i in range(3):
        out.b[i] = b[i]
    return out


# Bounds of the known-answer test, and what the oracle gives on these frames: |tilt - theta| <= 4e-5 deg, rms_dz <= 4.5e-6 m
# (float32 vertices and the 1/65536 m fixed point), off-axis gradient <= 1e-6, |centroid z - height| <= 1.2e-5 m.
TILT_TOL_DEG, RMS_MAX_M, OFF_AXIS_MAX, HEIGHT_TOL_M = 0.01, 0.05e-3, 1e-5, 1e-4


@pytest.mark.parametrize("axis", ["x", "y"])
@pytest.mark.parametrize("deg", [0.0, 0.5, -0.5])
def test_known_tilt_of_a_flat_staircase(S, oracle, axis, deg):
    import test_gpu_edge_cases as E
    cfg = S.default_config(E.W, E.HH)
    xf0 = E.shifted(E.identity_xf())
    xyz = flat_staircase(5)
    o0, _, _ = frame_surfaces(oracle, cfg, xf0, xyz)
    xf = rotated(xf0, axis, math.radians(deg))
    o, m, got = frame_surfaces(oracle, cfg, xf, xyz)
    # the tilt leaves the same steps detected
    assert o.info["status"] == o0.info["status"] == 0 and o.info["n_steps"] == o0.info["n_steps"] == 4
    assert L.step_plateaus(o.info, o.plateaus) == L.step_plateaus(o0.info, o0.plateaus)
    check_invariants(o, got, (axis, deg))
    t = math.tan(math.radians(deg))
    # rotation about x: z rises along y (dz/dy = tan theta); about y: dz/dx = -tan theta. ext_a is the identity here.
    want = (0.0, t) if axis == "x" else (-t, 0.0)
    for s, r in enumerate(got):
        assert r["fit_valid"] == 1, s
        assert abs(r["tilt_deg"] - abs(deg)) < TILT_TOL_DEG, (s, r["tilt_deg"])
        assert r["rms_dz"] < RMS_MAX_M, (s, r["rms_dz"])
        assert abs(r["gradient"][0] - want[0]) < OFF_AXIS_MAX and abs(r["gradient"][1] - want[1]) < OFF_AXIS_MAX, (s, r["gradient"])
        assert abs(r["centroid"][2] - o.steps[s]["height"]) < HEIGHT_TOL_M
    assert got == python_surfaces(cfg, [xf], xyz, m, o.info["n_steps"], xf)


# ---- on the GPU ----
def assert_surfaces(det, want, what, f0=0):
    for f, w in enumerate(want):
        got = det.step_surfaces(f0 + f)
        assert got == w, (what, f, got, w)


def want_frames(oracle, cfg, xfs, xyz):
    return [frame_surfaces(oracle, cfg, xf, x)[2] for xf, x in zip(xfs, xyz)]


@gpu
@pytest.mark.parametrize("w,h", [(320, 240), (640, 480), (1024, 768)])
def test_random_scenes_fused_and_seven_launch(S, oracle, w, h):
    cfg = S.default_config(w, h)
    for kw, seed, n in ((dict(), 11, 4), (dict(rotate180=1, n_occluders=2), 12, 18)):
        base, sc = L.scenes_of(S, w, h, seed, n, **kw)
        xf = S.scene_transform(base)
        depth = np.stack([S.synth_depth_host(s) for s in sc])
        xyz = np.stack([S.deproject_host(s, d) for s, d in zip(sc, depth)])
        want = want_frames(oracle, cfg, [xf] * n, xyz)
        assert sum(r["fit_valid"] for ws in want for r in ws) >= n
        intr = S.scene_intrinsics(base)
        with S.Detector(cfg, xf, max_frames=n) as det:
            det.set_step_labels(True)
            det.set_step_surfaces(True)
            det.process_host(xyz[:1])
            assert det.timing().n_launches == 6
            assert_surfaces(det, want[:1], "vertices/host one frame (fused)")
            det.process_host(xyz)
            assert_surfaces(det, want, ("vertices/host", n))
            d = H.to_device(det, xyz)
            det.process_device(d, n, A.FLAG_STAGE_TIMING)
            assert det.timing().n_launches == 8 * det.stage_times()["transform_bin"][1]
            assert_surfaces(det, want, "vertices/device seven-launch")
            det.free(d)
            det.process_depth_host(depth, intr)
            assert_surfaces(det, want, "z16/host")
            d = H.to_device(det, depth)
            det.process_depth_device(d, intr, n)
            assert_surfaces(det, want, "z16/device")
            det.free(d)


@gpu
def test_batch_larger_than_a_chunk(S, oracle):
    """more frames than a chunk: device input over two chunks of chunk_frames (1024) and host input over three chunks of
    the host chunk (32 frames), each chunk clearing and filling its own records; spot frames equal the oracle"""
    import ctypes as C_
    w, h = 320, 240
    N = w * h
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **L.NOISY)
    xf = S.scene_transform(base)
    n = 1100
    with S.Detector(cfg, xf, max_frames=n) as det:
        assert det.chunk_frames < n
        d_xyz = det.malloc(n * N * 12)
        det.synth_frames(base, 4243, 0, n, 3, 8, d_xyz)
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_device(d_xyz, n, A.FLAG_STAGE_TIMING)
        chunks = det.stage_times()["transform_bin"][1]
        assert chunks >= 2 and det.timing().n_launches == 8 * chunks
        spots = (0, 1, det.chunk_frames - 1, det.chunk_frames, n - 1)
        xyz = {}
        for f in spots:
            xyz[f] = np.empty((N, 3), np.float32)
            det.d2h(xyz[f], C_.c_void_p(d_xyz.value + f * N * 12))
            assert det.step_surfaces(f) == frame_surfaces(oracle, cfg, xf, xyz[f])[2], ("device", f)
        host = np.stack([xyz[f] for f in spots] * 14)  # 70 frames: three host chunks
        det.process_host(host)
        for f in (0, 31, 32, 64, 69):
            assert det.step_surfaces(f) == frame_surfaces(oracle, cfg, xf, host[f])[2], ("host", f)
        det.free(d_xyz)


@gpu
def test_hires_frame(S, oracle):
    import test_oracle_vs_ref as R
    _, _, ck, sk, _ = next(c for c in R.HIRES_CASES if c[:2] == (4096, 3072))
    cfg, xf, xyz = next(R.frames_hires_inputs(S, 4096, 3072, ck, sk, 1))
    want = want_frames(oracle, cfg, [xf], xyz[None])
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_host(xyz[None])
        assert_surfaces(det, want, "4096x3072 fused")
        d = H.to_device(det, np.ascontiguousarray(xyz[None]))
        det.process_device(d, 1, A.FLAG_STAGE_TIMING)
        assert_surfaces(det, want, "4096x3072 seven-launch")
        det.free(d)


@gpu
@pytest.mark.parametrize("name", ["BC", "IBC"])
def test_brown_conrady_lenses(S, oracle, name):
    import test_gpu_distortion as D
    w, h = 640, 480
    cfg = S.default_config(w, h)
    base, depth, xyz = D.lens_frames(S, w, h, D.LENSES[name], 5, 61)
    xf = S.scene_transform(base)
    want = want_frames(oracle, cfg, [xf] * 5, xyz)
    with S.Detector(cfg, xf, max_frames=5) as det:
        det.set_distortion(S.scene_distortion(base))
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_depth_host(depth, S.scene_intrinsics(base))
        assert_surfaces(det, want, (name, "z16/host"))
        d = H.to_device(det, depth)
        det.process_depth_device(d, S.scene_intrinsics(base), 5)
        assert_surfaces(det, want, (name, "z16/device"))
        det.free(d)


def mixed_lens_table(S):
    import test_gpu_distortion as D
    import test_gpu_groups as G
    w, h = 640, 480
    bases = [G.camera_scenes(S, w, h)[0], D.lens_scene(S, w, h, D.BC, **L.NOISY), D.lens_scene(S, w, h, D.IBC, rotate180=1, **L.NOISY)]
    idx = np.array([0, 1, 2, 2, 1, 0], np.int32)
    depth, xyz = G.frames_of(S, bases, idx, 47)
    return S.default_config(w, h), bases, [S.scene_camera(b) for b in bases], idx, depth, xyz


@gpu
def test_camera_table_with_mixed_lenses(S, oracle):
    """each frame reported through its own camera's ToExternalWorld, fixed at call time: replacing the camera table afterwards
    changes none of the surfaces"""
    cfg, bases, cams, idx, depth, xyz = mixed_lens_table(S)
    want = want_frames(oracle, cfg, [cams[c].xf for c in idx], xyz)
    with S.Detector(cfg, cams[0].xf, max_frames=len(idx)) as det:
        det.set_cameras(cams, [S.scene_distortion(b) for b in bases])
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_depth_cameras_host(depth, idx)
        assert_surfaces(det, want, "camera table z16")
        det.process_cameras_host(xyz, idx)
        assert_surfaces(det, want, "camera table vertices")
        det.set_cameras(cams[::-1])
        assert_surfaces(det, want, "after the camera table was replaced")


@gpu
def test_groups_of_1_3_and_8(S, oracle):
    """a group's surfaces from the points of all its members, each through its own camera, reported through the first member's
    ToExternalWorld; every member frame reads its group's"""
    sizes = [1, 3, 8]
    cfg, cams, idx, depth, xyz, groups = group_case(S, 320, 240, sizes, 31)
    want = []
    for (xfs, gx, m, rec), k in zip(groups, sizes):
        want += [oracle_surfaces(oracle, cfg, xfs, gx, m, rec.info["n_steps"], xfs[0])] * k
    assert sum(r["fit_valid"] for ws in want for r in ws) >= 3
    with S.Detector(cfg, cams[0].xf, max_frames=len(idx)) as det:
        det.set_cameras(cams)
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_groups_host(xyz, idx, sizes)
        assert_surfaces(det, want, "groups vertices/host")
        d = H.to_device(det, depth)
        det.process_depth_groups_device(d, idx, sizes)
        assert_surfaces(det, want, "groups z16/device")
        det.free(d)


def _edge(S, oracle, cfg, xf, xyz, bit):
    o, m, want = frame_surfaces(oracle, cfg, xf, xyz)
    assert o.info["status"] & bit, hex(o.info["status"])
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_host(xyz[None])
        assert_surfaces(det, [want], ("fused", bit))
        d = H.to_device(det, np.ascontiguousarray(xyz[None]))
        det.process_device(d, 1, A.FLAG_STAGE_TIMING)
        assert_surfaces(det, [want], ("seven-launch", bit))
        det.free(d)
    return o, want


@gpu
def test_edge_statuses(S, oracle):
    import test_gpu_edge_cases as E
    cfg = S.default_config(E.W, E.HH)
    xf = E.shifted(E.identity_xf())
    # invalid ground front edge: the all-zero step 0 still gets the surface of the pixels its step labels mark
    o, want = _edge(S, oracle, cfg, xf, L.unseen_front_edge_frame(E), A.STATUS_INVALID_FRONT_EDGE)
    assert not o.steps[0]["quad"].any()
    assert want[0]["n_points"] == o.plateaus[o.info["ground_index"]]["n_in_quad"] > 0 and want[0]["fit_valid"] == 1
    # ... and with no ground point in the quadrilateral: n == 0, an all-zero record
    rng = np.random.default_rng(13)
    xyz = E.frame_of([E.slab(rng, 9000, -0.45, 0.45, 1.0, 1.25, 0.004), E.slab(rng, 30000, -0.45, 0.45, 0.45, 0.75, 0.185)])
    o, want = _edge(S, oracle, cfg, xf, xyz, A.STATUS_INVALID_FRONT_EDGE)
    assert want[0] == as_dict(A.StepSurface()) and want[1]["n_points"] > 0
    # HMIN_WRAP: every plateau empty, n == 0 for every step
    rng = np.random.default_rng(11)
    xyz = E.frame_of([E.slab(rng, 1500, -0.4, 0.4, 0.2, 0.6, -0.095), E.slab(rng, 4000, -0.4, 0.4, 0.2, 0.6, -0.085),
                      E.slab(rng, 6000, -0.4, 0.4, 0.7, 1.1, 0.305)])
    o, want = _edge(S, oracle, cfg, xf, xyz, A.STATUS_HMIN_WRAP)
    assert all(r["n_points"] == 0 for r in want)
    # no steps
    for xyz in (np.zeros((E.N, 3), np.float32), E.frame_of([E.slab(rng, 20000, -0.45, 0.45, 0.2, 1.2, 0.004)])):
        o, want = _edge(S, oracle, cfg, xf, xyz, A.STATUS_NO_STEPS)
        assert want == []


def _everything(S, det, n):
    out = []
    for f in range(n):
        r = H.gpu_result(det, f)
        out.append((H.frame_record(r, 0xffffffff), r.line, H.digest(r.labels), H.digest(det.step_labels(f)), det.overlay(f).tobytes(),
                    det.vertical_faces(f)))
    return out


@gpu
def test_nothing_else_changes(S):
    """with surfaces on: steps, plateaus, frame info, labels, step labels, overlay and risers as with them off; one launch more
    per chunk. With them off the launch count is the chain's (5 fused / 7, plus the riser pass)."""
    w, h = 640, 480
    cfg = S.default_config(w, h)
    base, sc = L.scenes_of(S, w, h, 71, 20)
    xf = S.scene_transform(base)
    xyz = np.stack([S.deproject_host(s, S.synth_depth_host(s)) for s in sc])
    xfe = S.scene_transform_ex(base)
    with S.Detector(cfg, xf, max_frames=20) as det:
        det.set_overlay(xfe[1], S.scene_intrinsics(base))
        det.set_vertical_faces(True)
        det.set_step_labels(True)
        res = {}
        for on in (False, True, False):
            det.set_step_surfaces(on)
            for n in (1, 20):
                det.process_host(xyz[:n])
                res.setdefault((on, n), []).append((_everything(S, det, n), det.timing().n_launches))
        for n in (1, 20):
            off, on = res[(False, n)][0], res[(True, n)][0]
            assert off == res[(False, n)][1]
            assert on[0] == off[0], n
            chunks = on[1] - off[1]  # one more launch per chunk; a chunk is 5 (fused) or 7 launches, plus the riser pass
            assert chunks >= 1 and 6 * chunks <= off[1] <= 8 * chunks, (n, on[1], off[1])
        assert res[(False, 1)][0][1] == 6 and res[(True, 1)][0][1] == 7


@gpu
def test_launch_counts(S):
    """surfaces off: the parent's counts (5 fused / 7 per chunk, + 1 with risers); on: one more per chunk"""
    w, h = 320, 240
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h)
    xf = S.scene_transform(base)
    xyz = np.stack([S.deproject_host(base, S.synth_depth_host(base))] * 40)
    with S.Detector(cfg, xf, max_frames=40) as det:
        d = H.to_device(det, xyz)
        det.set_step_labels(True)
        for on in (False, True):
            det.set_step_surfaces(on)
            det.process_device(d, 1)
            assert det.timing().n_launches == 5 + on
            det.process_device(d, 40, A.FLAG_STAGE_TIMING)
            chunks = det.stage_times()["transform_bin"][1]
            assert det.timing().n_launches == (7 + on) * chunks
        det.free(d)


@gpu
def test_state_and_argument_errors(S):
    w, h = 320, 240
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h)
    xf = S.scene_transform(base)
    xyz = S.deproject_host(base, S.synth_depth_host(base))[None]
    with S.Detector(cfg, xf, max_frames=2) as det:
        def rc(fn, *a):
            return getattr(det._l, fn)(det._h, *a)
        out, n = (A.StepSurface * A.MAX_STEPS)(), C.c_int()
        get = lambda f: rc("ssd_gpu_get_step_surfaces", f, out, A.MAX_STEPS, C.byref(n))  # noqa: E731
        assert rc("ssd_gpu_set_step_surfaces", 1) == A.E_STATE  # the step labels are off
        det.process_host(xyz)
        assert get(0) == A.E_STATE  # not enabled
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        assert get(0) == A.E_STATE  # the last call ran without it
        assert rc("ssd_gpu_set_step_labels", 0) == A.E_STATE  # the surfaces read the step labels
        det.process_host(xyz)
        assert get(0) == A.OK and n.value > 0 and out[0].n_points > 0
        kept = [as_dict(r) for r in out[:n.value]]
        assert get(1) == A.E_RANGE and get(-1) == A.E_RANGE
        assert rc("ssd_gpu_get_step_surfaces", 0, None, 0, C.byref(n)) == A.OK and n.value == len(kept)
        # a rejected call leaves the surfaces readable
        assert det._l.ssd_gpu_process_host(det._h, H.ptr(np.ascontiguousarray(np.repeat(xyz, 3, 0))), 3) == A.E_RANGE
        assert det.step_surfaces(0) == kept
        # a single-stage entry point reuses the per-frame records: the surfaces go with the last call's other results
        det.detect_front_edge(np.zeros((h, w), np.uint8))
        assert get(0) == A.E_STATE
        det.process_host(xyz)
        det.set_step_surfaces(False)  # disabled after a call
        assert get(0) == A.E_STATE
        with pytest.raises(S.SsdError):
            det.step_surfaces(0)
        det.set_step_labels(False)  # allowed once the surfaces are off
    # ranges of 65536 m or more: the moments would not be exact
    with S.Detector(S.default_config(w, h, x_min=-40000.0, x_max=40000.0), xf, max_frames=1) as det:
        det.set_step_labels(True)
        assert det._l.ssd_gpu_set_step_surfaces(det._h, 1) == A.E_RANGE


@gpu
def test_cpp_step_surfaces(S, tmp_path):
    """tests/native/step_surfaces_check.cpp: Pointcloud::enableStepSurfaces / stepSurfaces on one frame equal the C getter's"""
    exe = str(tmp_path / "step_surfaces_check")
    libdir = os.path.join(H.ROOT, "stair_step_detector_b200", "lib")
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(H.ROOT, "tests", "native", "step_surfaces_check.cpp"),
                    "-L" + libdir, "-lssd_gpu", "-lssd_scene", "-Wl,-rpath," + libdir], check=True)
    w, h = 640, 480
    rec = tmp_path / "surfaces.bin"
    out = subprocess.run([exe, str(w), str(h), str(rec)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    raw = rec.read_bytes()
    got = [as_dict(A.StepSurface.from_buffer_copy(raw, i * 80)) for i in range(len(raw) // 80)]
    base = S.default_scene(w, h, noise_sigma=0.0025)
    with S.Detector(S.default_config(w, h), S.scene_transform(base), max_frames=1) as det:
        det.set_step_labels(True)
        det.set_step_surfaces(True)
        det.process_depth_host(S.synth_depth_host(base)[None], S.scene_intrinsics(base))
        assert out[0] == det.line(0)
        want = det.step_surfaces(0)
    assert got == want and len(got) >= 3
