"""Test infrastructure: loaders for the oracle (C restatement), the compiled reference (oracle/_ref)
and scene helpers. Only tests/, bench.py's CPU legs and __graft_entry__.smoke() use this."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stair_step_detector_b200 import _abi as A  # noqa: E402

ORACLE_DIR = os.path.join(ROOT, "oracle")
# the original project's sources (the C++ stair-step-detector); the tests that compare with it skip without them
REF_SRC = os.environ.get("SSD_REFERENCE_DIR", "")
_vp = C.c_void_p
_P = C.POINTER


class Derived(C.Structure):
    _fields_ = [("height_interval_reciprocal", C.c_double), ("min_height", C.c_int32), ("min_img_y_extent", C.c_int32),
                ("x_to_image", C.c_double), ("y_to_image", C.c_double), ("x_to_world", C.c_double), ("y_to_world", C.c_double),
                ("xy_ratio", C.c_double), ("n_bins", C.c_int32), ("pad", C.c_int32)]


def ref_tag(cfg):
    return f"{cfg.width}x{cfg.height}_y{cfg.y_max:g}_z{cfg.z_max:g}"


def build_oracle():
    """oracle/libssd_oracle.so, rebuilt if stale; in a read-only tree a stale library is rebuilt in a temporary directory"""
    path = os.path.join(ORACLE_DIR, "libssd_oracle.so")
    if os.access(ORACLE_DIR, os.W_OK):
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "oracle"], check=True)
        return path
    if subprocess.run(["make", "-s", "-q", "-C", ORACLE_DIR, "oracle"]).returncode == 0:
        return path
    tmp = tempfile.mkdtemp(prefix="ssd_oracle_")
    atexit.register(shutil.rmtree, tmp, True)
    path = os.path.join(tmp, "libssd_oracle.so")
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "oracle", f"ORACLE_LIB={path}"], check=True)
    return path


def load_oracle():
    lib = C.CDLL(build_oracle())
    lib.ssd_oracle_derive.argtypes = [_P(A.Config), _P(Derived)]
    lib.ssd_oracle_process.argtypes = [_P(A.Config), _P(A.Transform), _vp, _vp, _vp, C.c_int, _P(A.FrameInfo), _P(A.Plateau), _P(A.Step)]
    lib.ssd_oracle_process_batch.argtypes = [_P(A.Config), _P(A.Transform), _vp, C.c_int, _vp]
    lib.ssd_oracle_detect_outline.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_double, _P(C.c_double), _P(C.c_int)]
    lib.ssd_oracle_detect_front_edge.argtypes = [_vp, C.c_int, C.c_int, _P(C.c_double), _P(C.c_double), _P(C.c_int)]
    lib.ssd_oracle_close.argtypes = [_vp, C.c_int, C.c_int]
    lib.ssd_oracle_points_in_quad.argtypes = [_P(C.c_double), _vp, C.c_int, _vp, _P(C.c_int)]
    lib.ssd_oracle_camera_to_world.argtypes = [_P(A.Transform), _vp, C.c_int, _vp]
    lib.ssd_oracle_make_transform.argtypes = [_P(C.c_double), _P(C.c_double), _P(A.Transform)]
    lib.ssd_oracle_serialize.argtypes = [_P(A.Step), C.c_int, C.c_char_p, C.c_size_t]
    lib.ssd_oracle_inverse3.argtypes = [_P(C.c_double), _P(C.c_double)]
    lib.ssd_oracle_vertical_faces.argtypes = [_P(A.Config), _P(A.Transform), _vp, _vp, _P(A.Plateau), C.c_int, _P(A.Riser), C.c_int, _P(C.c_int)]
    lib.ssd_oracle_last_overlay.argtypes = [_P(A.Transform), _P(C.c_double), _P(A.Intrinsics), _P(A.Overlay), C.c_int, _P(C.c_int)]
    return lib


def ref_available():
    return bool(REF_SRC) and os.path.isdir(REF_SRC)


def ref_path(cfg):
    return os.path.join(ORACLE_DIR, "_ref", f"libssd_ref_{ref_tag(cfg)}.so")


def build_ref(cfg):
    """Compile the reference TUs by path for this configuration (needs SSD_REFERENCE_DIR)."""
    path = ref_path(cfg)
    if ref_available():
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "ref", f"REF={REF_SRC}", f"W={cfg.width}", f"H={cfg.height}",
                        f"XMIN={cfg.x_min:g}", f"XMAX={cfg.x_max:g}", f"YMIN={cfg.y_min:g}", f"YMAX={cfg.y_max:g}",
                        f"ZMIN={cfg.z_min:g}", f"ZMAX={cfg.z_max:g}", f"TAG={ref_tag(cfg)}"], check=True)
    return path if os.path.exists(path) else None


def load_ref(cfg):
    path = build_ref(cfg)
    if path is None:
        return None
    lib = C.CDLL(path)
    lib.ssd_ref_last_error.restype = C.c_char_p
    lib.ssd_ref_config.argtypes = [_P(A.Config)]
    lib.ssd_ref_derived.argtypes = [_P(C.c_int), _P(C.c_int), _P(C.c_double), _P(C.c_double), _P(C.c_int)]
    lib.ssd_ref_world_to_image.argtypes = [_vp, C.c_int, _vp]
    lib.ssd_ref_image_to_world.argtypes = [_vp, C.c_int, _vp]
    lib.ssd_ref_make_transform.argtypes = [_P(C.c_double), _P(C.c_double), _P(A.Transform)]
    lib.ssd_ref_process.argtypes = [_P(A.Transform), _vp, _vp, _vp, C.c_int, _P(A.FrameInfo), _P(A.Plateau), _P(A.Step), C.c_char_p, C.c_size_t]
    lib.ssd_ref_process_timed.argtypes = [_P(A.Transform), _vp, C.c_int, C.c_int, C.c_int, _P(C.c_double), _P(C.c_int)]
    lib.ssd_ref_detect_outline.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_double, _P(C.c_double), _P(C.c_int)]
    lib.ssd_ref_detect_front_edge.argtypes = [_vp, C.c_int, C.c_int, _P(C.c_double), _P(C.c_double), _P(C.c_int)]
    lib.ssd_ref_close.argtypes = [_vp, C.c_int, C.c_int]
    lib.ssd_ref_points_in_quad.argtypes = [_P(C.c_double), _vp, C.c_int, _vp, _P(C.c_int)]
    lib.ssd_ref_camera_to_world.argtypes = [_P(A.Transform), _vp, C.c_int, _vp]
    lib.ssd_ref_serialize.argtypes = [_P(A.Step), C.c_int, C.c_char_p, C.c_size_t]
    lib.ssd_ref_load_calibration.argtypes = [_P(A.Transform)]
    lib.ssd_ref_last_overlay.argtypes = [_vp, _vp, _vp, C.c_int, _P(C.c_int)]
    lib.ssd_ref_set_intrinsics.argtypes = [_P(A.Intrinsics)]
    lib.ssd_ref_a_inv.argtypes = [_P(A.Transform), _P(C.c_double)]
    got = A.Config()
    lib.ssd_ref_config(C.byref(got))
    for f, _ in A.Config._fields_:
        if f != "reserved" and getattr(got, f) != getattr(cfg, f):
            raise RuntimeError(f"reference build config mismatch on {f}: {getattr(got, f)} != {getattr(cfg, f)}")
    return lib


def ptr(a):
    return a.ctypes.data_as(_vp)


def hexf(v):
    """a double as exact text (float.hex) for golden JSON files; float.fromhex reads it back"""
    return float(v).hex()


def unhexf(v):
    return np.array([float.fromhex(x) for x in v]) if isinstance(v, list) else float.fromhex(v)


def digest(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


_PLATEAU_INTS = ("height", "hmin", "hmax", "n_points", "valid", "outlined", "n_in_quad", "quad_status")


def frame_record(r, status_mask):
    """a FrameResult as JSON: labels as a SHA-256 digest, doubles exact, status with the bits of status_mask only"""
    info = {k: int(v) for k, v in r.info.items()}
    info["status"] &= status_mask
    return dict(labels_sha256=digest(r.labels), hist=[int(v) for v in r.hist], info=info,
                plateaus=[dict({k: int(p[k]) for k in _PLATEAU_INTS}, quad_world=[hexf(v) for v in p["quad_world"].ravel()], mean_z=hexf(p["mean_z"]))
                          for p in r.plateaus],
                steps=[dict(height=hexf(s["height"]), quad=[hexf(v) for v in s["quad"].ravel()]) for s in r.steps])


def frame_from_record(d):
    """frame_record back to a FrameResult (labels None: compare d["labels_sha256"] with digest(labels))"""
    plats = [dict({k: p[k] for k in _PLATEAU_INTS}, quad_world=unhexf(p["quad_world"]).reshape(4, 2), mean_z=unhexf(p["mean_z"]))
             for p in d["plateaus"]]
    steps = [dict(height=unhexf(s["height"]), quad=unhexf(s["quad"]).reshape(4, 2)) for s in d["steps"]]
    return FrameResult(None, np.array(d["hist"], np.uint32), dict(d["info"]), plats, steps)


def compare_with_record(d, o, tol):
    """compare_results of a stored frame_record against the FrameResult o, labels by digest"""
    bad = compare_results(frame_from_record(d), o, tol=tol)
    if digest(o.labels) != d["labels_sha256"]:
        bad.append("labels differ")
    return bad


class FrameResult:
    """Everything one frame produces, in numpy/python form, from any of the three implementations."""

    def __init__(self, labels, hist, info, plats, steps, line=None):
        self.labels, self.hist, self.info, self.plateaus, self.steps, self.line = labels, hist, info, plats, steps, line


def _collect(labels, hist, info, plats, steps, line=None):
    K = info.n_plateaus
    P = [dict(height=p.height, hmin=p.hmin, hmax=p.hmax, n_points=p.n_points, valid=p.valid, outlined=p.outlined,
              n_in_quad=p.n_in_quad, quad_status=p.quad_status,
              quad_world=np.array([[p.quad_world[c][0], p.quad_world[c][1]] for c in range(4)]), mean_z=p.mean_z)
         for p in plats[:K]]
    S = [dict(height=s.height, quad=np.array([[s.quad[c][0], s.quad[c][1]] for c in range(4)])) for s in steps[:info.n_steps]]
    I = {f: getattr(info, f) for f, _ in A.FrameInfo._fields_}
    return FrameResult(labels, hist[:info.n_bins].copy(), I, P, S, line)


def oracle_process(lib, cfg, xf, xyz):
    N = cfg.width * cfg.height
    labels = np.empty(N, np.uint8)
    hist = np.zeros(A.MAX_BINS, np.uint32)
    info = A.FrameInfo()
    plats = (A.Plateau * A.MAX_PLATEAUS)()
    steps = (A.Step * A.MAX_STEPS)()
    xyz = np.ascontiguousarray(xyz, np.float32)
    rc = lib.ssd_oracle_process(C.byref(cfg), C.byref(xf), ptr(xyz), ptr(labels), ptr(hist), A.MAX_BINS, C.byref(info), plats, steps)
    assert rc == 0, rc
    return _collect(labels, hist, info, plats, steps)


def ref_process(lib, cfg, xf, xyz):
    N = cfg.width * cfg.height
    labels = np.empty(N, np.uint8)
    hist = np.zeros(A.MAX_BINS, np.uint32)
    info = A.FrameInfo()
    plats = (A.Plateau * A.MAX_PLATEAUS)()
    steps = (A.Step * A.MAX_STEPS)()
    line = C.create_string_buffer(1 << 14)
    xyz = np.ascontiguousarray(xyz, np.float32)
    rc = lib.ssd_ref_process(C.byref(xf), ptr(xyz), ptr(labels), ptr(hist), A.MAX_BINS, C.byref(info), plats, steps, line, len(line))
    assert rc == 0, (rc, lib.ssd_ref_last_error())
    return _collect(labels, hist, info, plats, steps, line.value.decode())


def oracle_vertical_faces(lib, cfg, xf, xyz, labels=None, plats=None):
    """ssd_gpu_riser records of one frame by the oracle's restatement of the definition (include/ssd_gpu.h). labels / plats: a
    FrameResult-independent way to feed the labels and plateau bands of another implementation (e.g. the compiled reference)."""
    xyz = np.ascontiguousarray(xyz, np.float32)
    N = cfg.width * cfg.height
    if labels is None:
        labels = np.empty(N, np.uint8)
        hist = np.zeros(A.MAX_BINS, np.uint32)
        info = A.FrameInfo()
        plats = (A.Plateau * A.MAX_PLATEAUS)()
        steps = (A.Step * A.MAX_STEPS)()
        assert lib.ssd_oracle_process(C.byref(cfg), C.byref(xf), ptr(xyz), ptr(labels), ptr(hist), A.MAX_BINS, C.byref(info), plats, steps) == 0
        K = info.n_plateaus
    else:
        K = len(plats)
        arr = (A.Plateau * A.MAX_PLATEAUS)()
        for k, pl in enumerate(plats):
            arr[k].hmin, arr[k].hmax = pl["hmin"], pl["hmax"]
        plats = arr
        labels = np.ascontiguousarray(labels, np.uint8)
    out = (A.Riser * A.MAX_PLATEAUS)()
    n = C.c_int()
    assert lib.ssd_oracle_vertical_faces(C.byref(cfg), C.byref(xf), ptr(xyz), ptr(labels), plats, K, out, A.MAX_PLATEAUS, C.byref(n)) == 0
    return [{f: getattr(r, f) for f, _ in A.Riser._fields_ if f != "pad"} for r in out[:n.value]]


def oracle_overlay(lib, xf, a_inv, intr):
    """drawStairStep's projected quadrilaterals of the last oracle_process on this thread: (n_steps, 4, 2) float32."""
    out = (A.Overlay * A.MAX_STEPS)()
    n = C.c_int()
    arr = (C.c_double * 9)(*[float(v) for v in np.asarray(a_inv, np.float64).ravel()])
    assert lib.ssd_oracle_last_overlay(C.byref(xf), arr, C.byref(intr), out, A.MAX_STEPS, C.byref(n)) == 0
    return np.array([[[o.px[c][0], o.px[c][1]] for c in range(4)] for o in out[:n.value]], np.float32).reshape(n.value, 4, 2)


def ref_overlay(lib):
    """The drawQuadrilateral calls of the last ref_process on this thread (the harness records the arguments the
    reference's drawStairStep passes): px (n_calls, 4, 2) float32, label (n_calls, 2, 2), z_label (n_calls)."""
    cap = 2 * A.MAX_STEPS
    px = np.zeros((cap, 4, 2), np.float32)
    label = np.zeros((cap, 2, 2), np.float64)
    z = np.zeros(cap, np.float64)
    n = C.c_int()
    assert lib.ssd_ref_last_overlay(ptr(px), ptr(label), ptr(z), cap, C.byref(n)) == 0
    return px[:n.value], label[:n.value], z[:n.value]


def ref_a_inv(lib, xf):
    out = (C.c_double * 9)()
    assert lib.ssd_ref_a_inv(C.byref(xf), out) == 0
    return np.array(out[:])


def deproject_np(scene, depth):
    """numpy restatement of ssd_deproject_pixel: single f32 operations in the same order."""
    H, W = depth.shape
    u = np.arange(W, dtype=np.float32)[None, :]
    v = np.arange(H, dtype=np.float32)[:, None]
    xn = (u - np.float32(scene.ppx)) / np.float32(scene.fx)
    yn = (v - np.float32(scene.ppy)) / np.float32(scene.fy)
    z = depth.astype(np.float32) * np.float32(scene.depth_unit)
    out = np.empty((H, W, 3), np.float32)
    out[..., 0] = z * xn
    out[..., 1] = z * yn
    out[..., 2] = z
    return out


def compare_results(a, b, tol=1e-4, check_labels=True):
    """a, b: FrameResult. Labels/histogram/peaks exact; step heights and corners within tol metres
    (0.1 mm, BASELINE.json north_star). Returns a list of mismatch strings."""
    bad = []
    if not np.array_equal(a.hist, b.hist):
        bad.append("histogram differs")
    if check_labels and a.labels is not None and b.labels is not None:
        n = int((a.labels != b.labels).sum())
        if n:
            bad.append(f"{n} labels differ")
    for k in ("n_bins", "n_plateaus", "ground_index", "first_valid_index", "n_steps", "n_nonzero", "n_in_range"):
        if a.info[k] != b.info[k]:
            bad.append(f"info.{k}: {a.info[k]} != {b.info[k]}")
    for i, (p, q) in enumerate(zip(a.plateaus, b.plateaus)):
        for k in ("height", "hmin", "hmax", "n_points", "valid", "outlined"):
            if p[k] != q[k]:
                bad.append(f"plateau {i}.{k}: {p[k]} != {q[k]}")
        if p["valid"] and q["valid"]:
            if not np.allclose(p["quad_world"], q["quad_world"], rtol=0, atol=tol):
                bad.append(f"plateau {i}.quad_world differs by {np.abs(p['quad_world'] - q['quad_world']).max():.3g}")
            if p["quad_status"] == 0 and q["quad_status"] == 0:
                if p["n_in_quad"] != q["n_in_quad"]:
                    bad.append(f"plateau {i}.n_in_quad: {p['n_in_quad']} != {q['n_in_quad']}")
                if not np.isclose(p["mean_z"], q["mean_z"], rtol=0, atol=tol, equal_nan=True):
                    bad.append(f"plateau {i}.mean_z: {p['mean_z']} != {q['mean_z']}")
    for i, (s, t) in enumerate(zip(a.steps, b.steps)):
        if not np.isclose(s["height"], t["height"], rtol=0, atol=tol, equal_nan=True):
            bad.append(f"step {i}.height: {s['height']} != {t['height']}")
        if not np.allclose(s["quad"], t["quad"], rtol=0, atol=tol, equal_nan=True):
            bad.append(f"step {i}.quad differs by {np.abs(s['quad'] - t['quad']).max():.3g}")
    return bad


# ---- the GPU results of a Detector, in the form of oracle_process's ----
def gpu_result(det, frame):
    """everything the last call produced for one frame (labels, histogram, plateaus, steps, result line)"""
    info = det.frame_info(frame)
    plats, _ = det.plateaus(frame)
    steps = (A.Step * A.MAX_STEPS)()
    n = C.c_int()
    det._ck(det._l.ssd_gpu_get_steps(det._h, frame, steps, A.MAX_STEPS, C.byref(n), None), "get_steps")
    hist = np.zeros(A.MAX_BINS, np.uint32)
    hist[:info.n_bins] = det.histogram(frame)
    return _collect(det.labels(frame), hist, info, plats, steps, det.line(frame))


def exact(r):
    """everything a frame produced, doubles as exact hex, labels as a digest, and the result line"""
    return frame_record(r, 0xffffffff), r.line


def to_device(det, a):
    """a copy of host array a in device memory (free with det.free)"""
    p = det.malloc(a.nbytes)
    det.h2d(p, a)
    return p
