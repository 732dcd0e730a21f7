"""stair_step_detector_b200 -- B200-native per-frame geometry hot path of stair-step-detector.

Python is only the thin ctypes binding over the C ABI (include/ssd_gpu.h) used by tests and bench.py;
the product is the CUDA library in csrc/ (kernels for sm_100a) and the C++ host classes in csrc/host/
that keep the reference's Pointcloud / Transformation / Segmentation / Stairs surface.

There is no CPU fallback: the shared library must have been built (``__graft_entry__.build()``) and
``Detector`` needs a CUDA device.
"""
import ctypes as C
import os

import numpy as np

from . import _abi as A
from ._abi import Config, FrameInfo, Plateau, Scene, Step, Timing, Transform  # noqa: F401

_lib = None


def lib():
    """The loaded libssd_gpu.so (raises ImportError if it has not been built)."""
    global _lib
    if _lib is None:
        _lib = A.load()
    return _lib


_scene_lib = None


def scene_lib():
    """libssd_scene.so: the synthetic input source (include/ssd_scene.h). Not the product: generating input never needs
    libssd_gpu.so."""
    global _scene_lib
    if _scene_lib is None:
        _scene_lib = A.load_scene()
    return _scene_lib


class SsdError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def default_config(width, height, **overrides):
    cfg = Config()
    lib().ssd_gpu_default_config(C.byref(cfg), width, height)
    for k, v in overrides.items():
        setattr(cfg, k, v)
    return cfg


def make_transform(world_pts, camera_pts):
    """GeometricTransformation(worldPoints, cameraPoints) -> Transform (reference transformation.cpp:196-215)."""
    w = (C.c_double * 9)(*np.asarray(world_pts, np.float64).ravel())
    c = (C.c_double * 9)(*np.asarray(camera_pts, np.float64).ravel())
    xf = Transform()
    rc = lib().ssd_make_transform(w, c, C.byref(xf))
    if rc:
        raise SsdError(f"ssd_make_transform failed ({rc})")
    return xf


def load_calibration(directory=""):
    """GeometricCalibration::load() (reference geometricCalibration.cpp:185-203): the transformation from the text files
    ``calibration-triangle`` and ``calibration-points`` in ``directory``. Returns (Transform, status, world_pts, camera_pts);
    status != 0 (SSD_CAL_*) means a file was missing or malformed and the transform is the identity, as in the reference."""
    xf = Transform()
    w = (C.c_double * 9)()
    c = (C.c_double * 9)()
    rc = lib().ssd_load_calibration(os.fsencode(directory), C.byref(xf), w, c)
    if rc < 0:
        raise SsdError(f"ssd_load_calibration failed ({rc})")
    return xf, rc, np.array(w).reshape(3, 3), np.array(c).reshape(3, 3)


def default_scene(width, height, **overrides):
    s = Scene()
    scene_lib().ssd_scene_default(C.byref(s), width, height)
    for k, v in overrides.items():
        setattr(s, k, v)
    return s


def scene_transform(scene):
    w = (C.c_double * 9)()
    c = (C.c_double * 9)()
    scene_lib().ssd_scene_calibration_points(C.byref(scene), w, c)
    xf = Transform()
    rc = lib().ssd_make_transform(w, c, C.byref(xf))
    if rc:
        raise SsdError(f"ssd_make_transform failed ({rc})")
    return xf


def scene_transform_ex(scene):
    """(Transform, a_inv): the camera transformation's _aInv (9 doubles, row-major) as the reference holds it,
    for Detector.set_overlay."""
    w = (C.c_double * 9)()
    c = (C.c_double * 9)()
    scene_lib().ssd_scene_calibration_points(C.byref(scene), w, c)
    xf = Transform()
    a_inv = (C.c_double * 9)()
    rc = lib().ssd_make_transform_ex(w, c, C.byref(xf), a_inv)
    if rc:
        raise SsdError(f"ssd_make_transform_ex failed ({rc})")
    return xf, np.array(a_inv[:])


def scene_camera(scene):
    """The full camera record of a synthetic scene, for Detector.set_cameras: its transform, the camera transformation's
    _aInv and the depth-stream intrinsics (ssd_gpu_camera)."""
    xf, a_inv = scene_transform_ex(scene)
    return make_camera(xf, a_inv, scene_intrinsics(scene))


def make_camera(xf, a_inv=None, intrinsics=None):
    """ssd_gpu_camera from a Transform, the 9 doubles of _aInv (overlay only) and Intrinsics (depth input and overlay; None: zero)."""
    cam = A.Camera()
    cam.xf = xf
    if a_inv is not None:
        for i, v in enumerate(np.asarray(a_inv, np.float64).ravel()):
            cam.a_inv[i] = float(v)
    if intrinsics is not None:
        cam.intr = intrinsics
    return cam


def inverse3(a):
    """boost::qvm::inverse of a 3x3 (row-major 9 doubles) as Transformation_<3>(rp, rpMapping) computes _aInv."""
    src = (C.c_double * 9)(*[float(v) for v in np.asarray(a, np.float64).ravel()])
    dst = (C.c_double * 9)()
    rc = lib().ssd_inverse3(src, dst)
    if rc:
        raise SsdError(f"ssd_inverse3 failed ({rc})")
    return np.array(dst[:])


def randomize_scene(base, base_seed, index, min_steps, max_steps):
    s = Scene()
    scene_lib().ssd_scene_randomize(C.byref(s), C.byref(base), base_seed, index, min_steps, max_steps)
    return s


def synth_depth_host(scene):
    d = np.empty((scene.height, scene.width), np.uint16)
    rc = scene_lib().ssd_synth_depth_host(C.byref(scene), _ptr(d))
    if rc:
        raise SsdError(f"ssd_synth_depth_host failed ({rc})")
    return d


def deproject_host(scene, depth):
    depth = np.ascontiguousarray(depth, np.uint16)
    xyz = np.empty((scene.height, scene.width, 3), np.float32)
    rc = scene_lib().ssd_deproject_host(C.byref(scene), _ptr(depth), _ptr(xyz))
    if rc:
        raise SsdError(f"ssd_deproject_host failed ({rc})")
    return xyz


def scene_intrinsics(scene):
    """Pin-hole intrinsics + depth unit of a synthetic scene (what rs2 would report for the depth stream)."""
    k = A.Intrinsics()
    scene_lib().ssd_scene_intrinsics(C.byref(scene), C.byref(k))
    return k


def scene_distortion(scene):
    """The lens of a synthetic scene (A.Distortion): its distortion_model and coeffs."""
    return make_distortion(scene.distortion_model, scene.coeffs[:])


def make_distortion(model, coeffs=(0.0, 0.0, 0.0, 0.0, 0.0)):
    """ssd_gpu_distortion from an rs2 model value (A.DISTORTION_*) and the five coefficients [k1, k2, p1, p2, k3]."""
    coeffs = [float(c) for c in coeffs]
    if len(coeffs) != 5:
        raise ValueError(f"a lens has 5 coefficients, got {len(coeffs)}")
    d = A.Distortion()
    d.model = int(model)
    for i, c in enumerate(coeffs):
        d.coeffs[i] = c
    return d


def serialize(steps):
    """Stairs::serialize (reference stairs.cpp:55-70) of a list of (height, 4x2 quad)."""
    arr = (Step * max(1, len(steps)))()
    for i, (h, q) in enumerate(steps):
        arr[i].height = h
        for c in range(4):
            arr[i].quad[c][0] = q[c][0]
            arr[i].quad[c][1] = q[c][1]
    n = lib().ssd_stairs_serialize(arr, len(steps), None, 0)
    buf = C.create_string_buffer(n + 1)
    lib().ssd_stairs_serialize(arr, len(steps), buf, n + 1)
    return buf.value.decode()


class Detector:
    """One GPU context: the constant transform + configuration bound to device buffers
    (replaces Pointcloud's constructor, reference pointcloud.cpp:602-606)."""

    def __init__(self, cfg, xf, device=0, max_frames=1):
        self._l = lib()
        self.cfg, self.xf, self.device, self.max_frames = cfg, xf, device, max_frames
        self.n_points = cfg.width * cfg.height
        h = C.c_void_p()
        rc = self._l.ssd_gpu_create(C.byref(cfg), C.byref(xf), device, max_frames, C.byref(h))
        if rc:
            raise SsdError(f"ssd_gpu_create failed ({rc}): {self._l.ssd_gpu_last_error(None).decode()}")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._l.ssd_gpu_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc, what):
        if rc:
            raise SsdError(f"{what} failed ({rc}): {self._l.ssd_gpu_last_error(self._h).decode()}")

    # ---- the hot path ----
    def process_host(self, xyz):
        """xyz: (n_frames, H, W, 3) or (n_frames, N, 3) float32 host array (pinned or pageable)."""
        xyz = np.ascontiguousarray(xyz, np.float32)
        n = xyz.size // (self.n_points * 3)
        self._ck(self._l.ssd_gpu_process_host(self._h, _ptr(xyz), n), "ssd_gpu_process_host")
        return n

    def process_host_ptr(self, ptr, n_frames):
        self._ck(self._l.ssd_gpu_process_host(self._h, ptr, n_frames), "ssd_gpu_process_host")

    def process_depth_host(self, depth, intrinsics):
        """depth: (n_frames, H, W) uint16 z16 depth frames in host memory -- what the reference's process() receives."""
        depth = np.ascontiguousarray(depth, np.uint16)
        n = depth.size // self.n_points
        self._ck(self._l.ssd_gpu_process_depth_host(self._h, _ptr(depth), C.byref(intrinsics), n), "ssd_gpu_process_depth_host")
        return n

    def process_depth_host_ptr(self, ptr, intrinsics, n_frames):
        self._ck(self._l.ssd_gpu_process_depth_host(self._h, ptr, C.byref(intrinsics), n_frames), "ssd_gpu_process_depth_host")

    def process_depth_device(self, dev_ptr, intrinsics, n_frames):
        self._ck(self._l.ssd_gpu_process_depth_device(self._h, dev_ptr, C.byref(intrinsics), n_frames), "ssd_gpu_process_depth_device")

    def deproject_device(self, depth_dev, intrinsics, n_frames, xyz_dev):
        self._ck(self._l.ssd_gpu_deproject_device(self._h, depth_dev, C.byref(intrinsics), n_frames, xyz_dev), "ssd_gpu_deproject_device")

    def process_device(self, dev_ptr, n_frames, flags=0):
        self._ck(self._l.ssd_gpu_process_device_ex(self._h, dev_ptr, n_frames, flags), "ssd_gpu_process_device")

    # ---- per-frame cameras ----
    def set_cameras(self, cameras, distortions=None):
        """Replace the camera table with a list of A.Camera (scene_camera / make_camera); an empty list frees it.
        distortions: one A.Distortion per camera (make_distortion / scene_distortion), or None for pin-hole lenses."""
        arr = (A.Camera * max(1, len(cameras)))(*cameras)
        if distortions is None:
            self._ck(self._l.ssd_gpu_set_cameras(self._h, arr, len(cameras)), "ssd_gpu_set_cameras")
            return
        if len(distortions) != len(cameras):
            raise ValueError(f"{len(distortions)} distortions for {len(cameras)} cameras")
        dist = (A.Distortion * max(1, len(distortions)))(*distortions)
        self._ck(self._l.ssd_gpu_set_cameras_ex(self._h, arr, dist, len(cameras)), "ssd_gpu_set_cameras_ex")

    def set_distortion(self, distortion):
        """Lens of the plain calls (depth input, deproject_device, overlay); None switches it off (pin-hole)."""
        self._ck(self._l.ssd_gpu_set_distortion(self._h, None if distortion is None else C.byref(distortion)), "ssd_gpu_set_distortion")

    @property
    def n_ray_tables(self):
        return self._l.ssd_gpu_n_ray_tables(self._h)

    @property
    def n_cameras(self):
        return self._l.ssd_gpu_n_cameras(self._h)

    @staticmethod
    def _cams(camera_of_frame, n):
        cams = np.ascontiguousarray(camera_of_frame, np.int32)
        if cams.size != n:
            raise ValueError(f"camera_of_frame has {cams.size} entries for {n} frames")
        return cams

    def process_cameras_host(self, xyz, camera_of_frame):
        """xyz as for process_host; camera_of_frame: camera table index of each frame."""
        xyz = np.ascontiguousarray(xyz, np.float32)
        n = xyz.size // (self.n_points * 3)
        cams = self._cams(camera_of_frame, n)
        self._ck(self._l.ssd_gpu_process_cameras_host(self._h, _ptr(xyz), _ptr(cams), n), "ssd_gpu_process_cameras_host")
        return n

    def process_cameras_device(self, dev_ptr, camera_of_frame, n_frames, flags=0):
        cams = self._cams(camera_of_frame, n_frames)
        self._ck(self._l.ssd_gpu_process_cameras_device_ex(self._h, dev_ptr, _ptr(cams), n_frames, flags), "ssd_gpu_process_cameras_device")

    def process_depth_cameras_host(self, depth, camera_of_frame):
        """depth as for process_depth_host; each frame is deprojected with its camera's intrinsics."""
        depth = np.ascontiguousarray(depth, np.uint16)
        n = depth.size // self.n_points
        cams = self._cams(camera_of_frame, n)
        self._ck(self._l.ssd_gpu_process_depth_cameras_host(self._h, _ptr(depth), _ptr(cams), n), "ssd_gpu_process_depth_cameras_host")
        return n

    def process_depth_cameras_device(self, dev_ptr, camera_of_frame, n_frames):
        cams = self._cams(camera_of_frame, n_frames)
        self._ck(self._l.ssd_gpu_process_depth_cameras_device(self._h, dev_ptr, _ptr(cams), n_frames), "ssd_gpu_process_depth_cameras_device")

    # ---- results ----
    def steps(self, frame):
        out = (Step * A.MAX_STEPS)()
        n = C.c_int()
        st = C.c_uint32()
        self._ck(self._l.ssd_gpu_get_steps(self._h, frame, out, A.MAX_STEPS, C.byref(n), C.byref(st)), "ssd_gpu_get_steps")
        return [(s.height, np.array([[s.quad[c][0], s.quad[c][1]] for c in range(4)])) for s in out[:n.value]], st.value

    def set_overlay(self, a_inv, intrinsics):
        """Enable drawStairStep's projection of the step corners into the camera image (pointcloud.cpp:583-597);
        a_inv None switches it off."""
        if a_inv is None:
            self._ck(self._l.ssd_gpu_set_overlay(self._h, None, None), "ssd_gpu_set_overlay")
            return
        arr = (C.c_double * 9)(*[float(v) for v in np.asarray(a_inv, np.float64).ravel()])
        self._ck(self._l.ssd_gpu_set_overlay(self._h, arr, C.byref(intrinsics)), "ssd_gpu_set_overlay")

    def overlay(self, frame):
        """(n_steps, 4, 2) float32 pixel coordinates, corner order of steps()."""
        out = (A.Overlay * A.MAX_STEPS)()
        n = C.c_int()
        self._ck(self._l.ssd_gpu_get_overlay(self._h, frame, out, A.MAX_STEPS, C.byref(n)), "ssd_gpu_get_overlay")
        return np.array([[[o.px[c][0], o.px[c][1]] for c in range(4)] for o in out[:n.value]], np.float32).reshape(n.value, 4, 2)

    def set_vertical_faces(self, enable=True):
        """Vertical faces (risers) from the remainder points (include/ssd_gpu.h: ssd_gpu_riser); one more pass over the points."""
        self._ck(self._l.ssd_gpu_set_vertical_faces(self._h, 1 if enable else 0), "ssd_gpu_set_vertical_faces")

    def vertical_faces(self, frame):
        """list of dicts, one per pair of consecutive plateaus (riser k joins plateau k and k + 1)"""
        out = (A.Riser * A.MAX_PLATEAUS)()
        n = C.c_int()
        self._ck(self._l.ssd_gpu_get_vertical_faces(self._h, frame, out, A.MAX_PLATEAUS, C.byref(n)), "ssd_gpu_get_vertical_faces")
        return [{f: getattr(r, f) for f, _ in A.Riser._fields_ if f != "pad"} for r in out[:n.value]]

    def n_steps_all(self, n_frames):
        out = np.empty(n_frames, np.int32)
        n = C.c_int()
        for f in range(n_frames):
            self._ck(self._l.ssd_gpu_get_steps(self._h, f, None, 0, C.byref(n), None), "ssd_gpu_get_steps")
            out[f] = n.value
        return out

    def frame_info(self, frame):
        info = FrameInfo()
        self._ck(self._l.ssd_gpu_get_frame_info(self._h, frame, C.byref(info)), "ssd_gpu_get_frame_info")
        return info

    def plateaus(self, frame):
        out = (Plateau * A.MAX_PLATEAUS)()
        n = C.c_int()
        self._ck(self._l.ssd_gpu_get_plateaus(self._h, frame, out, A.MAX_PLATEAUS, C.byref(n)), "ssd_gpu_get_plateaus")
        return out, n.value

    def labels(self, frame):
        out = np.empty(self.n_points, np.uint8)
        self._ck(self._l.ssd_gpu_get_labels(self._h, frame, _ptr(out)), "ssd_gpu_get_labels")
        return out

    def histogram(self, frame):
        out = np.zeros(A.MAX_BINS, np.uint32)
        n = C.c_int()
        self._ck(self._l.ssd_gpu_get_histogram(self._h, frame, out.ctypes.data_as(C.POINTER(C.c_uint32)), A.MAX_BINS, C.byref(n)),
                 "ssd_gpu_get_histogram")
        return out[:n.value]

    def timing(self):
        t = Timing()
        self._ck(self._l.ssd_gpu_get_timing(self._h, C.byref(t)), "ssd_gpu_get_timing")
        return t

    def stats(self):
        st = A.Stats()
        self._ck(self._l.ssd_gpu_get_stats(self._h, C.byref(st)), "ssd_gpu_get_stats")
        return st

    def stage_times(self):
        """{stage: (sum of launch durations in ms, launches)} of the last call made with FLAG_STAGE_TIMING."""
        ms = (C.c_float * A.N_STAGES)()
        n = (C.c_int * A.N_STAGES)()
        self._ck(self._l.ssd_gpu_get_stage_times(self._h, ms, n), "ssd_gpu_get_stage_times")
        return {self._l.ssd_gpu_stage_name(i).decode(): (ms[i], n[i]) for i in range(A.N_STAGES)}

    @property
    def chunk_frames(self):
        return self._l.ssd_gpu_chunk_frames(self._h)

    def line(self, frame):
        """The result line the reference prints for this frame (pointcloud.cpp:625)."""
        s, _ = self.steps(frame)
        return serialize(s)

    # ---- single-stage entry points ----
    def detect_outline(self, image, min_img_y_extent, xy_ratio):
        image = np.ascontiguousarray(image, np.uint8)
        q = (C.c_double * 8)()
        v = C.c_int()
        self._ck(self._l.ssd_gpu_detect_outline(self._h, _ptr(image), min_img_y_extent, xy_ratio, q, C.byref(v)), "ssd_gpu_detect_outline")
        return np.array(q[:]).reshape(4, 2), v.value

    def detect_front_edge(self, image):
        image = np.ascontiguousarray(image, np.uint8)
        l = (C.c_double * 2)()
        r = (C.c_double * 2)()
        v = C.c_int()
        self._ck(self._l.ssd_gpu_detect_front_edge(self._h, _ptr(image), l, r, C.byref(v)), "ssd_gpu_detect_front_edge")
        return np.array(l[:]), np.array(r[:]), v.value

    def points_in_quad(self, quad, xy):
        xy = np.ascontiguousarray(xy, np.float64)
        n = xy.size // 2
        q = (C.c_double * 8)(*np.asarray(quad, np.float64).ravel())
        inside = np.empty(n, np.uint8)
        st = C.c_int()
        self._ck(self._l.ssd_gpu_points_in_quad(self._h, q, _ptr(xy), n, _ptr(inside), C.byref(st)), "ssd_gpu_points_in_quad")
        return inside, st.value

    def camera_to_world(self, xyz):
        xyz = np.ascontiguousarray(xyz, np.float32)
        n = xyz.size // 3
        out = np.empty((n, 3), np.float64)
        self._ck(self._l.ssd_gpu_camera_to_world(self._h, _ptr(xyz), n, _ptr(out)), "ssd_gpu_camera_to_world")
        return out

    # ---- device memory + synthetic frames ----
    def malloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self._l.ssd_gpu_malloc(self._h, nbytes, C.byref(p)), "ssd_gpu_malloc")
        return p

    def free(self, p):
        self._ck(self._l.ssd_gpu_free(self._h, p), "ssd_gpu_free")

    def h2d(self, dst, src):
        src = np.ascontiguousarray(src)
        self._ck(self._l.ssd_gpu_memcpy_h2d(self._h, dst, _ptr(src), src.nbytes), "ssd_gpu_memcpy_h2d")

    def d2h(self, dst, src, nbytes=None):
        self._ck(self._l.ssd_gpu_memcpy_d2h(self._h, _ptr(dst), src, dst.nbytes if nbytes is None else nbytes), "ssd_gpu_memcpy_d2h")

    def synth_frames(self, base_scene, base_seed, first_index, n_frames, min_steps, max_steps, xyz_dev, depth_dev=None):
        """fill device buffers of this context's GPU with synthetic frames (libssd_scene.so: input source, not the product)"""
        rc = scene_lib().ssd_scene_synth_frames_device(self.device, C.byref(base_scene), base_seed, first_index, n_frames, min_steps, max_steps,
                                                       xyz_dev, depth_dev)
        if rc != A.OK:
            raise SsdError(f"ssd_scene_synth_frames_device failed ({rc})")


def pinned_empty(shape, dtype):
    """numpy array over pinned host memory (cudaMallocHost); keep the returned handle alive."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    rc = lib().ssd_gpu_malloc_host(n, C.byref(p))
    if rc:
        raise SsdError("ssd_gpu_malloc_host failed")
    buf = (C.c_char * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    return arr, p


def register_host(array):
    """Page-lock a numpy array the caller owns (ssd_gpu_register_host); pair with unregister_host(array)."""
    rc = lib().ssd_gpu_register_host(_ptr(array), array.nbytes)
    if rc != 0:
        raise SsdError(f"ssd_gpu_register_host failed ({rc})")


def unregister_host(array):
    rc = lib().ssd_gpu_unregister_host(_ptr(array))
    if rc != 0:
        raise SsdError(f"ssd_gpu_unregister_host failed ({rc})")


def free_pinned(p):
    lib().ssd_gpu_free_host(p)
