"""ctypes mirror of include/ssd_gpu.h (struct layouts, constants, prototypes).

The shared library is built in-tree by ``build.py`` / ``__graft_entry__.build()`` and loaded from
``stair_step_detector_b200/lib/libssd_gpu.so``. There is no Python or CPU fallback: if the library is
missing, importing the package raises.
"""
import ctypes as C
import os

MAX_BINS = 253
MAX_PLATEAUS = 32
MAX_STEPS = 32
MAX_GROUP_FRAMES = 32  # members of one frame group (ssd_gpu_process_groups_*)
LABEL_REMAINDER = 253
LABEL_OUT_OF_RANGE = 254
LABEL_INVALID = 255
STEP_LABEL_NONE = 255  # step labels: pixel on no step (ssd_gpu_set_step_labels)

OK = 0
E_INVALID_ARG, E_CUDA, E_NOMEM, E_RANGE, E_STATE = -1, -2, -3, -4, -5

STATUS_NO_STEPS = 0x1
STATUS_DEGENERATE_QUAD = 0x2
STATUS_INVALID_FRONT_EDGE = 0x4
STATUS_EMPTY_MEAN = 0x8
STATUS_TOO_MANY_PLATEAUS = 0x10
STATUS_BEV_OOB = 0x20
STATUS_HMIN_WRAP = 0x40

# lens models (rs2_distortion values); 1, 3 and 5 are rejected
DISTORTION_NONE = 0
DISTORTION_MODIFIED_BROWN_CONRADY = 1
DISTORTION_INVERSE_BROWN_CONRADY = 2
DISTORTION_FTHETA = 3
DISTORTION_BROWN_CONRADY = 4
DISTORTION_KANNALA_BRANDT4 = 5

FLAG_STAGE_TIMING = 0x2
FLAG_SINGLE_STREAM = 0x4
N_STAGES = 7


class Config(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32),
                ("x_min", C.c_double), ("x_max", C.c_double),
                ("y_min", C.c_double), ("y_max", C.c_double),
                ("z_min", C.c_double), ("z_max", C.c_double),
                ("height_interval", C.c_double), ("min_height_above_ground", C.c_double),
                ("min_step_depth", C.c_double),
                ("min_peak_points", C.c_uint32), ("reserved", C.c_uint32)]


class Transform(C.Structure):
    _fields_ = [("a", C.c_double * 9), ("b", C.c_double * 3),
                ("ext_a", C.c_double * 4), ("ext_b", C.c_double * 2), ("ext_z", C.c_double)]


class Intrinsics(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("ppx", C.c_float), ("ppy", C.c_float),
                ("depth_unit", C.c_float), ("reserved", C.c_int32 * 3)]


class Camera(C.Structure):
    """ssd_gpu_camera: one entry of a context's camera table (ssd_gpu_set_cameras)."""
    _fields_ = [("xf", Transform), ("a_inv", C.c_double * 9), ("intr", Intrinsics)]


class Distortion(C.Structure):
    """ssd_gpu_distortion: rs2_intrinsics.model and .coeffs [k1, k2, p1, p2, k3]."""
    _fields_ = [("model", C.c_int32), ("coeffs", C.c_float * 5)]


class Overlay(C.Structure):
    _fields_ = [("px", (C.c_float * 2) * 4)]


class Riser(C.Structure):
    _fields_ = [("lower_plateau", C.c_int32), ("upper_plateau", C.c_int32), ("n_points", C.c_uint32), ("pad", C.c_uint32),
                ("x_min", C.c_double), ("x_max", C.c_double), ("y_min", C.c_double), ("y_max", C.c_double),
                ("x_mean", C.c_double), ("y_mean", C.c_double), ("z_bottom", C.c_double), ("z_top", C.c_double)]


class StepSurface(C.Structure):
    _fields_ = [("n_points", C.c_uint32), ("fit_valid", C.c_int32), ("centroid", C.c_double * 3), ("gradient", C.c_double * 2),
                ("tilt_deg", C.c_double), ("rms_dz", C.c_double), ("z_lo", C.c_double), ("z_hi", C.c_double)]


class Step(C.Structure):
    _fields_ = [("height", C.c_double), ("quad", (C.c_double * 2) * 4)]


class Plateau(C.Structure):
    _fields_ = [("height", C.c_int32), ("hmin", C.c_int32), ("hmax", C.c_int32),
                ("n_points", C.c_uint32), ("valid", C.c_int32), ("outlined", C.c_int32),
                ("n_in_quad", C.c_uint32), ("quad_status", C.c_int32),
                ("quad_world", (C.c_double * 2) * 4), ("mean_z", C.c_double)]


class FrameInfo(C.Structure):
    _fields_ = [("status", C.c_uint32), ("n_bins", C.c_int32), ("n_plateaus", C.c_int32),
                ("ground_index", C.c_int32), ("first_valid_index", C.c_int32), ("n_steps", C.c_int32),
                ("n_nonzero", C.c_uint32), ("n_in_range", C.c_uint32)]


class Timing(C.Structure):
    _fields_ = [("total_ms", C.c_float), ("h2d_ms", C.c_float), ("reserved0", C.c_float),
                ("label_ms", C.c_float), ("n_launches", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_points", C.c_uint64), ("n_exact_fallback", C.c_uint64), ("n_quad_fast", C.c_uint64), ("n_quad_exact", C.c_uint64), ("filter_eps0", C.c_double), ("filter_eps1", C.c_double), ("n_bev_exact", C.c_uint64)]


class Scene(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32),
                ("fx", C.c_float), ("fy", C.c_float), ("ppx", C.c_float), ("ppy", C.c_float),
                ("depth_unit", C.c_float), ("cam_height", C.c_float), ("cam_pitch_deg", C.c_float),
                ("cam_roll_deg", C.c_float), ("cam_yaw_deg", C.c_float),
                ("cam_x", C.c_float), ("cam_y", C.c_float), ("ground_z", C.c_float),
                ("n_steps", C.c_int32), ("riser", C.c_float), ("tread", C.c_float), ("width_m", C.c_float),
                ("first_riser_y", C.c_float), ("x_center", C.c_float), ("top_landing", C.c_float),
                ("noise_sigma", C.c_float), ("dropout", C.c_float),
                ("n_holes", C.c_int32), ("n_occluders", C.c_int32), ("rotate180", C.c_int32), ("randomize_camera", C.c_int32),
                ("seed", C.c_uint64), ("distortion_model", C.c_int32), ("coeffs", C.c_float * 5)]


_P = C.POINTER
_vp = C.c_void_p

# name -> (restype, argtypes); every symbol include/ssd_gpu.h declares
PROTOTYPES = {
    "ssd_gpu_default_config": (None, [_P(Config), C.c_int32, C.c_int32]),
    "ssd_gpu_abi_version": (C.c_int, []),
    "ssd_gpu_device_count": (C.c_int, []),
    "ssd_gpu_create": (C.c_int, [_P(Config), _P(Transform), C.c_int, C.c_int, _P(_vp)]),
    "ssd_gpu_create_bev": (C.c_int, [_P(Config), C.c_int32, C.c_int32, _P(Transform), C.c_int, C.c_int, _P(_vp)]),
    "ssd_gpu_destroy": (None, [_vp]),
    "ssd_gpu_last_error": (C.c_char_p, [_vp]),
    "ssd_gpu_process_host": (C.c_int, [_vp, _vp, C.c_int]),
    "ssd_gpu_process_device": (C.c_int, [_vp, _vp, C.c_int]),
    "ssd_gpu_process_device_ex": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "ssd_gpu_set_cameras": (C.c_int, [_vp, _P(Camera), C.c_int]),
    "ssd_gpu_n_cameras": (C.c_int, [_vp]),
    "ssd_gpu_set_distortion": (C.c_int, [_vp, _P(Distortion)]),
    "ssd_gpu_set_cameras_ex": (C.c_int, [_vp, _P(Camera), _P(Distortion), C.c_int]),
    "ssd_gpu_n_ray_tables": (C.c_int, [_vp]),
    "ssd_gpu_process_cameras_host": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_cameras_device": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_cameras_device_ex": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int]),
    "ssd_gpu_process_depth_cameras_host": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_depth_cameras_device": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_groups_host": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_groups_device": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "ssd_gpu_process_depth_groups_host": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_depth_groups_device": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "ssd_gpu_process_depth_host": (C.c_int, [_vp, _vp, _P(Intrinsics), C.c_int]),
    "ssd_gpu_process_depth_device": (C.c_int, [_vp, _vp, _P(Intrinsics), C.c_int]),
    "ssd_gpu_process_depth_f32_host": (C.c_int, [_vp, _vp, _P(Intrinsics), C.c_int]),
    "ssd_gpu_process_depth_f32_device": (C.c_int, [_vp, _vp, _P(Intrinsics), C.c_int]),
    "ssd_gpu_process_depth_f32_cameras_host": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_depth_f32_cameras_device": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_depth_f32_groups_host": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int]),
    "ssd_gpu_process_depth_f32_groups_device": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "ssd_gpu_deproject_device": (C.c_int, [_vp, _vp, _P(Intrinsics), C.c_int, _vp]),
    "ssd_gpu_get_steps": (C.c_int, [_vp, C.c_int, _P(Step), C.c_int, _P(C.c_int), _P(C.c_uint32)]),
    "ssd_gpu_set_overlay": (C.c_int, [_vp, _P(C.c_double), _P(Intrinsics)]),
    "ssd_gpu_get_overlay": (C.c_int, [_vp, C.c_int, _P(Overlay), C.c_int, _P(C.c_int)]),
    "ssd_gpu_set_vertical_faces": (C.c_int, [_vp, C.c_int]),
    "ssd_gpu_get_vertical_faces": (C.c_int, [_vp, C.c_int, _P(Riser), C.c_int, _P(C.c_int)]),
    "ssd_gpu_set_step_labels": (C.c_int, [_vp, C.c_int]),
    "ssd_gpu_get_step_labels": (C.c_int, [_vp, C.c_int, _vp]),
    "ssd_gpu_step_labels_device_ptr": (C.c_int, [_vp, _P(_vp)]),
    "ssd_gpu_set_step_surfaces": (C.c_int, [_vp, C.c_int]),
    "ssd_gpu_get_step_surfaces": (C.c_int, [_vp, C.c_int, _P(StepSurface), C.c_int, _P(C.c_int)]),
    "ssd_gpu_get_frame_info": (C.c_int, [_vp, C.c_int, _P(FrameInfo)]),
    "ssd_gpu_get_plateaus": (C.c_int, [_vp, C.c_int, _P(Plateau), C.c_int, _P(C.c_int)]),
    "ssd_gpu_get_labels": (C.c_int, [_vp, C.c_int, _vp]),
    "ssd_gpu_get_histogram": (C.c_int, [_vp, C.c_int, _P(C.c_uint32), C.c_int, _P(C.c_int)]),
    "ssd_gpu_get_timing": (C.c_int, [_vp, _P(Timing)]),
    "ssd_gpu_get_stats": (C.c_int, [_vp, _P(Stats)]),
    "ssd_gpu_get_stage_times": (C.c_int, [_vp, _P(C.c_float), _P(C.c_int)]),
    "ssd_gpu_stage_name": (C.c_char_p, [C.c_int]),
    "ssd_gpu_chunk_frames": (C.c_int, [_vp]),
    "ssd_gpu_labels_device_ptr": (C.c_int, [_vp, _P(_vp)]),
    "ssd_stairs_serialize": (C.c_int, [_P(Step), C.c_int, C.c_char_p, C.c_size_t]),
    "ssd_gpu_detect_outline": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _P(C.c_double), _P(C.c_int)]),
    "ssd_gpu_detect_front_edge": (C.c_int, [_vp, _vp, _P(C.c_double), _P(C.c_double), _P(C.c_int)]),
    "ssd_gpu_points_in_quad": (C.c_int, [_vp, _P(C.c_double), _vp, C.c_int, _vp, _P(C.c_int)]),
    "ssd_gpu_camera_to_world": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "ssd_make_transform": (C.c_int, [_P(C.c_double), _P(C.c_double), _P(Transform)]),
    "ssd_make_transform_ex": (C.c_int, [_P(C.c_double), _P(C.c_double), _P(Transform), _P(C.c_double)]),
    "ssd_inverse3": (C.c_int, [_P(C.c_double), _P(C.c_double)]),
    "ssd_gpu_malloc": (C.c_int, [_vp, C.c_size_t, _P(_vp)]),
    "ssd_gpu_free": (C.c_int, [_vp, _vp]),
    "ssd_gpu_memcpy_h2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "ssd_gpu_memcpy_d2h": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "ssd_load_calibration": (C.c_int, [C.c_char_p, _P(Transform), _P(C.c_double), _P(C.c_double)]),
    "ssd_gpu_malloc_host": (C.c_int, [C.c_size_t, _P(_vp)]),
    "ssd_gpu_free_host": (C.c_int, [_vp]),
    "ssd_gpu_register_host": (C.c_int, [_vp, C.c_size_t]),
    "ssd_gpu_unregister_host": (C.c_int, [_vp]),
}

# every symbol include/ssd_scene.h declares (libssd_scene.so: the synthetic input source, not part of the product)
SCENE_PROTOTYPES = {
    "ssd_scene_default": (None, [_P(Scene), C.c_int32, C.c_int32]),
    "ssd_scene_randomize": (None, [_P(Scene), _P(Scene), C.c_uint64, C.c_int64, C.c_int, C.c_int]),
    "ssd_scene_calibration_points": (None, [_P(Scene), _P(C.c_double), _P(C.c_double)]),
    "ssd_scene_intrinsics": (None, [_P(Scene), _P(Intrinsics)]),
    "ssd_synth_depth_host": (C.c_int, [_P(Scene), _vp]),
    "ssd_deproject_host": (C.c_int, [_P(Scene), _vp, _vp]),
    "ssd_scene_synth_frames_device": (C.c_int, [C.c_int, _P(Scene), C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp]),
}
SCENE_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libssd_scene.so")

# SSD_GPU_LIB: developer override (A/B builds of the same library on the GPU box); never a different implementation
LIB_PATH = os.environ.get("SSD_GPU_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libssd_gpu.so")


def bind(lib, prototypes=PROTOTYPES):
    for name, (res, args) in prototypes.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib


def load_scene(path=SCENE_LIB_PATH):
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build first (python -c 'import __graft_entry__ as g; g.build()')")
    return bind(C.CDLL(path), SCENE_PROTOTYPES)


def load(path=LIB_PATH):
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
            "There is no CPU fallback.")
    return bind(C.CDLL(path))
