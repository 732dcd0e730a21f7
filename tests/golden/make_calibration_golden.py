"""Generate tests/golden/calibration/ -- a pair of calibration text files in the reference's own formats
(calibrationTriangle.cpp:127-146 save(), geometricCalibration.cpp:43-71 savePoints()) and the transformation the
REFERENCE's GeometricCalibration::load() builds from them (oracle/_ref, reference TUs compiled by path).
Run with SSD_REFERENCE_DIR set to the original project's sources:   python tests/golden/make_calibration_golden.py
"""
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import helpers as H  # noqa: E402
import stair_step_detector_b200 as S  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402

OUT = os.path.join(HERE, "calibration")


def write_files(directory, world, samples, lower="right"):
    """world: 3x3 external-world corners; samples: (10, 3, 3) float camera coordinates of the marks."""
    with open(os.path.join(directory, "calibration-triangle"), "w") as f:
        f.write("calibration triangle\n")
        for n, c in enumerate(world, 1):
            f.write(f"x{n} = {c[0]:g}, y{n} = {c[1]:g}, z{n} = {c[2]:g}\n")
        f.write(f"lowerQuadrant = {lower}\n")
    with open(os.path.join(directory, "calibration-points"), "w") as f:
        f.write("calibration points\n")
        for row in samples:
            f.write("; ".join(f"{p[0]:9.6f}, {p[1]:9.6f}, {p[2]:8.6f}" for p in row) + "\n")


def reference_load(directory):
    ref = H.load_ref(S.default_config(320, 240))
    xf = A.Transform()
    cwd = os.getcwd()
    os.chdir(directory)
    try:
        rc = ref.ssd_ref_load_calibration(C.byref(xf))
    finally:
        os.chdir(cwd)
    assert rc == 0, rc
    return xf


def xf_dict(xf):
    return dict(a=list(xf.a), b=list(xf.b), ext_a=list(xf.ext_a), ext_b=list(xf.ext_b), ext_z=xf.ext_z)


def main():
    assert H.ref_available(), "needs SSD_REFERENCE_DIR (the original project's sources)"
    os.makedirs(OUT, exist_ok=True)
    # a camera 1.3 m above the floor looking 48 degrees down sees the three marks of a 2.2 m wide triangle
    sc = S.default_scene(640, 480, cam_height=1.3, cam_pitch_deg=48.0)
    world = (C.c_double * 9)()
    cam = (C.c_double * 9)()
    S.lib().ssd_scene_calibration_points(C.byref(sc), world, cam)
    world = np.array(world).reshape(3, 3) + np.array([0.0, 0.0, 0.004])
    cam = np.array(cam).reshape(3, 3)
    rng = np.random.default_rng(20261017)
    samples = (cam[None] + rng.normal(0, 0.002, (10, 3, 3))).astype(np.float32)
    write_files(OUT, world, samples)
    xf = reference_load(OUT)
    with open(os.path.join(OUT, "expected.json"), "w") as f:
        json.dump(dict(transform=xf_dict(xf), note="GeometricCalibration::load() of the compiled reference on the two files here"), f, indent=1)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
