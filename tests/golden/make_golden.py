"""Generate the golden vectors in tests/golden/ from the REFERENCE ITSELF (oracle/_ref: the reference's
translation units compiled by path, see oracle/Makefile). Run with SSD_REFERENCE_DIR set to the original project's sources:

    python tests/golden/make_golden.py

Each case stores the synthetic z16 depth image (the input; vertices are re-derived with single f32 operations,
helpers.deproject_np), the calibration points, and what the reference computed for it: per-pixel segment labels,
height histogram, plateau records, Stairs and the serialized line. The fixtures are small (320x240 / 640x480).
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

NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)

CASES = [
    # name, (w,h), scene overrides, randomize index or None
    ("clean3_320", (320, 240), dict(), None),
    ("noisy3_320", (320, 240), dict(**NOISY), None),
    ("clean3_640", (640, 480), dict(), None),
    ("noisy_rand5_640", (640, 480), dict(**NOISY), 5),
    ("descending_occluded_640", (640, 480), dict(rotate180=1, n_occluders=2, **NOISY), 3),
    ("yawed_rolled_320", (320, 240), dict(cam_yaw_deg=6.0, cam_roll_deg=-3.0, **NOISY), None),
    ("low_camera_no_steps_320", (320, 240), dict(n_steps=0, **NOISY), None),
]


def scene_fields(sc):
    return {f: getattr(sc, f) for f, _ in A.Scene._fields_}


def main():
    assert H.ref_available(), "needs SSD_REFERENCE_DIR (the original project's sources)"
    for name, (w, h), kw, ridx in CASES:
        cfg = S.default_config(w, h)
        ref = H.load_ref(cfg)
        sc = S.default_scene(w, h, **kw)
        if ridx is not None:
            sc = S.randomize_scene(sc, 2026, ridx, 3, 8)
        world = (C.c_double * 9)()
        cam = (C.c_double * 9)()
        S.lib().ssd_scene_calibration_points(C.byref(sc), world, cam)
        xf = A.Transform()
        assert ref.ssd_ref_make_transform(world, cam, C.byref(xf)) == 0
        depth = S.synth_depth_host(sc)
        xyz = H.deproject_np(sc, depth)
        r = H.ref_process(ref, cfg, xf, xyz)
        meta = dict(name=name, width=w, height=h, scene=scene_fields(sc), world_pts=list(world), camera_pts=list(cam),
                    transform=dict(a=list(xf.a), b=list(xf.b), ext_a=list(xf.ext_a), ext_b=list(xf.ext_b), ext_z=xf.ext_z),
                    info=r.info, line=r.line,
                    plateaus=[{k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in p.items()} for p in r.plateaus],
                    steps=[dict(height=s["height"], quad=s["quad"].tolist()) for s in r.steps])
        np.savez_compressed(os.path.join(HERE, name + ".npz"), depth=depth, labels=r.labels.reshape(h, w), hist=r.hist,
                            meta=json.dumps(meta))
        print(name, r.info["n_steps"], "steps", os.path.getsize(os.path.join(HERE, name + ".npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
