"""Generate tests/golden/overlay.json from the REFERENCE ITSELF (oracle/_ref, the reference's translation units
compiled by path): for every golden case (*.npz, make_golden.py) the quadrilaterals drawStairStep
(pointcloud.cpp:583-597) hands to drawQuadrilateral, as recorded by the harness' stub. Run in the build container:

    python tests/golden/make_overlay_golden.py

Stored per case: the depth-stream intrinsics the stub frame reported, the reference's _aInv (inverse(_a), as the harness
sets it), and the projected pixels as the uint32 bit patterns of the f32 values (depth-viewport pass; the infrared
pass is checked equal here).
"""
import ctypes as C
import glob
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import helpers as H  # noqa: E402
import stair_step_detector_b200 as S  # noqa: E402
from test_oracle_golden import load_case  # noqa: E402


def main():
    assert H.ref_available(), "needs SSD_REFERENCE_DIR (the original project's sources)"
    out = {}
    for i, path in enumerate(sorted(glob.glob(os.path.join(HERE, "*.npz")))):
        z, meta, sc, xf = load_case(path)
        w, h = meta["width"], meta["height"]
        cfg = S.default_config(w, h)
        ref = H.load_ref(cfg)
        # alternate between the scene's own intrinsics and an off-centre set
        intr = S.scene_intrinsics(sc)
        if i % 2:
            intr.fx, intr.fy, intr.ppx, intr.ppy = w * 0.93, w * 0.95, w * 0.5 + 3.25, h * 0.5 - 2.5
        ref.ssd_ref_set_intrinsics(C.byref(intr))
        try:
            r = H.ref_process(ref, cfg, xf, H.deproject_np(sc, z["depth"]))
            px, _, _ = H.ref_overlay(ref)
        finally:
            ref.ssd_ref_set_intrinsics(None)
        ns = r.info["n_steps"]
        assert len(px) == 2 * ns and np.array_equal(px[:ns].view(np.uint32), px[ns:].view(np.uint32))
        out[meta["name"]] = dict(intrinsics=[intr.fx, intr.fy, intr.ppx, intr.ppy], a_inv=H.ref_a_inv(ref, xf).tolist(),
                                 px_bits=px[:ns].view(np.uint32).reshape(ns, 8).tolist(), px=px[:ns].reshape(ns, 8).tolist())
        print(meta["name"], ns, "steps")
    with open(os.path.join(HERE, "overlay.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
