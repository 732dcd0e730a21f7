"""Generate tests/golden/reference_runs.json: the reference's results for the seeded inputs of the tests that compare the
oracle with the compiled reference (tests/test_oracle_vs_ref.py, test_calibration.py::test_random_files_against_the_compiled_reference,
test_vertical_faces.py::test_risers_from_the_reference_labels). Those tests read this file when the reference is not available.

    SSD_REFERENCE_DIR=<checkout of the original project> python tests/golden/make_reference_runs.py

With the reference available the results come from it. `--from-oracle` writes them from the oracle instead (and, for the
calibration files, the product's loader); that is only valid for code at which these tests have passed live against the
compiled reference, because each of them asserts that the two agree: labels, histograms, counts, statuses, pixel bits,
outline / front-edge / calibration doubles bit for bit, step and plateau coordinates within 1e-12 m. The file says which.
"""
import ctypes as C
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(TESTS))
import helpers as H  # noqa: E402
import stair_step_detector_b200 as S  # noqa: E402
import test_calibration as TC  # noqa: E402
import test_oracle_vs_ref as R  # noqa: E402
import test_vertical_faces as TV  # noqa: E402
from stair_step_detector_b200 import _abi as A  # noqa: E402


class OracleSource:
    """the oracle's side, in the form RefSource gives the reference's"""

    def __init__(self):
        self.o = H.load_oracle()

    def frame(self, cfg, xf, xyz):
        return H.oracle_process(self.o, cfg, xf, xyz)

    def overlay(self, cfg, xf, xyz, intr):
        w, h = cfg.width, cfg.height
        r = H.oracle_process(self.o, cfg, xf, xyz)
        a_inv = np.empty(9)
        assert self.o.ssd_oracle_inverse3(xf.a, a_inv.ctypes.data_as(C.POINTER(C.c_double))) == 0
        ov = H.oracle_overlay(self.o, xf, a_inv, intr if intr is not None else A.Intrinsics(fx=w, fy=w, ppx=w * 0.5, ppy=h * 0.5))
        px = np.concatenate([ov, ov])  # drawStairStep draws every step twice (depth and infrared viewport)
        return dict(a_inv=[H.hexf(v) for v in a_inv], n_steps=r.info["n_steps"], n_calls=len(px), px_bits=[int(v) for v in px.view(np.uint32).ravel()])

    def derived(self, cfg, px):
        d = H.Derived()
        assert self.o.ssd_oracle_derive(C.byref(cfg), C.byref(d)) == 0
        out = np.stack([cfg.x_min + px[:, 0] * d.x_to_world, cfg.y_max - px[:, 1] * d.y_to_world], 1)
        return dict(min_height=d.min_height, min_img_y_extent=d.min_img_y_extent, n_bins=d.n_bins, xy_ratio=H.hexf(d.xy_ratio),
                    height_interval_reciprocal=H.hexf(d.height_interval_reciprocal), image_to_world_sha256=H.digest(out))

    def outline(self, img, w, h):
        q, l, r = (C.c_double * 8)(), (C.c_double * 2)(), (C.c_double * 2)()
        v, fv = C.c_int(), C.c_int()
        assert self.o.ssd_oracle_detect_outline(H.ptr(img), w, h, 20, 4 / 3, q, C.byref(v)) == 0
        assert self.o.ssd_oracle_detect_front_edge(H.ptr(img), w, h, l, r, C.byref(fv)) == 0
        return dict(valid=v.value, quad=[H.hexf(x) for x in q], front_valid=fv.value, left=[H.hexf(x) for x in l], right=[H.hexf(x) for x in r])

    def points_in_quad(self, q, xy):
        inside, st = np.empty(len(xy), np.uint8), C.c_int()
        self.o.ssd_oracle_points_in_quad((C.c_double * 8)(*q.ravel()), H.ptr(xy), len(xy), H.ptr(inside), C.byref(st))
        return dict(status=st.value, inside_sha256=H.digest(inside))

    def calibration(self, d):
        xf, status, _, _ = S.load_calibration(d)
        assert status == 0
        return xf


def main():
    from_oracle = "--from-oracle" in sys.argv
    if from_oracle:
        src = OracleSource()
        note = ("written by the oracle (oracle/ssd_oracle.c) and, for the calibration files, the product's loader, with the oracle, "
                "the scene generator and these tests as at commit 1360c0b, where every one of these tests ran live against the compiled "
                "reference and passed: the values are the reference's, exactly where the tests compare exactly, and within 1e-12 m "
                "for step and plateau coordinates and mean heights")
    else:
        assert H.ref_available(), "needs SSD_REFERENCE_DIR (the original project's sources), or --from-oracle"
        src = R.RefSource(S)
        note = "written by the compiled reference (oracle/_ref, the original project's translation units compiled by path)"
    runs = {}
    for w, h, n in ((320, 240, 10), (640, 480, 6), (1024, 768, 3)):
        runs[f"frames_random_scenes/{w}x{h}"] = [H.frame_record(src.frame(cfg, xf, xyz), ~R.QUIRKS & 0xffffffff)
                                                 for cfg, xf, xyz in R.frames_random_scenes_inputs(S, w, h, n)]
    for w, h, ck, sk, n in R.HIRES_CASES:
        runs[f"frames_hires/{w}x{h}"] = [H.frame_record(src.frame(cfg, xf, xyz), ~R.QUIRKS & 0xffffffff)
                                         for cfg, xf, xyz in R.frames_hires_inputs(S, w, h, ck, sk, n)]
    for w, h, n in ((320, 240, 6), (640, 480, 4), (1024, 768, 2)):
        runs[f"overlay_projection/{w}x{h}"] = [src.overlay(cfg, xf, xyz, intr) for cfg, xf, xyz, intr in R.overlay_inputs(S, w, h, n)]
    for w, h in ((320, 240), (640, 480), (1024, 768)):
        runs[f"derived_constants/{w}x{h}"] = src.derived(S.default_config(w, h), R.derived_px(w))
    runs["outline_front_edge_fuzz"] = [src.outline(img, 320, 240) for img in R.outline_inputs(320, 240)]
    runs["points_in_quad_fuzz"] = [src.points_in_quad(q, xy) for q, xy in R.points_in_quad_inputs()]
    with tempfile.TemporaryDirectory() as tmp:
        import pathlib
        load = src.calibration if from_oracle else __import__("make_calibration_golden").reference_load
        runs["calibration_random_files"] = [{k: [H.hexf(x) for x in np.atleast_1d(v)] if k != "ext_z" else H.hexf(v[0])
                                             for k, v in TC.as_dict(load(d)).items()}
                                            for d in TC.random_calibration_files(S, pathlib.Path(tmp))]
    runs["risers_from_the_reference_labels"] = [TV.reference_bands(src.frame(cfg, xf, xyz)) for cfg, xf, xyz in TV.riser_inputs(S)]
    out = os.path.join(HERE, "reference_runs.json")
    with open(out, "w") as f:
        json.dump(dict(source=note, runs=runs), f, separators=(",", ":"))
        f.write("\n")
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
