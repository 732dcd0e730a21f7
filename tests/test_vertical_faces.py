"""Vertical faces (risers) from the remainder: SURVEY.md 8(f) row 4, second half. The reference collects the remainder and leaves
"TODO use remainder to detect vertical faces" (pointcloud.cpp:283-293): there is no reference behaviour, so the checker is the
oracle's restatement of the DEFINITION in include/ssd_gpu.h (ssd_gpu_riser) -- parity for this row is unpinned by construction --
cross-checked here against an independent numpy evaluation and against the compiled reference's own label / band output
(live where the compiled reference is available, else its stored output, tests/golden/reference_runs.json)."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
from stair_step_detector_b200 import _abi as A

NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
FIELDS = ("lower_plateau", "upper_plateau", "n_points", "x_min", "x_max", "y_min", "y_max", "x_mean", "y_mean", "z_bottom", "z_top")


def numpy_risers(oracle, cfg, xf, xyz, labels, plats):
    """the definition once more, vectorised: exact double CameraToWorld by the oracle, everything else numpy"""
    N = cfg.width * cfg.height
    w = np.empty((N, 3), np.float64)
    assert oracle.ssd_oracle_camera_to_world(C.byref(xf), H.ptr(np.ascontiguousarray(xyz, np.float32)), N, H.ptr(w)) == 0
    rem = labels == A.LABEL_REMAINDER if hasattr(A, "LABEL_REMAINDER") else labels == 253
    h = ((w[:, 2] - cfg.z_min) * (1.0 / cfg.height_interval)).astype(np.int64) & 0xffff
    out = []
    for k in range(len(plats) - 1):
        m = rem & (h > plats[k]["hmax"]) & (h < plats[k + 1]["hmin"])
        X = ((w[m, 0] - cfg.x_min) * 65536.0).astype(np.int64)
        Y = ((w[m, 1] - cfg.y_min) * 65536.0).astype(np.int64)
        r = dict(lower_plateau=k, upper_plateau=k + 1, n_points=int(m.sum()), x_min=0.0, x_max=0.0, y_min=0.0, y_max=0.0, x_mean=0.0, y_mean=0.0,
                 z_bottom=cfg.z_min + float(plats[k]["hmax"] + 1) * cfg.height_interval, z_top=cfg.z_min + float(plats[k + 1]["hmin"]) * cfg.height_interval)
        if r["n_points"]:
            r.update(x_min=cfg.x_min + float(X.min()) / 65536.0, x_max=cfg.x_min + float(X.max()) / 65536.0,
                     y_min=cfg.y_min + float(Y.min()) / 65536.0, y_max=cfg.y_min + float(Y.max()) / 65536.0,
                     x_mean=cfg.x_min + float(int(X.sum())) / float(r["n_points"]) / 65536.0,
                     y_mean=cfg.y_min + float(int(Y.sum())) / float(r["n_points"]) / 65536.0)
        out.append(r)
    return out


def same(a, b):
    return len(a) == len(b) and all(x[f] == y[f] for x, y in zip(a, b) for f in FIELDS)


@pytest.mark.parametrize("w,h", [(320, 240), (640, 480), (1024, 768)])
def test_oracle_risers_match_the_definition(S, oracle, w, h):
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    xf = S.scene_transform(base)
    seen = 0
    for i in range(3):
        sc = S.randomize_scene(base, 4100 + w, i, 3, 8)
        xyz = S.deproject_host(sc, S.synth_depth_host(sc)).reshape(-1, 3)
        o = H.oracle_process(oracle, cfg, xf, xyz)
        got = H.oracle_vertical_faces(oracle, cfg, xf, xyz)
        want = numpy_risers(oracle, cfg, xf, xyz, o.labels, o.plateaus)
        assert same(got, want), (got, want)
        assert len(got) == max(0, o.info["n_plateaus"] - 1)
        seen += sum(r["n_points"] for r in got)
        # every riser of a staircase seen from the front lies between the two treads it joins: behind the lower step's front
        # edge, not beyond the upper step's back edge (steps valid only)
        for r in got:
            lo, up = o.plateaus[r["lower_plateau"]], o.plateaus[r["upper_plateau"]]
            if r["n_points"] > 500 and lo["valid"] and up["valid"]:
                assert lo["quad_world"][:, 1].min() - 0.05 < r["y_mean"] < up["quad_world"][:, 1].max() + 0.05
    assert seen > 0


def riser_inputs(S):
    cfg = S.default_config(640, 480)
    base = S.default_scene(640, 480, **NOISY)
    xf = S.scene_transform(base)
    for i in range(3):
        sc = S.randomize_scene(base, 4200, i, 3, 8)
        yield cfg, xf, S.deproject_host(sc, S.synth_depth_host(sc)).reshape(-1, 3)


def reference_bands(r):
    """what the riser definition takes from a frame: the labels (as a digest) and the plateaus' height bands"""
    return dict(labels_sha256=H.digest(r.labels), bands=[[int(p["hmin"]), int(p["hmax"])] for p in r.plateaus])


def test_risers_from_the_reference_labels(S, oracle):
    """the compiled reference's remainder (its labels) and bands give the same risers as the oracle's: live, the risers from
    the reference's labels and bands are computed; from the stored output, its labels and bands must equal the oracle's"""
    import test_oracle_vs_ref as R
    ref = H.load_ref(S.default_config(640, 480))
    want = None if ref is not None else R.stored("risers_from_the_reference_labels")
    for i, (cfg, xf, xyz) in enumerate(riser_inputs(S)):
        mine = H.oracle_vertical_faces(oracle, cfg, xf, xyz)
        if ref is not None:
            r = H.ref_process(ref, cfg, xf, xyz)
            assert same(mine, H.oracle_vertical_faces(oracle, cfg, xf, xyz, r.labels, r.plateaus))
            continue
        o = H.oracle_process(oracle, cfg, xf, xyz)
        assert reference_bands(o) == want[i], i
        assert same(mine, H.oracle_vertical_faces(oracle, cfg, xf, xyz, o.labels, o.plateaus))


def test_no_riser_without_two_plateaus(S, oracle):
    cfg = S.default_config(320, 240)
    xf = S.scene_transform(S.default_scene(320, 240))
    xyz = np.zeros((320 * 240, 3), np.float32)  # every vertex invalid
    assert H.oracle_vertical_faces(oracle, cfg, xf, xyz) == []


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n", [(320, 240, 4), (640, 480, 6), (1024, 768, 6)])
def test_gpu_risers_equal_the_oracle(S, oracle, w, h, n):
    """k_riser_reduce through the C ABI: every field of every riser equal to the oracle's (integer extremes and sums of exact
    double coordinates: nothing to tolerate); vertex input and fused depth input; the steps are what they are without it"""
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, rotate180=int(w == 640), n_occluders=2 if w == 640 else 0, **NOISY)
    xf = S.scene_transform(base)
    intr = S.scene_intrinsics(base)
    scenes = [S.randomize_scene(base, 4300 + w, i, 0 if i == 1 else 3, 8) for i in range(n)]
    depth = np.stack([S.synth_depth_host(sc) for sc in scenes])
    xyz = np.stack([S.deproject_host(sc, d) for sc, d in zip(scenes, depth)])
    with S.Detector(cfg, xf, max_frames=n) as det:
        det.process_host(xyz)
        plain = [det.steps(f) for f in range(n)]
        with pytest.raises(S.SsdError, match="not enabled"):
            det.vertical_faces(0)
        det.set_vertical_faces(True)
        with pytest.raises(S.SsdError):
            det.vertical_faces(0)  # results of the earlier call carry no risers
        for run in ("vertices", "depth"):
            if run == "vertices":
                det.process_host(xyz)
            else:
                det.process_depth_host(depth, intr)
            total = 0
            for f in range(n):
                want = H.oracle_vertical_faces(oracle, cfg, xf, xyz[f].reshape(-1, 3))
                got = det.vertical_faces(f)
                assert same(got, want), (run, f, got, want)
                total += sum(r["n_points"] for r in got)
                s0, s1 = plain[f], det.steps(f)
                assert s0[1] == s1[1] and len(s0[0]) == len(s1[0])
                for (ha, qa), (hb, qb) in zip(s0[0], s1[0]):
                    assert (ha == hb or (np.isnan(ha) and np.isnan(hb))) and np.array_equal(qa, qb)
            assert total > 0
        det.set_vertical_faces(False)
        det.process_host(xyz)
        with pytest.raises(S.SsdError, match="not enabled"):
            det.vertical_faces(0)
