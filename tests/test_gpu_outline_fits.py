"""The outline and front-edge line fits on the GPU (k_outline, k_single_front_edge, k_finalize) against the oracle on the designed
lists of tests/outline_frames.py: hypot-dependent ties, exact ties between mirror lines in the residual branches of both frame-size
classes, front-edge lists up to the hi-res bisection, the decisions around the fit, and every construction under three settings of
SSD_GPU_OUTLINE_SMEM_KB (unset, 0: all global memory, 227: the largest band; outline_frames.band_path and
test_outline_fits.test_band_paths state which band path each size takes). The full chain runs on scene frames under
SSD_GPU_OUTLINE_SMEM_KB=0 and SSD_GPU_OUTLINE_GRIDX=1 / 32, fused and seven-launch. valid is compared exactly, coordinates to
1e-7 px (as test_gpu_parity.py)."""
import numpy as np
import pytest

import helpers as H
import outline_frames as O
from stair_step_detector_b200 import _abi as A

pytestmark = pytest.mark.gpu
ATOL = 1e-7
SMEM = [None, "0", "227"]
NOISY = dict(noise_sigma=0.0025, dropout=0.03, n_holes=3)
ENV = ("SSD_GPU_OUTLINE_SMEM_KB", "SSD_GPU_OUTLINE_GRIDX")


def _detector(S, monkeypatch, w, h, smem=None, gridx=None, max_frames=1, cfg=None, xf=None):
    for name, v in zip(ENV, (smem, gridx)):  # read once, in ssd_gpu_create
        if v is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, v)
    cfg = cfg or S.default_config(w, h)
    xf = xf or S.scene_transform(S.default_scene(w, h))
    return S.Detector(cfg, xf, max_frames=max_frames)


def _check_outline(det, img):
    gq, gv = det.detect_outline(img, O.MIN_EXT, 1.0)
    oq, ov = O.run_outline(img, O.MIN_EXT, 1.0)
    assert gv == ov
    assert np.allclose(gq, oq, rtol=0, atol=ATOL), (gq, oq)
    return gq, gv


def _check_front(det, img):
    gl, gr, gv = det.detect_front_edge(img)
    ol, orr, ov = O.run_front_edge(img)
    assert gv == ov
    assert np.allclose(gl, ol, rtol=0, atol=ATOL) and np.allclose(gr, orr, rtol=0, atol=ATOL), (gl, ol, gr, orr)
    return gl, gr, gv


def _under_every_band(S, monkeypatch, img, check):
    """the construction under every SMEM setting: each matches the oracle, and all give identical results"""
    out = []
    for smem in SMEM:
        with _detector(S, monkeypatch, img.shape[1], img.shape[0], smem) as det:
            out.append(check(det, img))
    for r in out[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(r, out[0]))


def _need_hypot_tie():
    if not O.libm_rounds_apart() or O.hypot_tie_profile() is None:
        pytest.skip("this libm rounds hypot(175, 338) and hypot(250, 287) alike: no hypot-dependent tie to construct")


def test_hypot_tie_outline(S, monkeypatch):
    """two lines of equal a*a + b*b and equal distance sums: glibc's hypot, which the reference divides by, makes the later pair
    strictly better; a correctly rounded denominator would tie them and pick the earlier one"""
    _need_hypot_tie()
    _under_every_band(S, monkeypatch, O.hypot_outline_case()[0], _check_outline)


def test_hypot_tie_front_edge(S, monkeypatch):
    _need_hypot_tie()
    _under_every_band(S, monkeypatch, O.hypot_front_case()[0], _check_front)


@pytest.mark.parametrize("w,h,n", O.MIRROR_SIZES)
def test_mirror_ties(S, monkeypatch, w, h, n):
    """exact ties between mirror lines (first in pair order wins) and all-pair ties at residual 0, per residual branch and class"""
    _under_every_band(S, monkeypatch, O.mirror_case(w, h, n)[0], _check_outline)


@pytest.mark.parametrize("w,h,n", O.FRONT_SIZES)
def test_front_edge_tents(S, monkeypatch, w, h, n):
    """front-edge lists from 6 to 41 points: sum_smallest<4 / 8 / 12> and the hi-res bisection of k_single_front_edge"""
    _under_every_band(S, monkeypatch, O.front_tent_case(w, h, n)[0], _check_front)


@pytest.mark.parametrize("name", sorted(O.decision_cases()))
def test_decisions(S, monkeypatch, name):
    """scan extent at min_img_y_extent and one less, 2 and 3 scans, a plateau on the image border, scans on columns 0 / W - 1"""
    img = O.decision_cases()[name][0]
    _under_every_band(S, monkeypatch, img, _check_outline)
    _under_every_band(S, monkeypatch, img, _check_front)


@pytest.mark.parametrize("w,h,n", [(640, 480, 4), (1024, 768, 4), (4096, 3072, 2)])
def test_chain_band_and_grid_stride(S, oracle, monkeypatch, w, h, n):
    """scene frames through the full chain (k_outline, k_finalize) with every band in global memory and with one and 32 blocks
    per plateau column, fused and seven-launch: identical to the default run and to the oracle"""
    cfg = S.default_config(w, h)
    base = S.default_scene(w, h, **NOISY)
    xf = S.scene_transform(base)
    scenes = [S.randomize_scene(base, 77 + w, i, 3, 8) for i in range(n)]
    xyz = np.stack([S.deproject_host(sc, S.synth_depth_host(sc)) for sc in scenes])

    def run(smem, gridx, against_oracle=False):
        with _detector(S, monkeypatch, w, h, smem, gridx, max_frames=n, cfg=cfg, xf=xf) as det:
            det.process_host(xyz)
            fused = []
            for f in range(n):
                g = H.gpu_result(det, f)
                fused.append((H.frame_record(g, 0xffffffff), g.line))
                if against_oracle:
                    o = H.oracle_process(oracle, cfg, xf, xyz[f])
                    assert not H.compare_results(o, g, tol=1e-4), (f, H.compare_results(o, g, tol=1e-4))
            p = det.malloc(xyz.nbytes)
            det.h2d(p, xyz)
            det.process_device(p, n, A.FLAG_STAGE_TIMING)
            seven = [(H.frame_record(H.gpu_result(det, f), 0xffffffff), H.gpu_result(det, f).line) for f in range(n)]
            assert seven == fused, (smem, gridx)
            return fused

    want = run(None, None, against_oracle=True)
    for smem, gridx in (("0", None), (None, "1"), (None, "32"), ("0", "32")):
        assert run(smem, gridx) == want, (smem, gridx)
