"""Designed scan-point lists for the outline and front-edge line fits (tests/outline_frames.py), checked on the host through the
oracle's own scans (tests/native/oracle_outline.c): the lists are as designed, the claimed ties and the hypot dependence are
present, and a different winner would move the output far beyond the 1e-7 px bar of tests/test_gpu_outline_fits.py."""
import numpy as np
import pytest

import outline_frames as O


def test_hypot_tie_outline_list_and_winner():
    if not O.libm_rounds_apart():
        pytest.skip("this libm rounds hypot(175, 338) and hypot(250, 287) alike: no hypot-dependent tie on this host")
    img, right = O.hypot_outline_case()
    scans, lists = O.outline_lists(img, O.MIN_EXT)
    assert len(scans) == 21
    assert np.array_equal(lists[1], right), lists[1]
    ref, cr = O.Fit(lists[1]), O.Fit(lists[1], use_sqrt=True)
    # correctly rounded denominator: an exact tie of two distinct lines, the first (0, 7) wins; glibc's: (0, 10) alone
    assert (cr.at_min, cr.distinct, O.pair_of(cr.winner, 11)) == (2, 2, (0, 7))
    assert (ref.at_min, O.pair_of(ref.winner, 11)) == (1, (0, 10))
    assert O.branch(ref.cnt, True) == O.branch(ref.cnt, False) == "sum_smallest<4>"
    q0, v0 = O.run_outline(img, O.MIN_EXT, 1.0, 0)
    q1, v1 = O.run_outline(img, O.MIN_EXT, 1.0, 1)
    assert v0 != v1 or np.abs(q0 - q1).max() > 1e-3, (q0, q1)


def test_hypot_tie_front_edge_list_and_winner():
    if not O.libm_rounds_apart():
        pytest.skip("this libm rounds hypot(175, 338) and hypot(250, 287) alike: no hypot-dependent tie on this host")
    img, pts = O.hypot_front_case()
    lst = O.front_list(img)
    assert np.array_equal(lst, pts), lst
    ref, cr = O.Fit(lst), O.Fit(lst, use_sqrt=True)
    assert (cr.at_min, cr.distinct, O.pair_of(cr.winner, 11)) == (2, 2, (0, 7))
    assert (ref.at_min, O.pair_of(ref.winner, 11)) == (1, (0, 10))
    l0, r0, v0 = O.run_front_edge(img, 0)
    l1, r1, v1 = O.run_front_edge(img, 1)
    assert v0 == v1 == 1
    assert max(np.abs(l0 - l1).max(), np.abs(r0 - r1).max()) > 1e-3, (l0, l1, r0, r1)


# residual branch of the frontRight list per construction, in the frame's own size class
MIRROR_BRANCH = {(320, 240, 5): "sum_smallest<4>", (320, 240, 7): "sum_smallest<4>", (1348, 1108, 9): "sum_smallest<4>",
                 (1348, 1108, 13): "sum_smallest<8>", (1348, 1108, 21): "sum_smallest<12>", (1348, 1108, 27): "sum_smallest<12>",
                 (1352, 1108, 21): "sum_smallest<12>", (1352, 1108, 27): "sum_smallest<12>", (4096, 3072, 29): "hi-res bisection",
                 (4096, 3072, 45): "hi-res bisection", (4096, 3072, 81): "hi-res bisection"}


@pytest.mark.parametrize("w,h,n", O.MIRROR_SIZES)
def test_mirror_ties(w, h, n):
    """each size: the designed frontRight list, the residual branch its class runs, an exact tie of two distinct lines at the
    minimum of a front list, every pair tied at 0 on the one-row back lists; the tied lines part by more than 1e-7 px"""
    img, right = O.mirror_case(w, h, n)
    scans, lists = O.outline_lists(img, O.MIN_EXT)
    assert np.array_equal(lists[1], np.stack([w // 2 + 25 * np.arange(n), right], 1)), lists[1]
    assert len(lists[0]) == len(lists[2]) == len(lists[3]) == n
    fits = [O.Fit(l) for l in lists]
    assert O.branch(fits[1].cnt, O.small_class(w, h)) == MIRROR_BRANCH[(w, h, n)]
    assert fits[1].distinct >= 2, (fits[1].at_min, fits[1].distinct)
    for f, pts in zip(fits[:2], lists[:2]):
        if f.distinct >= 2:
            xs = pts[:, 0]
            d = max(abs(O.line_y(f.line, x) - O.line_y(f.other, x)) for x in (xs.min(), xs.max()))
            assert d > 1e-3, d
    for f, pts in zip(fits[2:], lists[2:]):
        assert f.residual == 0 and f.winner == 0 and f.at_min == len(pts) * (len(pts) - 1) // 2


FRONT_BRANCH = {(640, 480, 6): "sum_smallest<4>", (1348, 1108, 14): "sum_smallest<8>", (4096, 3072, 27): "sum_smallest<12>",
                (4096, 3072, 41): "hi-res bisection"}


@pytest.mark.parametrize("w,h,n", O.FRONT_SIZES)
def test_front_edge_tents(w, h, n):
    """front-edge lists (k_single_front_edge always runs the large class): the designed list, its branch, a tie of two distinct
    lines at the minimum that would move the end points by more than 1e-7 px"""
    img, pts = O.front_tent_case(w, h, n)
    lst = O.front_list(img)
    assert np.array_equal(lst, pts), lst
    f = O.Fit(lst)
    assert O.branch(f.cnt, False) == FRONT_BRANCH[(w, h, n)]
    assert f.distinct >= 2
    xs = lst[:, 0]
    assert max(abs(O.line_y(f.line, x) - O.line_y(f.other, x)) for x in (xs.min(), xs.max())) > 1e-3


def test_band_paths():
    """which band path each single-stage construction of tests/test_gpu_outline_fits.py takes under SSD_GPU_OUTLINE_SMEM_KB
    unset / 0 / 227: both paths are taken, and 640 x 480 takes the global path by default and shared memory at 227"""
    sizes = {(320, 240), (640, 480), (2048, 1536)} | {(w, h) for w, h, _ in O.MIRROR_SIZES + O.FRONT_SIZES}
    table = {s: tuple(O.band_path(*s, k) for k in (None, "0", "227")) for s in sorted(sizes)}
    print(table)
    assert table[(320, 240)] == ("smem", "global", "smem")
    assert table[(640, 480)] == ("global", "global", "smem")
    assert table[(2048, 1536)] == table[(4096, 3072)] == ("global", "global", "global")
    assert all(t[1] == "global" for t in table.values())


@pytest.mark.parametrize("name", sorted(O.decision_cases()))
def test_decision_constructions(name):
    """the scans the oracle sees for each decision construction: the designed number, the scan on the border column where one
    is designed"""
    img, n_scans = O.decision_cases()[name]
    scans, lists = O.outline_lists(img, O.MIN_EXT)
    assert len(scans) == n_scans, scans
    H, W = img.shape
    if name == "scan_on_column_0":
        assert 0 in scans[:, 0]
    if name == "scan_on_column_W-1":
        assert W - 1 in scans[:, 0]
    assert (len(lists[0]) > 0) == (n_scans >= 3)
