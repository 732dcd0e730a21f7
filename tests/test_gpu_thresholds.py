"""Points placed on every threshold a single-precision filter guards, so that the exact double chain has to decide them
(DESIGN.md section 2: bit-exact including points near a threshold). The frames come from tests/threshold_frames.py:
- height-bin boundaries inside each plateau's band (histogram only) and at its edges (labels), and all six range limits
  (point_code_scaled in k_transform_bin);
- BEV pixel column / row boundaries along the sides and front edge of each step, kept on the step's side (fast_pixel2 in
  k_label_bev): a pixel decided outwards moves the quadrilateral, compared at 1e-9 m;
- the four sides and corners of each step's quadrilateral (quadfilter_eval in k_quad_reduce): n_in_quad exactly, mean z.
Six transforms stress the bounds (scene pose, large translation, scaled and sheared, near-singular, singular, identity with a
dyadic range so that points lie exactly on the limits). Each construct runs as a one-frame fused call and as a seven-launch
call, and through a three-camera table; z16 frames of constant-depth rectangles one height interval apart sit on consecutive
bin boundaries for host and device z16 input, a Brown-Conrady lens and a camera-table depth call.

Every GPU test asserts that the constructed points reached the exact pass (n_exact_fallback, n_bev_exact, n_quad_exact against
a floor of half the constructed points); the tests without the gpu mark check the constructions themselves."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import threshold_frames as T
from stair_step_detector_b200 import _abi as A

TOL = 1e-4  # metres, as tests/test_gpu_parity.py
QUAD_TOL = 1e-9  # quadrilateral corners come from integer pixels: a pixel off moves them by a millimetre
gpu = pytest.mark.gpu
NAMES = ["scene", "translated", "sheared", "near_singular", "singular", "axis"]
CONSTRUCTS = ["bins_range", "bev", "quad"]


def setup(S, oracle, name, construct):
    """cfg, xf, frame, constructed camera points, Bounds"""
    xf, kw = T.transforms(S)[name]
    cfg = S.default_config(640, 480, **kw)
    if construct == "bins_range":
        f, binp, rngp, B = T.bins_and_range(cfg, xf)
        return cfg, xf, f, np.concatenate([binp] + list(rngp.values())), B
    if construct == "bev":
        f, pts, B = T.bev_edges(cfg, xf)
        return cfg, xf, f, pts, B
    o0 = H.oracle_process(oracle, cfg, xf, T.base_frame(cfg, xf))
    f, pts, B = T.quad_edges(cfg, xf, {s: o0.plateaus[s]["quad_world"] for s in (1, 2, 3)})
    return cfg, xf, f, pts, B


_CACHE = {}


def cached(S, oracle, name, construct):
    key = (name, construct)
    if key not in _CACHE:
        _CACHE[key] = setup(S, oracle, name, construct)
    return _CACHE[key]


# ---- the constructions (no GPU) ----
@pytest.mark.parametrize("name", NAMES)
def test_world_coordinates_equal_the_oracle(S, oracle, name):
    for construct in CONSTRUCTS:
        cfg, xf, f, pts, B = cached(S, oracle, name, construct)
        valid = f[:, 2] > 0
        got = T.world(xf, f[valid])
        want = np.empty_like(got)
        xyz = np.ascontiguousarray(f[valid])
        oracle.ssd_oracle_camera_to_world(C.byref(xf), H.ptr(xyz), len(xyz), H.ptr(want))
        assert np.isfinite(got).all() and np.array_equal(got.view(np.uint64), want.view(np.uint64)), construct


def test_transforms_reach_their_bounds(S):
    cfg = S.default_config(640, 480)
    tr = T.transforms(S)
    B = {n: T.Bounds(S.default_config(640, 480, **kw), xf) for n, (xf, kw) in tr.items()}
    assert np.abs(np.array(tr["translated"][0].b[:])).max() > 4.0
    assert B["near_singular"].hu < 0 and B["near_singular"].hv < 0 and np.isfinite(B["near_singular"].Mmax)
    assert B["singular"].Mmax == np.inf and abs(B["singular"].det) <= 1e-12
    for n in ("scene", "translated", "sheared", "axis"):
        assert 0 < B[n].hu < 0.5 and 0 < B[n].epsc < 1e-4, n
    assert cfg.x_min == -0.6  # the other transforms run the default range


@pytest.mark.parametrize("name", NAMES)
def test_bins_and_range_construct(S, oracle, name):
    """each bin boundary cube splits over its two bins, inside point_code_scaled's bound; each range cube has points on both
    sides of its limit (the identity: exactly on it too); the bands come out as designed"""
    xf, kw = T.transforms(S)[name]
    cfg = S.default_config(640, 480, **kw)
    f, binp, rngp, B = T.bins_and_range(cfg, xf)
    n_cube = len(binp) // (3 * len(T.PLATEAU_BINS))
    for i in range(3 * len(T.PLATEAU_BINS)):
        p = binp[i * n_cube:(i + 1) * n_cube]
        w = T.world(xf, p)
        b = B.bin_of(w)
        assert len(np.unique(b)) == 2 and min(np.bincount(b - b.min())) > n_cube // 10, (i, np.unique(b, return_counts=True))
        assert B.in_bin_band(p, w).mean() >= 0.5, i
    for lim, p in rngp.items():
        i = "xyz".index(lim[0])
        w = T.world(xf, p)
        v, L = w[:, i], getattr(cfg, lim)
        inside = v > L if lim.endswith("min") else v < L
        assert 0.1 < inside.mean() < 0.9, lim
        assert B.in_range_band(p, w, i).mean() >= 0.5, lim
        if name == "axis":
            assert (v == L).sum() > 0, lim
    o = H.oracle_process(oracle, cfg, xf, f)
    assert o.info["n_steps"] == 4
    for k, pl in enumerate(o.plateaus):
        assert (pl["hmin"], pl["hmax"]) == (T.PLATEAU_BINS[k], T.PLATEAU_BINS[k] + 1), k


@pytest.mark.parametrize("name", NAMES)
def test_bev_construct(S, oracle, name):
    """the kept points lie on their step's side of a pixel boundary and inside fast_pixel2's bound on that axis"""
    cfg, xf, f, pts, B = cached(S, oracle, name, "bev")
    w = T.world(xf, pts)
    band = B.in_bev_band(w, 0) | B.in_bev_band(w, 1)
    assert band.mean() >= 0.95, band.mean()
    o = H.oracle_process(oracle, cfg, xf, f)
    assert o.info["n_steps"] == 4 and all(p["valid"] for p in o.plateaus)


@pytest.mark.parametrize("name", NAMES)
def test_quad_construct(S, oracle, name):
    """points inside and outside each step's quadrilateral, within quadfilter_eval's margin of a side; the quadrilaterals are
    those of the frame without them"""
    cfg, xf, f, pts, B = cached(S, oracle, name, "quad")
    o0 = H.oracle_process(oracle, cfg, xf, T.base_frame(cfg, xf))
    o = H.oracle_process(oracle, cfg, xf, f)
    w = T.world(xf, pts)
    n_in = n_out = 0
    for s in (1, 2, 3):
        q = o0.plateaus[s]["quad_world"]
        assert np.array_equal(o.plateaus[s]["quad_world"], q), s
        d = T.quad_side(q, w)
        near = np.abs(d) <= 3 * B.epsc
        n_in += int((near & (d > 0)).sum())
        n_out += int((near & (d < 0)).sum())
        assert o.plateaus[s]["n_in_quad"] > o0.plateaus[s]["n_in_quad"], s
    assert n_in > len(pts) // 10 and n_out > len(pts) // 10, (n_in, n_out, len(pts))


# ---- on the GPU ----
def check_against_oracle(o, g, what):
    bad = H.compare_results(o, g, tol=TOL)
    assert not bad, (what, bad)
    assert g.info["status"] == o.info["status"], what
    for k, (p, q) in enumerate(zip(o.plateaus, g.plateaus)):
        if p["valid"]:
            assert np.allclose(p["quad_world"], q["quad_world"], rtol=0, atol=QUAD_TOL), (what, k)
            assert p["n_in_quad"] == q["n_in_quad"], (what, k)


def floor_counter(construct, st):
    return {"bins_range": st.n_exact_fallback, "bev": st.n_bev_exact, "quad": st.n_quad_exact}[construct]


@gpu
@pytest.mark.parametrize("construct", CONSTRUCTS)
@pytest.mark.parametrize("name", NAMES)
def test_thresholds_fused_and_seven_launch(S, oracle, name, construct):
    cfg, xf, f, pts, B = cached(S, oracle, name, construct)
    o = H.oracle_process(oracle, cfg, xf, f)
    with S.Detector(cfg, xf, max_frames=1) as det:
        det.process_host(f[None])
        assert det.timing().n_launches == 5
        g = H.gpu_result(det, 0)
        check_against_oracle(o, g, "fused")
        st = det.stats()
        assert floor_counter(construct, st) >= len(pts) // 2, (floor_counter(construct, st), len(pts))
        want = H.frame_record(g, 0xffffffff)
        d = det.malloc(f.nbytes)
        det.h2d(d, f)
        det.process_device(d, 1, A.FLAG_STAGE_TIMING)
        assert det.timing().n_launches == 7
        assert H.frame_record(H.gpu_result(det, 0), 0xffffffff) == want, "seven-launch"
        assert floor_counter(construct, det.stats()) >= len(pts) // 2, "seven-launch"
        det.free(d)
    if construct == "bins_range":
        # the band-edge cubes (b - 1 | b and b + 1 | b + 2 of plateau k): the exact decisions put points of each on both sides,
        # the plateau's label and the remainder's
        n_cube = (2 * 8 + 1) ** 3
        for k in range(len(T.PLATEAU_BINS)):
            for e in (0, 2):
                i0 = T.BASE_POINTS + (3 * k + e) * n_cube
                ls = g.labels[i0:i0 + n_cube]
                assert (ls == k).any() and (ls == A.LABEL_REMAINDER).any(), (k, e)


@gpu
@pytest.mark.parametrize("construct", CONSTRUCTS)
def test_thresholds_camera_table(S, oracle, construct):
    """frames built for three different cameras in one camera-table call: each frame's bounds are its camera's. The context's
    own transform is the one with the smallest bounds (scene), so bounds taken from the context instead of the frame's camera
    would be too narrow for the other two frames"""
    names = ["scene", "translated", "sheared"]
    cases = [cached(S, oracle, n, construct) for n in names]
    cfg = cases[0][0]
    frames = np.stack([c[2] for c in cases])
    order = np.array([2, 0, 1], np.int32)
    assert all(cases[0][4].epsc < c[4].epsc and cases[0][4].euc < c[4].euc for c in cases[1:])
    with S.Detector(cfg, cases[0][1], max_frames=3) as det:
        det.set_cameras([S.make_camera(c[1]) for c in cases])
        det.process_cameras_host(frames[order], order)
        st = det.stats()
        for i, c in enumerate(order):
            check_against_oracle(H.oracle_process(oracle, cfg, cases[c][1], frames[c]), H.gpu_result(det, i), (construct, names[c]))
        assert floor_counter(construct, st) >= sum(len(c[3]) for c in cases) // 2


# ---- z16 ----
def depth_case(S, lens=None):
    cfg = S.default_config(640, 480)
    sc = S.default_scene(640, 480)
    sc.depth_unit = T.DEPTH_UNIT
    if lens is not None:
        sc.distortion_model = lens[0]
        for i, c in enumerate(lens[1]):
            sc.coeffs[i] = c
    xf = T.depth_transform(S.scene_transform(sc), cfg)
    depth = T.depth_frame(640, 480)
    xyz = S.deproject_host(sc, depth).reshape(-1, 3)
    w = T.world(xf, xyz)
    # range limits on the exact world coordinates of chosen pixels: x_max at column 540, y_max at row 460
    cfg.x_max = float(w[10 * 640 + 540, 0])
    cfg.y_max = float(w[460 * 640 + 100, 1])
    return cfg, xf, sc, depth, xyz, w


def test_depth_construct(S):
    """each rectangle sits on a bin boundary: its points fall in one of the two bins next to it (f32 rounding of d * unit
    decides which), both outcomes occur, and every point is inside point_code_scaled's bound"""
    cfg, xf, sc, depth, xyz, w = depth_case(S)
    B = T.Bounds(cfg, xf)
    d = depth.reshape(-1)
    sides = set()
    for k in range(20):
        m = d == T.DEPTH0 + 10 * k
        b = np.unique(B.bin_of(w[m]))
        assert len(b) == 1 and b[0] in (19 + k, 20 + k), (k, b)
        sides.add(int(b[0]) - k)
        assert B.in_bin_band(xyz[m], w[m]).all(), k
    assert sides == {19, 20}
    assert (w[:, 0] == cfg.x_max).sum() > 0 and (w[:, 1] == cfg.y_max).sum() > 0


@gpu
def test_depth_rectangles_on_bin_boundaries(S, oracle):
    """vertex input against the oracle; z16 host and device input, a camera-table depth call and a Brown-Conrady lens against
    the vertex input of the same vertices, bit for bit; nearly every in-range point takes the exact pass"""
    BC = (A.DISTORTION_BROWN_CONRADY, (0.12, -0.08, 0.002, -0.0015, 0.03))
    for lens in (None, BC):
        cfg, xf, sc, depth, xyz, w = depth_case(S, lens)
        intr = S.scene_intrinsics(sc)
        o = H.oracle_process(oracle, cfg, xf, xyz)
        assert o.info["n_in_range"] > 100000
        with S.Detector(cfg, xf, max_frames=1) as det:
            det.process_host(xyz[None])
            g = H.gpu_result(det, 0)
            check_against_oracle(o, g, ("vertex", lens))
            assert det.stats().n_exact_fallback >= o.info["n_in_range"] // 2
            want = H.frame_record(g, 0xffffffff)
            dist = S.make_distortion(*lens) if lens else None
            det.set_distortion(dist)
            det.set_cameras([S.make_camera(xf, None, intr)], None if lens is None else [dist])
            d = det.malloc(depth.nbytes)
            det.h2d(d, depth)
            for kind, run in (("z16 host", lambda: det.process_depth_host(depth[None], intr)),
                              ("z16 device", lambda: det.process_depth_device(d, intr, 1)),
                              ("z16 camera table", lambda: det.process_depth_cameras_host(depth[None], np.zeros(1, np.int32)))):
                run()
                assert H.frame_record(H.gpu_result(det, 0), 0xffffffff) == want, (kind, lens)
                assert det.stats().n_exact_fallback >= o.info["n_in_range"] // 2, (kind, lens)
            det.free(d)
