"""Vertex and z16 frames whose points sit on the thresholds the single-precision filters guard (tests/test_gpu_thresholds.py).

The filters (DESIGN.md section 2) decide in f32 with a proven error bound and hand a point inside the bound to the exact double
chain: point_code_scaled (range test and height bin, k_transform_bin), fast_pixel2 (BEV pixel, k_label_bev) and quadfilter_eval
(point in quadrilateral, k_quad_reduce). A point is put on a threshold like this: take a world target w* on it, solve
p* = A^-1 (w* - b) in double, round to f32, and take the cube of p* +- K ulps per coordinate. The world coordinates of the cube
are computed here in float64 in the reference's order, ((a0 x + a1 y) + a2 z) + b0 (numpy does not contract), so they are the
oracle's bit for bit, and points can be kept on the side of a threshold a construct needs.

Frames are built in world coordinates: a ground slab and three step slabs, each in the lower half of one height bin, so their
bands are [b, b + 1] and the boundaries b - 1 | b, b | b + 1 and b + 1 | b + 2 are known in advance."""
import numpy as np

from stair_step_detector_b200 import _abi as A

U = 2.0 ** -24
f32 = np.float32

# dyadic measuring range: with the "axis" transform (A = I, b = (0, 0, -1)) every limit is an exact f32 world coordinate
DYADIC = dict(x_min=-0.625, x_max=0.625, y_min=0.125, y_max=1.375, z_min=-0.125, z_max=1.125)
PLATEAU_BINS = (10, 27, 45, 62)  # ground, steps 1-3 (default height interval 0.01)
STEP_X = (-0.45, 0.45)
STEP_Y0, TREAD = 0.45, 0.28


def transform(base, a, b):
    xf = A.Transform.from_buffer_copy(bytes(base))
    for i, v in enumerate(np.asarray(a, np.float64).ravel()):
        xf.a[i] = float(v)
    for i, v in enumerate(np.asarray(b, np.float64).ravel()):
        xf.b[i] = float(v)
    return xf


def mats(xf):
    return np.array(xf.a[:]).reshape(3, 3), np.array(xf.b[:])


def transforms(S):
    """name -> (transform, configuration overrides). The scene pose; the same world frame seen from a camera displaced by
    several metres (|b| large); a scaled and sheared A (a poorly conditioned calibration triangle); a near-singular A whose BEV
    bound exceeds half a pixel (hu < 0: every BEV pixel takes the exact pass); an A with det <= 1e-12 (Mmax = inf: every
    decision of k_label_bev / k_quad_reduce is exact); the identity with a dyadic range (world limits hit exactly)."""
    base = S.scene_transform(S.default_scene(640, 480))
    a, b = mats(base)
    out = {"scene": (base, {})}
    d = np.array([-3.0, 2.0, 5.0])  # camera frame shifted: p' = p + d
    out["translated"] = (transform(base, a, b - a @ d), {})
    M = np.array([[2.5, 0.7, 0.0], [0.0, 0.4, 0.3], [0.0, 0.0, 1.3]])
    out["sheared"] = (transform(base, a @ M, b), {})
    out["near_singular"] = (transform(base, a @ np.diag([1.0, 1.0, 2e-4]), b), {})
    out["singular"] = (transform(base, a @ np.diag([1.0, 1.0, 1e-13]), b), {})
    out["axis"] = (transform(base, np.eye(3), [0.0, 0.0, -1.0]), dict(DYADIC))
    return out


def world(xf, p):
    """camera_to_world of f32 points in float64, the reference's order of operations"""
    a, b = mats(xf)
    x, y, z = (np.asarray(p, f32)[:, i].astype(np.float64) for i in range(3))
    return np.stack([((a[i, 0] * x + a[i, 1] * y) + a[i, 2] * z) + b[i] for i in range(3)], axis=1)


def camera(xf, w):
    a, b = mats(xf)
    return np.linalg.solve(a, (np.atleast_2d(w) - b).T).T.astype(f32)


def cube(xf, w_star, k):
    """camera points: f32(A^-1 (w* - b)) +- k ulps per coordinate, (2k + 1)^3 of them"""
    p = camera(xf, w_star)[0]
    axes = []
    for c in p:
        up, down = [c], [c]
        for _ in range(k):
            up.append(np.nextafter(up[-1], f32(np.inf)))
            down.append(np.nextafter(down[-1], f32(-np.inf)))
        axes.append(np.array(down[:0:-1] + up, f32))
    g = np.meshgrid(*axes, indexing="ij")
    return np.stack([c.ravel() for c in g], axis=1)


class Bounds:
    """derive_params's filter constants (ssd_gpu.cu) restated in numpy"""

    def __init__(self, cfg, xf):
        a, b = mats(xf)
        lo = np.array([cfg.x_min, cfg.y_min, cfg.z_min])
        hi = np.array([cfg.x_max, cfg.y_max, cfg.z_max])
        self.lo, self.hi = lo, hi
        self.hir = 1.0 / cfg.height_interval
        self.n_bins = int((cfg.z_max - cfg.z_min) * self.hir) + 1
        T = np.abs(np.concatenate([lo, hi])).max()
        self.E0 = f32(f32((10 * U * np.abs(b).max() + 16 * U * T) * 1.001) + f32(1e-12))
        self.E1 = f32(10 * U * np.abs(a).sum(1).max() * 1.001)
        c, h = (lo + hi) * 0.5, (hi - lo) * 0.5
        S1 = (np.abs(a).sum(1) / h).max()
        B1 = (np.abs(b - c) / h + 1).max()
        X1 = ((np.abs(b) + np.abs(c)) / h).max()
        self.E1s = f32(8 * U * S1 * 1.001)
        self.E0s = f32((8 * U * B1 + 1e-15 * X1) * 1.001)
        G = (cfg.z_max - cfg.z_min) * 0.5 * self.hir
        self.Gup = f32(G * 1.001)
        self.thr0 = f32((0.5 - (8 * U * (2 * G + self.n_bins + 2) + 1e-9)) * 0.9999)
        self.sx, self.sy = cfg.width / (cfg.x_max - cfg.x_min), cfg.height / (cfg.y_max - cfg.y_min)
        Su, Sv = np.abs(a[0] * self.sx).sum(), np.abs(a[1] * self.sy).sum()
        bu, bv = (b[0] - cfg.x_min) * self.sx, (cfg.y_max - b[1]) * self.sy
        Eu1, Ev1 = f32(6 * U * Su * 1.001), f32(6 * U * Sv * 1.001)
        Eu0, Ev0 = f32(6 * U * abs(bu) * 1.001 + 1e-6), f32(6 * U * abs(bv) * 1.001 + 1e-6)
        det = np.linalg.det(a)
        with np.errstate(over="ignore", invalid="ignore"):
            if abs(a[0, 0] * (a[1, 1] * a[2, 2] - a[1, 2] * a[2, 1]) - a[0, 1] * (a[1, 0] * a[2, 2] - a[1, 2] * a[2, 0])
                   + a[0, 2] * (a[1, 0] * a[2, 1] - a[1, 1] * a[2, 0])) > 1e-12:
                inv = np.linalg.inv(a)
                self.Mmax = (np.abs(inv) * (np.maximum(np.abs(lo), np.abs(hi)) + np.abs(b))[None, :]).sum(1).max() * 1.01
            else:
                self.Mmax = np.inf
            self.epsc = f32(f32(self.E1 * self.Mmax * 1.0001) + self.E0)
            self.euc = f32(f32(Eu1 * self.Mmax * 1.0001) + Eu0)
            self.evc = f32(f32(Ev1 * self.Mmax * 1.0001) + Ev0)
        self.hu = f32(0.5) - self.euc - f32(2.0 ** -20)
        self.hv = f32(0.5) - self.evc - f32(2.0 ** -20)
        self.det = det

    def eps_scaled(self, p):
        return self.E1s.astype(np.float64) * np.abs(p).max(1) + self.E0s

    def in_range_band(self, p, w, i):
        """the range decision on coordinate i is within point_code_scaled's bound"""
        v = (w[:, i] - (self.lo[i] + self.hi[i]) * 0.5) / ((self.hi[i] - self.lo[i]) * 0.5)
        return np.abs(np.abs(v) - 1) <= self.eps_scaled(p)

    def bin_of(self, w):
        return ((w[:, 2] - self.lo[2]) * self.hir).astype(np.int64)

    def in_bin_band(self, p, w):
        t = (w[:, 2] - self.lo[2]) * self.hir
        return np.abs(t - np.round(t)) <= 0.5 - (self.thr0 - self.Gup * self.eps_scaled(p))

    def pixel(self, w):
        """Projection2D::worldToImage of the oracle (no wrap handling: the constructs stay inside the image)"""
        return ((w[:, 0] - self.lo[0]) * self.sx).astype(np.int64), ((self.hi[1] - w[:, 1]) * self.sy).astype(np.int64)

    def in_bev_band(self, w, axis):
        u = (w[:, 0] - self.lo[0]) * self.sx if axis == 0 else (self.hi[1] - w[:, 1]) * self.sy
        return np.abs(u - np.round(u)) <= (self.euc if axis == 0 else self.evc) + 2.0 ** -20 if self.hu >= 0 else np.ones(len(w), bool)


def z_of_bin(cfg, k, frac):
    return cfg.z_min + (k + frac) * cfg.height_interval


def slab(rng, n, x0, x1, y0, y1, z0, z1):
    return np.stack([rng.uniform(x0, x1, n), rng.uniform(y0, y1, n), rng.uniform(z0, z1, n)], axis=1)


def step_rect(cfg, k, margin_px=0.3):
    """world rectangle of step k (1..3) with its four sides margin_px inside BEV pixel boundaries"""
    sx, sy = cfg.width / (cfg.x_max - cfg.x_min), cfg.height / (cfg.y_max - cfg.y_min)
    cl, cr = int(np.ceil((STEP_X[0] - cfg.x_min) * sx)), int(np.floor((STEP_X[1] - cfg.x_min) * sx))
    y0, y1 = STEP_Y0 + TREAD * (k - 1), STEP_Y0 + TREAD * k
    rb, rt = int(np.floor((cfg.y_max - y0) * sy)), int(np.ceil((cfg.y_max - y1) * sy))  # front (bottom) and back rows
    return dict(cl=cl, cr=cr, rf=rb, rb=rt, x0=cfg.x_min + (cl + margin_px) / sx, x1=cfg.x_min + (cr - margin_px) / sx,
                y0=cfg.y_max - (rb - margin_px) / sy, y1=cfg.y_max - (rt + margin_px) / sy)


BASE_POINTS = 40000 + 3 * 30000  # base_world's points come first in every frame


def base_world(cfg, rng, n_ground=40000, n_step=30000):
    """ground and three steps, each in the lower half of its height bin (PLATEAU_BINS scaled to the configuration's z range)"""
    parts = [slab(rng, n_ground, cfg.x_min + 0.02, cfg.x_max - 0.02, cfg.y_min + 0.02, STEP_Y0 - 0.01,
                  z_of_bin(cfg, PLATEAU_BINS[0], 0.15), z_of_bin(cfg, PLATEAU_BINS[0], 0.55))]
    for k in (1, 2, 3):
        r = step_rect(cfg, k)
        parts.append(slab(rng, n_step, r["x0"], r["x1"], r["y0"], r["y1"], z_of_bin(cfg, PLATEAU_BINS[k], 0.15),
                          z_of_bin(cfg, PLATEAU_BINS[k], 0.55)))
    return np.concatenate(parts)


def frame(cfg, xf, parts):
    """N x 3 f32 camera points: the parts (camera points), then invalid (0, 0, 0) vertices"""
    pts = np.concatenate(parts).astype(f32)
    N = cfg.width * cfg.height
    assert len(pts) <= N, len(pts)
    out = np.zeros((N, 3), f32)
    out[:len(pts)] = pts
    return out


# ---- the constructs: each returns (frame, constructed camera points, what they test) ----
def bins_and_range(cfg, xf, seed=1, k_bin=8, k_range=5):
    """height-bin boundaries b - 1 | b (band edge), b | b + 1 (inside the band: histogram only) and b + 1 | b + 2 (band edge) of
    every plateau, at the plateau's centre; cubes on all six range limits, small enough (k_range) not to make a peak of their
    own: x and y limits at the ground's height, z limits in bins no plateau uses"""
    rng = np.random.default_rng(seed)
    B = Bounds(cfg, xf)
    bins, rng_pts = [], {}
    for k, hb in enumerate(PLATEAU_BINS):
        if k == 0:
            cx, cy = 0.0, (cfg.y_min + STEP_Y0) * 0.5
        else:
            r = step_rect(cfg, k)
            cx, cy = (r["x0"] + r["x1"]) * 0.5, (r["y0"] + r["y1"]) * 0.5
        for edge in (hb, hb + 1, hb + 2):
            bins.append(cube(xf, [cx, cy, z_of_bin(cfg, edge, 0.0)], k_bin))
    zg = z_of_bin(cfg, PLATEAU_BINS[0], 0.35)
    ymid = (cfg.y_min + STEP_Y0) * 0.5
    targets = {"x_min": [cfg.x_min, ymid, zg], "x_max": [cfg.x_max, ymid, zg], "y_min": [0.0, cfg.y_min, zg],
               "y_max": [0.3, cfg.y_max, zg], "z_min": [-0.3, ymid, cfg.z_min], "z_max": [0.3, 1.0, cfg.z_max]}
    for name, t in targets.items():
        rng_pts[name] = cube(xf, t, k_range)
    w0 = camera(xf, base_world(cfg, rng))
    f = frame(cfg, xf, [w0] + bins + list(rng_pts.values()))
    return f, np.concatenate(bins), rng_pts, B


def bev_edges(cfg, xf, seed=2, k=2, every=1):
    """points of each step on the BEV pixel boundaries of its left and right sides (one cube per BEV row) and of its front edge
    (one cube per column), kept on the step's side of the boundary: a pixel decided one column or row outwards
    widens the step's image and moves its quadrilateral"""
    rng = np.random.default_rng(seed)
    B = Bounds(cfg, xf)
    w0 = base_world(cfg, rng)
    keep = []
    for s in (1, 2, 3):
        r = step_rect(cfg, s)
        z = z_of_bin(cfg, PLATEAU_BINS[s], 0.35)
        X = lambda c: cfg.x_min + c / B.sx
        Y = lambda row: cfg.y_max - row / B.sy
        for row in range(r["rb"] + 1, r["rf"] - 1):
            yc = Y(row + 0.5)
            for c, inner in ((r["cl"], r["cl"]), (r["cr"], r["cr"] - 1)):
                p = cube(xf, [X(c), yc, z], k)
                ix, iy = B.pixel(world(xf, p))
                keep.append(p[(ix == inner) & (iy == row)])
        for c in range(r["cl"] + 1, r["cr"] - 1, every):
            p = cube(xf, [X(c + 0.5), Y(r["rf"]), z], k)
            ix, iy = B.pixel(world(xf, p))
            keep.append(p[(ix == c) & (iy == r["rf"] - 1)])
    pts = np.concatenate(keep)
    return frame(cfg, xf, [camera(xf, w0), pts]), pts, B


QUAD_EDGES = ((0, 1), (1, 3), (3, 2), (2, 0))


def quad_thresholds(q):
    """QuadrilateralTest's row thresholds (the middle vertex y's), cell thresholds (the middle vertex x's) and the corners of the
    inner box quadtest_inner_box tries first (ssd_device.cuh): the sorted vertex coordinates 1 and 2, shrunk by 0.1 % + 1e-6"""
    xs, ys = np.sort(q[:, 0]), np.sort(q[:, 1])
    sx, sy = 0.001 * (xs[2] - xs[1]) + 1e-6, 0.001 * (ys[2] - ys[1]) + 1e-6
    box = [(x, y) for x in (xs[1] + sx, xs[2] - sx) for y in (ys[1] + sy, ys[2] - sy)]
    return xs[1:3], ys[1:3], box


def quad_edges(cfg, xf, quads, seed=3, k=4, n_along=11, k_vertex=8):
    """points on the thresholds of each step's quadrilateral (quads: step index -> 4x2 quad_world of the plateau in the frame
    without them): cubes along its four sides and on its row / cell thresholds across its interior, kept only where the step's
    own points already set the BEV pixel, so the image and with it the quadrilateral stay as they were; cubes at the inner box's
    corners; and larger cubes at the four vertices, where the sides meet the bounding box. The sides run through the step's
    pixels, so both sides keep points."""
    rng = np.random.default_rng(seed)
    B = Bounds(cfg, xf)
    p0 = camera(xf, base_world(cfg, rng))
    w0 = world(xf, p0)
    ix0, iy0 = B.pixel(w0)
    b0 = B.bin_of(w0)
    pts = []
    for s, q in quads.items():
        z = z_of_bin(cfg, PLATEAU_BINS[s], 0.35)
        own = list(set((iy0 * cfg.width + ix0)[(b0 == PLATEAU_BINS[s]) | (b0 == PLATEAU_BINS[s] + 1)].tolist()))
        targets = [q[i] + (q[j] - q[i]) * t for i, j in QUAD_EDGES for t in np.linspace(0.0, 1.0, n_along)]
        xt, yt, box = quad_thresholds(q)
        lo, hi = q.min(0), q.max(0)
        targets += [(x, y) for x in xt for y in np.linspace(lo[1], hi[1], 7)[1:-1]]
        targets += [(x, y) for y in yt for x in np.linspace(lo[0], hi[0], 7)[1:-1]]
        for c in targets:
            p = cube(xf, [c[0], c[1], z], k)
            ix, iy = B.pixel(world(xf, p))
            pts.append(p[np.isin(iy * cfg.width + ix, own)])
        pts += [cube(xf, [c[0], c[1], z], k) for c in box]
        pts += [cube(xf, [c[0], c[1], z], k_vertex) for c in q]
    pts = np.concatenate(pts)
    return frame(cfg, xf, [p0, pts]), pts, B


def base_frame(cfg, xf, seed=3):
    """the frame quad_edges adds its points to, without them"""
    return frame(cfg, xf, [camera(xf, base_world(cfg, np.random.default_rng(seed)))])


def quad_side(q, w):
    """signed distance (metres, normalised like QuadrilateralTest's steep / flat lines) of each point to the nearest side"""
    best = np.full(len(w), np.inf)
    for i, j in QUAD_EDGES:
        dx, dy = q[j] - q[i]
        val = (w[:, 0] - q[i][0]) * dy - (w[:, 1] - q[i][1]) * dx
        d = val / max(abs(dx), abs(dy))
        best = np.where(np.abs(d) < np.abs(best), d, best)
    return best


# ---- z16 frames ----
DEPTH_UNIT = 0.001
DEPTH0 = 1000  # depth of the first rectangle, in units


def depth_transform(base, cfg, first_bin=20):
    """x = p_x, y = p_y + 0.7, z = p_z + b_z: rectangle k (depth DEPTH0 + 10 k units, one height interval apart) lands on the
    boundary first_bin + k - 1 | first_bin + k"""
    bz = cfg.z_min + first_bin * cfg.height_interval - DEPTH0 * DEPTH_UNIT
    return transform(base, np.eye(3), [0.0, 0.7, bz])


def depth_frame(w, h, cols=4, rows=5):
    """cols x rows rectangles of constant depth, DEPTH0 + 10 k units"""
    d = np.zeros((h, w), np.uint16)
    k = 0
    for r in range(rows):
        for c in range(cols):
            d[r * h // rows:(r + 1) * h // rows, c * w // cols:(c + 1) * w // cols] = DEPTH0 + 10 * k
            k += 1
    return d
