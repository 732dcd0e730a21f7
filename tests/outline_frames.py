"""Binary images with designed scan-point lists for the outline and front-edge line fits (tests/test_outline_fits.py,
tests/test_gpu_outline_fits.py), and the native helper that inspects them (tests/native/oracle_outline.c).

A scan point is the first / last set row of a closed-image column W/2 + 25 k (detectOutline) or the bottom-most set row below
H/2 of a column W/2 + 50 k (detectFrontEdge). Each scanned column's segment is drawn over the block of columns around it
(+-12 for the outline, +-24 for the front edge), so the 3x3 close cannot move a scanned pixel: it only fills the corners where
neighbouring blocks meet, 12 or more columns away from any scanned one.

Branch table of the device line fit (pair_residual, ssd_kernels_outline.cuh): cnt = (n - 3) / 2 for n > 6 points, else 1;
cnt <= 4, 8, 12: sum_smallest<4 / 8 / 12>; above that the small frame-size class (OutlineSharedSmall: W / 25 + 4 <= 64,
W / 50 + 6 <= 32, H / 10 + 2 <= 112, i.e. W <= 1349 and H <= 1109) extracts repeated minima (cnt <= 24) and the large class
(OutlineShared, and k_single_front_edge at any size) runs the hi-res bisection with the pruning probe."""
import atexit
import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_vp, _P = C.c_void_p, C.POINTER
OUTLINE_STEP, FRONT_STEP = 25, 50
LIST_NAMES = ("frontLeft", "frontRight", "backLeft", "backRight")
_LIB = {}


def helper():
    """tests/native/oracle_outline.c compiled with oracle/Makefile's flags into a temporary directory"""
    if "lib" not in _LIB:
        tmp = tempfile.mkdtemp(prefix="ssd_oracle_outline_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libssd_oracle_outline.so")
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", out,
                        os.path.join(ROOT, "tests", "native", "oracle_outline.c"), "-lm"], check=True)
        lib = C.CDLL(out)
        lib.oo_outline_lists.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, _P(C.c_int), _P(C.c_int), _vp, _vp]
        lib.oo_front_list.argtypes = [_vp, C.c_int, C.c_int, _vp]
        lib.oo_fit_stats.argtypes = [_vp, C.c_int, C.c_int, _vp]
        lib.oo_set_hypot_mode.argtypes = [C.c_int]
        lib.ssd_oracle_detect_outline.argtypes = [_vp, C.c_int, C.c_int, C.c_int, C.c_double, _P(C.c_double), _P(C.c_int)]
        lib.ssd_oracle_detect_front_edge.argtypes = [_vp, C.c_int, C.c_int, _P(C.c_double), _P(C.c_double), _P(C.c_int)]
        _LIB["lib"] = lib
    return _LIB["lib"]


def _libm_hypot():
    m = C.CDLL("libm.so.6")
    m.hypot.restype, m.hypot.argtypes = C.c_double, [C.c_double, C.c_double]
    return m.hypot


libm_hypot = _libm_hypot()


# ---- construction ----
def outline_image(W, H, segs):
    """segs: {column: (yFirst, ySecond)} for scan columns W/2 + 25 k; each segment filled over the column's +-12 block"""
    img = np.zeros((H, W), np.uint8)
    for x, (yf, ys) in segs.items():
        img[yf:ys + 1, max(0, x - 12):min(W, x + 13)] = 255
    return img


def outline_segs(W, right, left, y_first=None):
    """scan segments from profiles: right[k] / left[k] are the ySecond of columns W/2 + 25 k / W/2 - 25 (k + 1); y_first: a
    constant yFirst or per-column lists (right_first, left_first)"""
    c = W // 2
    rf, lf = (y_first if isinstance(y_first, tuple) else ([y_first or 0] * len(right), [y_first or 0] * len(left)))
    segs = {c + OUTLINE_STEP * k: (int(rf[k]), int(y)) for k, y in enumerate(right)}
    segs.update({c - OUTLINE_STEP * (k + 1): (int(lf[k]), int(y)) for k, y in enumerate(left)})
    return segs


def front_image(W, H, bottoms, top=None):
    """bottoms: {column: bottom-most set row (> H/2)}; each column's block +-24 filled from row `top` (default H/2 + 1)"""
    img = np.zeros((H, W), np.uint8)
    t = H // 2 + 1 if top is None else top
    for x, y in bottoms.items():
        img[min(t, y):y + 1, max(0, x - 24):min(W, x + 26)] = 255
    return img


# ---- inspection ----
def outline_lists(img, min_ext):
    """(scans, lists): scans the (x, yFirst, ySecond) rows of the right then left scans; lists the four (n, 2) point lists in
    LIST_NAMES order (empty when the fit does not run)"""
    H, W = img.shape
    lib = helper()
    cap2 = W // 25 + 4
    scans = np.zeros((2 * (W // 25 + 2), 3), np.int32)
    lists = np.zeros((4, cap2, 2), np.int32)
    n = np.zeros(4, np.int32)
    nr, nl = C.c_int(), C.c_int()
    img = np.ascontiguousarray(img, np.uint8)
    lib.oo_outline_lists(img.ctypes.data, W, H, min_ext, scans.ctypes.data, C.byref(nr), C.byref(nl), lists.ctypes.data, n.ctypes.data)
    return scans[:nr.value + nl.value], [lists[e, :n[e]].copy() for e in range(4)]


def front_list(img):
    H, W = img.shape
    pts = np.zeros((W // 50 + 3, 2), np.int32)
    img = np.ascontiguousarray(img, np.uint8)
    n = helper().oo_front_list(img.ctypes.data, W, H, pts.ctypes.data)
    return pts[:n].copy()


class Fit:
    """BestLine statistics of one list (oo_fit_stats)"""

    def __init__(self, pts, use_sqrt=False):
        pts = np.ascontiguousarray(pts, np.int32)
        out = np.zeros(13)
        helper().oo_fit_stats(pts.ctypes.data, len(pts), int(use_sqrt), out.ctypes.data)
        self.n = len(pts)
        self.cnt, self.residual, self.at_min, self.distinct = int(out[0]), out[1], int(out[2]), int(out[3])
        self.winner, self.isum, self.max_sum = int(out[4]), int(out[5]), int(out[6])
        self.line, self.other = tuple(int(v) for v in out[7:10]), tuple(int(v) for v in out[10:13])


def pair_of(idx, n):
    """(p, q) of the pair index in (p, q) lexicographic order"""
    p = 0
    while idx >= n - 1 - p:
        idx -= n - 1 - p
        p += 1
    return p, p + 1 + idx


def branch(cnt, small):
    """the residual evaluator pair_residual runs for a list with this cnt (small: OutlineSharedSmall)"""
    for s in (4, 8, 12):
        if cnt <= s:
            return f"sum_smallest<{s}>"
    if small:
        return "extraction" if cnt <= 24 else "small bisection"
    return "hi-res bisection"


def small_class(W, H):
    return W // 25 + 4 <= 64 and W // 50 + 6 <= 32 and H // 10 + 2 <= 112


def line_y(line, x):
    """FlatLine y at column x (segmentation.cpp:490-519) of an integer line (a, b, c)"""
    a, b, c = line
    return x * ((-a) / b) + (-c) / b


def run_outline(img, min_ext, xy_ratio, hypot_mode=0):
    """the oracle's detectOutline; hypot_mode 1: integer hypots correctly rounded (what the line fit gives with sqrt)"""
    H, W = img.shape
    lib = helper()
    lib.oo_set_hypot_mode(hypot_mode)
    q, v = (C.c_double * 8)(), C.c_int()
    img = np.ascontiguousarray(img, np.uint8)
    lib.ssd_oracle_detect_outline(img.ctypes.data, W, H, min_ext, xy_ratio, q, C.byref(v))
    lib.oo_set_hypot_mode(0)
    return np.array(q[:]).reshape(4, 2), v.value


def run_front_edge(img, hypot_mode=0):
    H, W = img.shape
    lib = helper()
    lib.oo_set_hypot_mode(hypot_mode)
    l, r, v = (C.c_double * 2)(), (C.c_double * 2)(), C.c_int()
    img = np.ascontiguousarray(img, np.uint8)
    lib.ssd_oracle_detect_front_edge(img.ctypes.data, W, H, l, r, C.byref(v))
    lib.oo_set_hypot_mode(0)
    return np.array(l[:]), np.array(r[:]), v.value


# ---- designed profiles ----
# (175, 338) and (250, 287): a*a + b*b = 144869 for both, and glibc's hypot rounds them to neighbouring doubles
# (0x1.7c9dd9d33bcfcp+8 and ...cfdp+8) where the correctly rounded value is ...cfcp+8 for both.
HYPOT_PAIR = ((7, 338), (10, 287))  # (column steps, row difference)


def libm_rounds_apart():
    """whether this host's libm rounds the two norms of HYPOT_PAIR to different doubles (the premise of the hypot-tie cases)"""
    (k1, u1), (k2, u2) = HYPOT_PAIR
    return libm_hypot(25 * k1, u1) != libm_hypot(25 * k2, u2)


_PROFILE = {}


def hypot_tie_profile():
    """(cached) 11 rows y_0..y_10 over consecutive scan columns (step s): the lines through points (0, 7) and (0, 10) have the two
    equal-norm directions of HYPOT_PAIR (in units of s = 25 columns), and four further points lie close to each line at
    distances whose sums are equal. So the two lines tie exactly under a correctly rounded hypot (the first, pair (0, 7), wins)
    while glibc's hypot makes the line through (0, 10) strictly better."""
    if "p" in _PROFILE:
        return _PROFILE["p"]
    (k1, u1), (k2, u2) = HYPOT_PAIR
    y = [None] * 11
    y[0], y[k1], y[k2] = 0, u1, u2
    # near the first line (338 k / 7) at k = 3, 4, 1, 6 and the second (287 k / 10) at k = 2, 5, 8, 9; integer distances
    # |338 k - 7 y| * 25 and |287 k - 10 y| * 25
    near1, near2 = (1, 3, 4, 6), (2, 5, 8, 9)
    best = None
    for choice in _choices(near1, near2):
        yy = list(y)
        for k, v in choice.items():
            yy[k] = v
        f = Fit(np.stack([np.arange(11) * 25, yy], 1), use_sqrt=True)
        g = Fit(np.stack([np.arange(11) * 25, yy], 1))
        if f.at_min == 2 and f.distinct == 2 and pair_of(f.winner, 11) == (0, k1) and pair_of(g.winner, 11) == (0, k2):
            best = yy
            break
    _PROFILE["p"] = best
    return best


def _choices(near1, near2):
    """row choices for the free points: within 4 rows of each line, ordered by total offset"""
    import itertools
    cand = {}
    for k in near1:
        c = 338 * k / 7
        cand[k] = sorted(range(math.floor(c) - 3, math.ceil(c) + 4), key=lambda v: abs(v - c))
    for k in near2:
        c = 287 * k / 10
        cand[k] = sorted(range(math.floor(c) - 3, math.ceil(c) + 4), key=lambda v: abs(v - c))
    keys = list(near1) + list(near2)
    for combo in itertools.product(*[cand[k][:4] for k in keys]):
        yield dict(zip(keys, combo))


def mirror_profile(n, rng, amp=3):
    """a tent over n columns with a mirror-symmetric perturbation: y_k = y_(n-1-k), so a line and its mirror image tie exactly
    (same |a|, |b| and the same multiset of distances)"""
    k = np.arange(n)
    tent = 40 * np.minimum(k, n - 1 - k)
    noise = rng.integers(-amp, amp + 1, n)
    noise = np.where(k < n - 1 - k, noise, noise[::-1])
    return tent + noise


# ---- the constructions the tests share ----
MIN_EXT = 10  # min_img_y_extent passed to detect_outline: every designed segment is longer


def hypot_outline_case():
    """640 x 480: the hypot-tie profile as frontRight (ySecond of columns W/2 + 25 k, k = 0..10), ten left scans on one row"""
    W, H = 640, 480
    y = hypot_tie_profile()
    right = [100 + v for v in y]
    img = outline_image(W, H, outline_segs(W, right, [120] * 10, y_first=20))
    return img, np.stack([W // 2 + 25 * np.arange(11), right], 1)


def hypot_front_case():
    """2048 x 1536: the hypot-tie profile scaled by two (column step 50, rows doubled: glibc's hypot is exact under scaling by
    two, so the same two directions tie) as the bottom rows of columns W/2 + 50 k; nothing left of W/2"""
    W, H = 2048, 1536
    y = hypot_tie_profile()
    bottoms = {W // 2 + 50 * k: 800 + 2 * v for k, v in enumerate(y)}
    return front_image(W, H, bottoms, top=780), np.array(sorted(bottoms.items()))


# Band path of the single-stage calls (band_setup, ssd_kernels_outline.cuh): the band is rows 0..H-1, staged in shared memory
# when H * (wpr + 1) words fit the dynamic allocation ssd_gpu_create makes: min(SSD_GPU_OUTLINE_SMEM_KB (default 32) KB, the
# whole image, the opt-in limit (227 KB on B200) minus the kernels' static shared memory (30464 bytes, ptxas) minus 1 KB),
# rounded down to 16 bytes; otherwise every probe reads the global bitmap.
SMEM_OPTIN, SMEM_STATIC = 227 * 1024, 30464


def band_path(W, H, smem_kb=None):
    """'smem' or 'global' for the single-stage band of a W x H frame under SSD_GPU_OUTLINE_SMEM_KB=smem_kb (None: unset);
    None when the band is within 8 KB of the limit (the static size may move with the build)"""
    full = H * ((W + 31) // 32 + 1) * 4
    want = 32 * 1024 if smem_kb is None else int(smem_kb) * 1024
    cap = SMEM_OPTIN - SMEM_STATIC - 1024
    if want < full and want < cap - 8192:
        return "global"
    if full <= want and full <= cap - 8192:
        return "smem"
    if full > cap + 8192:
        return "global"
    return None


def front_tent_case(W, H, n):
    """bottom rows of n consecutive columns W/2 + 50 k (nothing left of W/2): a mirror-symmetric tent with a perturbation, so
    the front-edge list has n points and a tie between two distinct lines at its minimum"""
    for seed in range(200):
        rng = np.random.default_rng(seed)
        amp = max(1, min(12, (H // 2 - 40) // max(1, n)))
        ys = H - 20 - mirror_profile(n, rng) * amp // 40 - 3
        pts = np.stack([W // 2 + 50 * np.arange(n), ys], 1)
        if Fit(pts).distinct >= 2:
            return front_image(W, H, {int(x): int(y) for x, y in pts}), pts
    raise AssertionError(f"no front-edge tie found for {W}x{H} n={n}")


FRONT_SIZES = [(640, 480, 6), (1348, 1108, 14), (4096, 3072, 27), (4096, 3072, 41)]


# (W, H, n): list lengths per frame size chosen to reach every residual branch of its class (n = nr, nl = n - 1)
MIRROR_SIZES = [(320, 240, 5), (320, 240, 7), (1348, 1108, 9), (1348, 1108, 13), (1348, 1108, 21), (1348, 1108, 27),
                (1352, 1108, 21), (1352, 1108, 27), (4096, 3072, 29), (4096, 3072, 45), (4096, 3072, 81)]


def mirror_case(W, H, n):
    """right front list: a mirror-symmetric tent of n points with an exact tie between two distinct lines at its minimum; left
    front list: another; back lists: one row (every pair ties at residual 0, so the first pair must win). Returns (img, right)."""
    base = 30
    for seed in range(200):
        rng = np.random.default_rng(seed)
        slope = max(1, min(40, (H - 2 * base) // max(1, n)))
        right = base + mirror_profile(n, rng) * slope // 40 + 3
        left = base + mirror_profile(n - 1, rng) * slope // 40 + 3
        f = Fit(np.stack([W // 2 + 25 * np.arange(n), right], 1))
        if f.distinct >= 2:
            return outline_image(W, H, outline_segs(W, right, left, y_first=5)), right
    raise AssertionError(f"no mirror tie found for {W}x{H} n={n}")


def decision_cases():
    """constructions for the decisions around the fit: name -> (img, n_scans the oracle must see). Scan extents exactly
    MIN_EXT (kept) and MIN_EXT - 1 (stops the scan); 2 scans (rejected before the fit) and 3 (the smallest fit); a plateau
    touching rows 0 and H - 1 and columns 0 and W - 1 (the erosion's border rule); widths whose scan columns land on column 0
    (W = 550: 275 - 25 * 11 = 0) and on column W - 1 (W = 552: 276 + 25 * 11 = 551)."""
    out = {}
    W, H = 640, 480
    c = W // 2
    prof = [200, 210, 220, 230]
    segs = outline_segs(W, prof, [205, 215], y_first=100)
    segs[c + 100] = (300, 300 + MIN_EXT)          # extent exactly MIN_EXT: kept
    out["extent_equal"] = (outline_image(W, H, segs), 7)
    segs = dict(segs)
    segs[c + 100] = (300, 300 + MIN_EXT - 1)      # one less: the right scan stops before it
    out["extent_one_less"] = (outline_image(W, H, segs), 6)
    out["two_scans"] = (outline_image(W, H, outline_segs(W, [200], [230], y_first=100)), 2)
    out["three_scans"] = (outline_image(W, H, outline_segs(W, [200, 240], [230], y_first=100)), 3)
    img = np.zeros((H, W), np.uint8)
    img[:, :] = 255
    img[H // 2:, : W // 3] = 0                     # every scanned column touches row 0; columns 0 and W - 1 are set
    img[H - 40:, W // 3:] = 255
    out["touching_borders"] = (img, len(range(c, W, 25)) + len(range(c - 25, -1, -25)))
    for W2, tag in ((550, "scan_on_column_0"), (552, "scan_on_column_W-1")):
        c2 = W2 // 2
        nr, nl = len(range(c2, W2, 25)), len(range(c2 - 25, -1, -25))
        right = [150 + 7 * k for k in range(nr)]
        left = [160 + 5 * k for k in range(nl)]
        out[tag] = (outline_image(W2, H, outline_segs(W2, right, left, y_first=(list(range(20, 20 + 3 * nr, 3)),
                                                                                  list(range(30, 30 + 2 * nl, 2))))), nr + nl)
    return out
