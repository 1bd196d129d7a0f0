"""The filter stage at every bird's-eye width class its kernels branch on, and process() at reduced scales.

The filter kernels work on pair-packed planes: packed column x holds image columns x and x + p2, p2 = 32 * ceil(bv_w /
64), so 2 * p2 - bv_w high lanes lie beyond the image (0 to 62).  The erosion, the dilation and the threshold windows
read across the seam between the two strips through column halos of LT_HALO_X = 32 entries that three producers stitch
(the plane store, the warp and the erosion epilogue).  The morphology runs in tiles of 192 packed columns; the
threshold kernels in 32-row tiles, 96- or 288-row bands, 64-row bands and 8- or 32-row bands with 28 mask words per
warp, and the last mask word of a row may be partial.  The shipped 1080x1100 view takes one remainder of each; the
table below takes the others, down to the smallest view lt_create accepts (66x16: 62 high lanes beyond the image) and
up to the widest (the prefix-sum row kernel at its shared-memory limit).  At 64 columns (p2 = 32) every packed column
would feed both seam halos, which the erosion epilogue does not write: lt_create refuses it.

Inputs are adversarial bird's-eye images fed through lt_filter_lane_points: impulses and 2x2 dots of both polarities
at the corners, edge rows and columns and around the seam, plateaus exactly the shape of the 29x29 and 55x55 ellipses
(they survive the opening) and one column narrower (they do not), random ellipse blobs, salt and pepper, bright edges
and stripes across the seam.  Their colours run from (0, 0, 255) to (255, 255, 0), so the R plane and the Lab-b plane
(20 .. 223) both carry the pattern.  Every stream is checked bit for bit: the R and Lab-b planes and the merged
threshold mask against the NumPy oracle, the top-hats against cv2.morphologyEx called directly, the final mask against
the cv2 oracle.

The last tests run process() at half and quarter scale (540x550 and 270x275 views, the second of odd height) with the
pixel-valued options and validity windows scaled, against the oracle; below a view width of 720 the hard-coded second
attempt's ignore_sides = 360 leaves the histogram slices empty or reversed.  And lt_create refuses odd widths and
widths at which a threshold kernel could not launch, on both sides of the limit."""
import os
import re
import time
import warnings

import numpy as np
import pytest

from _oracle_pool import frame_from_spec
from lane_tracker_b200 import synth
from oracle.tracker import OracleLaneTracker

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

FIT_RTOL = 1e-6
WIDEST_B200 = 3614                  # widest accepted view at the 227 KB shared-memory opt-in limit of a B200
OPTIN_B200 = 227 * 1024


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)        # the launcher's own band split, unless a test pins one
    t0 = time.perf_counter()
    yield
    print("\ntest_gpu_filter_geometry: %.1f s wall in this module" % (time.perf_counter() - t0))


@pytest.fixture(scope="module")
def widest(torch_mod):
    """The widest bird's-eye view lt_create accepts on this device, from its refusal of a wider one."""
    from lane_tracker_b200 import BatchedLaneTracker, _lib
    with pytest.raises(_lib.LaneTrackerError, match="unsupported geometry") as e:
        BatchedLaneTracker(1, **calibration(32766, 16))
    w = int(re.search(r"at most (\d+)", str(e.value)).group(1))
    if torch_mod.cuda.get_device_properties(0).shared_memory_per_block_optin == OPTIN_B200:
        assert w == WIDEST_B200, w
    return w


def calibration(W, H):
    """The shipped camera with its own bird's-eye size: M and Minv rescaled anisotropically to W x H."""
    cal = synth.shipped_calibration()
    sx, sy = W / synth.WARPED_SIZE[0], H / synth.WARPED_SIZE[1]
    S, Si = np.diag([sx, sy, 1.0]), np.diag([1.0 / sx, 1.0 / sy, 1.0])
    M, Minv = cal["warp_matrices"]
    cal.update(warped_size=(W, H), warp_matrices=(S @ M, Minv @ Si), mpp_conversion=(synth.MPPV / sy, synth.MPPH / sx))
    return cal


def p2_of(W):
    return 32 * ((W + 63) // 64)


# ---- adversarial bird's-eye images ---------------------------------------------------------------------------------

def level(v):
    """RGB of grey level v in [0, 255]: R = v and Lab-b from 20 (v = 0, blue) to 223 (v = 255, yellow)."""
    v = np.asarray(v, dtype=np.int64)
    return np.stack([v, v, 255 - v], axis=-1).astype(np.uint8)


def _ellipse(k):
    return cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k)).astype(bool)


def _paste(img, mask, y0, x0, val):
    """img[y0 + i, x0 + j] = val where mask[i, j], clipped to the image."""
    H, W = img.shape[:2]
    h, w = mask.shape
    ya, xa = max(y0, 0), max(x0, 0)
    yb, xb = min(y0 + h, H), min(x0 + w, W)
    if ya >= yb or xa >= xb:
        return
    sub = mask[ya - y0:yb - y0, xa - x0:xb - x0]
    img[ya:yb, xa:xb][sub] = val


def img_impulses(W, H, rng):
    """Single pixels and 2x2 dots of both polarities at the corners, rows 0, 1, H-2, H-1 and columns 0, 1, 13-15,
    26-28, p2-28 .. p2+27 and W-1, on a mid-grey background."""
    img = np.full((H, W), int(rng.integers(90, 170)), np.int64)
    p2 = p2_of(W)
    cols = sorted({c for c in [0, 1, 13, 14, 15, 26, 27, 28, W - 1] + list(range(p2 - 28, p2 + 28)) if 0 <= c < W})
    rows = sorted({0, 1, H - 2, H - 1})
    for i, y in enumerate(rows):
        for j, x in enumerate(cols[i % 3::3]):
            img[y, x] = 255 if (i + j) % 2 else 0
    mid = list(range(3, H - 3, 5))
    for i, y in enumerate(mid):
        for j, x in enumerate(cols[(i + 1) % 4::4]):
            v = 0 if (i + j) % 2 else 255
            img[y:y + 2, x:x + 2] = v
    for y, x in ((0, 0), (0, W - 2), (H - 2, 0), (H - 2, W - 2)):
        img[y:y + 2, x:x + 2] = 255 - img[y, x]
    return level(img)


def img_plateaus(W, H, rng):
    """Bright plateaus exactly the shape of the 29x29 and 55x55 ellipses and the same shapes one column narrower,
    across the seam, at the left and right edges and in the middle, on a dark background."""
    img = np.full((H, W), int(rng.integers(0, 40)), np.int64)
    p2 = p2_of(W)
    hi = int(rng.integers(200, 256))
    shapes = [_ellipse(29), _ellipse(55), _ellipse(29)[:, :-1], _ellipse(55)[:, :-1]]
    spots = [(p2 - 14, H // 2 - 14), (0, 0), (W - 55, H - 55), (W // 4, H // 3), (3 * W // 4 - 27, 0),
             (p2 - 40, H - 29), (p2 + 3, 2)]
    for i, (x0, y0) in enumerate(spots):
        _paste(img, shapes[(i + int(rng.integers(0, 4))) % 4], y0, x0, hi - 5 * i)
    return level(img)


def img_blobs(W, H, rng):
    """Ellipse blobs of diameters 3 .. 80 at random levels on a background of random level."""
    img = np.full((H, W), int(rng.integers(0, 256)), np.int64)
    for _ in range(max(8, W * H // 1500)):
        d = int(rng.integers(3, 81))
        m = _ellipse(d)
        _paste(img, m, int(rng.integers(-d // 2, H)), int(rng.integers(-d // 2, W)), int(rng.integers(0, 256)))
    return level(img)


def img_salt_pepper(W, H, rng, density):
    img = np.full((H, W), int(rng.integers(60, 200)), np.int64)
    hit = rng.random((H, W)) < density
    img[hit] = np.where(rng.random(int(hit.sum())) < 0.5, 0, 255)
    return level(img)


def img_edges(W, H, rng):
    """Bright first and last rows and columns, vertical stripes of widths 1 .. 4 across the seam and horizontal
    stripes, on a dark background."""
    img = np.full((H, W), int(rng.integers(0, 30)), np.int64)
    img[0, :] = img[-1, :] = 255
    img[:, 0] = img[:, -1] = 250
    p2 = p2_of(W)
    x = max(0, p2 - 40)
    w = 1
    while x < min(W - 1, p2 + 40):
        img[1:-1, x:x + w] = 240 - 3 * w
        x += 2 * w + 1
        w = w % 4 + 1
    img[H // 2:H // 2 + 2, :] = 230
    if H > 8:
        img[3, ::3] = 255
    return level(img)


KINDS = ["impulses", "plateaus", "blobs", "salt1", "salt50", "edges"]


def make_image(kind, W, H, seed):
    rng = np.random.default_rng(seed)
    if kind == "impulses":
        return img_impulses(W, H, rng)
    if kind == "plateaus":
        return img_plateaus(W, H, rng)
    if kind == "blobs":
        return img_blobs(W, H, rng)
    if kind == "salt1":
        return img_salt_pepper(W, H, rng, 0.01)
    if kind == "salt50":
        return img_salt_pepper(W, H, rng, 0.5)
    return img_edges(W, H, rng)


def test_adversarial_images_reach_both_planes_and_extremes():
    """The image set itself: Lab-b reaches 20 and 223, the planes carry the same pattern, and the ellipse plateaus
    survive a cv2 opening while the narrower ones do not."""
    b = cv2.cvtColor(level(np.arange(256))[None], cv2.COLOR_RGB2LAB)[0, :, 2].astype(int)
    assert b[0] == 20 and b[-1] == 223 and (np.diff(b) >= 0).all()       # Lab-b follows R
    for kind in KINDS:
        bv = make_image(kind, 130, 56, 1)
        assert np.array_equal(bv[:, :, 0], bv[:, :, 1]) and bv[:, :, 0].min() < bv[:, :, 0].max(), kind
    for k in (29, 55):
        se = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))
        img = np.zeros((k + 20, k + 20), np.uint8)
        img[10:10 + k, 10:10 + k][_ellipse(k)] = 200
        assert cv2.morphologyEx(img, cv2.MORPH_OPEN, se).max() == 200
        img[:] = 0
        img[10:10 + k, 10:10 + k - 1][_ellipse(k)[:, :-1]] = 200
        assert cv2.morphologyEx(img, cv2.MORPH_OPEN, se).max() == 0


# ---- A-C. the filter at every width class ----------------------------------------------------------------------------

# (W, H): what the size reaches
GEOMETRIES = [
    (66, 16),        # smallest accepted size; shorter than either ellipse
    (66, 17),        # p2 = 64 with 62 high lanes beyond the image; odd height
    (128, 55),       # no lanes beyond the image; height = 55
    (130, 56),       # p2 = 96, 62 lanes beyond
    (384, 96),       # p2 = 192: exactly one morphology tile; height = the few-streams vertical band
    (386, 97),       # a second tile of 32 columns; band + 1
    (1088, 289),     # p2 = 544, no lanes beyond; 288-row band + 1
    (1080, 1100),    # shipped
]

# (filter_type, ksize_r, C_r, ksize_b, C_b, mask_noise, ksize_noise, C_noise, noise_thresh)
DEFAULTS = ("bilateral", 15, 8, 35, 5, False, 65, 10, 135)
OPTIONS = [
    DEFAULTS,
    ("bilateral", 1, 0, 2, 1, False, 65, 10, 135),
    ("bilateral", 2, 3, 1, 0, False, 65, 10, 135),
    ("bilateral", 40, 8, 41, 5, False, 65, 10, 135),       # TMA column kernel / cp.async ring
    ("bilateral", 41, 2, 40, 9, False, 65, 10, 135),
    ("bilateral", 127, 3, 128, 2, False, 65, 10, 135),     # packed row kernel / prefix-sum row kernel
    ("bilateral", 128, 1, 127, 5, False, 65, 10, 135),     # 127 * 255 + 5 * 127 >= 2^15: unpacked
    ("bilateral", 255, 0, 255, 0, False, 65, 10, 135),
    ("bilateral", 100, 80, 41, 5, False, 65, 10, 135),     # unpacked at k <= 127
    ("neighborhood", 3, 5, 255, 2, False, 65, 10, 135),
    ("neighborhood", 35, 5, 3, 0, False, 65, 10, 135),
    ("neighborhood", 255, 10, 35, 5, False, 65, 10, 135),
    ("bilateral", 15, 8, 35, 5, True, 65, 10, 135),
    ("bilateral", 15, 8, 35, 5, True, 255, 0, 128),
]
assert {1, 2, 40, 41, 127, 128, 255} <= {o[k] for o in OPTIONS if o[0] == "bilateral" for k in (1, 3)}
assert any(o[1] * 255 + o[2] * o[1] >= 2 ** 15 and o[1] <= 127 for o in OPTIONS if o[0] == "bilateral")


class _Oracle:
    """Oracle results of one image, computed once per option set."""

    def __init__(self, cal, bv):
        self.cal, self.bv = cal, bv
        self.r_plane = np.ascontiguousarray(bv[:, :, 0])
        o = OracleLaneTracker(**cal)
        o.filter_lane_points(bv, *DEFAULTS)
        self.b_plane = o.trace["b_plane"]
        b_cv = cv2.cvtColor(bv, cv2.COLOR_RGB2LAB)[:, :, 2]
        self.r_top = cv2.morphologyEx(self.r_plane, cv2.MORPH_TOPHAT, cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (29, 29)))
        self.b_top = cv2.morphologyEx(b_cv, cv2.MORPH_TOPHAT, cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (55, 55)))
        self._res = {}

    def get(self, opt):
        if opt not in self._res:
            o = OracleLaneTracker(**self.cal)
            o.filter_lane_points(self.bv, *opt)
            mask = OracleLaneTracker(**self.cal, backend="cv2").filter_lane_points(self.bv, *opt)
            self._res[opt] = (o.trace["merged"], mask)
        return self._res[opt]


_ORACLES = {}


def _oracle(cal, W, H, kind, seed):
    key = (W, H, kind, seed)
    if key not in _ORACLES:
        _ORACLES[key] = _Oracle(cal, make_image(kind, W, H, seed))
    return _ORACLES[key]


def _mism(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    d = np.argwhere(a != b)
    return "%d mismatches, first at (row, col) %s" % (len(d), d[:4].tolist()) if len(d) else ""


def _run_filter(torch, bt, oracles, opts, tag, planes=True):
    bv = torch.as_tensor(np.stack([o.bv for o in oracles])).cuda()
    for opt in opts:
        got = bt.filter_lane_points(bv, *opt).cpu().numpy()
        for s, o in enumerate(oracles):
            t = (tag, opt, s)
            if planes and opt == opts[0]:
                assert not _mism(bt.debug_read("r_plane", s), o.r_plane), (t, "r_plane", _mism(bt.debug_read("r_plane", s), o.r_plane))
                assert not _mism(bt.debug_read("b_plane", s), o.b_plane), (t, "b_plane", _mism(bt.debug_read("b_plane", s), o.b_plane))
            if opt[0] == "bilateral":
                m = _mism(bt.debug_read("r_tophat", s), o.r_top)
                assert not m, (t, "r_tophat", m)
                m = _mism(bt.debug_read("b_tophat", s), o.b_top)
                assert not m, (t, "b_tophat", m)
            merged, mask = o.get(opt)
            m = _mism(bt.debug_read("merged", s), merged)
            assert not m, (t, "merged", m)
            m = _mism(got[s], mask)
            assert not m, (t, "mask", m)


def _check_geometry(bt, W, H):
    g = bt.geometry
    assert (g["plane_width"], g["mask_words"]) == (p2_of(W), 2 * p2_of(W) // 32), (W, H, g)


@pytest.mark.parametrize("S", [1, 17])
@pytest.mark.parametrize("W,H", GEOMETRIES, ids=["%dx%d" % g for g in GEOMETRIES])
def test_filter_geometry_matches_oracle(torch_mod, W, H, S):
    """Every option set of the table on S streams of distinct adversarial images at one bird's-eye size: planes,
    top-hats, merged threshold mask and final mask of every stream bit for bit.  At the shipped size the 17-stream
    batch runs the defaults and both mask_noise sets (the other options run on one stream)."""
    from lane_tracker_b200 import BatchedLaneTracker
    cal = calibration(W, H)
    seeds = [(KINDS[(i + W + H) % len(KINDS)], 1000 * W + 10 * H + i) for i in range(S)]
    oracles = [_oracle(cal, W, H, k, sd) for k, sd in seeds]
    opts = OPTIONS if (S == 1 or W * H < 500_000) else [o for o in OPTIONS if o == DEFAULTS or o[5]]
    bt = BatchedLaneTracker(S, **cal)
    try:
        _check_geometry(bt, W, H)
        _run_filter(torch_mod, bt, oracles, opts, (W, H, S))
    finally:
        bt.close()


@pytest.mark.parametrize("bands", ["1,1", "24,10"])
@pytest.mark.parametrize("S", [1, 17])
@pytest.mark.parametrize("W,H", [g for g in GEOMETRIES if g[1] <= 17], ids=["%dx%d" % g for g in GEOMETRIES if g[1] <= 17])
def test_filter_short_views_pinned_bands(torch_mod, W, H, S, bands):
    """Views shorter than either ellipse with the morphology band split pinned: one band, and more bands than rows
    (empty bands that only warm up)."""
    from lane_tracker_b200 import BatchedLaneTracker
    cal = calibration(W, H)
    oracles = [_oracle(cal, W, H, KINDS[i % len(KINDS)], 7000 + 10 * W + i) for i in range(S)]
    os.environ["LT_MORPH_BANDS"] = bands
    try:
        bt = BatchedLaneTracker(S, **cal)
        try:
            _check_geometry(bt, W, H)
            _run_filter(torch_mod, bt, oracles, [DEFAULTS, OPTIONS[7]], (W, H, S, bands))
            assert bt.morph_bands() == tuple(int(v) for v in bands.split(","))
        finally:
            bt.close()
    finally:
        os.environ.pop("LT_MORPH_BANDS", None)


@pytest.mark.parametrize("S", [1, 17])
def test_filter_at_the_widest_view(torch_mod, widest, S):
    """The widest view lt_create accepts (40 rows): the packed row kernel up to k = 127, the prefix-sum row kernel
    for k > 127 and for unpacked lanes at k <= 127, the box row kernel at block 255."""
    from lane_tracker_b200 import BatchedLaneTracker
    W, H = widest, 40
    cal = calibration(W, H)
    oracles = [_oracle(cal, W, H, KINDS[i % len(KINDS)], 9000 + i) for i in range(S)]
    bt = BatchedLaneTracker(S, **cal)
    try:
        _check_geometry(bt, W, H)
        _run_filter(torch_mod, bt, oracles, OPTIONS, (W, H, S))
    finally:
        bt.close()


# ---- E. geometry refusals --------------------------------------------------------------------------------------------

def test_create_refuses_odd_and_too_wide_views(torch_mod, widest):
    """lt_create refuses an odd bird's-eye width, a width of 64 (one pair-plane column would feed both seam halos)
    and any width beyond the widest at which every threshold kernel can launch with every kernel size the parameter
    checks accept; it accepts the widest and the narrowest."""
    from lane_tracker_b200 import BatchedLaneTracker, _lib
    for W, H in ((64, 16), (65, 16), (1081, 1100), (widest - 1, 16), (widest + 2, 16), (widest + 64, 16), (32766, 16)):
        with pytest.raises(_lib.LaneTrackerError, match="unsupported geometry"):
            BatchedLaneTracker(1, **calibration(W, H))
    for W, H in ((66, 16), (widest, 16), (1080, 1100)):
        BatchedLaneTracker(1, **calibration(W, H)).close()


# ---- D. process() at reduced scales ----------------------------------------------------------------------------------

def _scaled_options(s):
    r = lambda v: max(1, int(round(v * s)))
    return dict(ksize_r=r(15), ksize_b=r(35), window_width=r(30), window_height=r(40), search_range=r(20),
                ignore_sides=r(360), ignore_bottom=r(30), bandwidth=r(25), ksize_noise=r(65))


def _scaled_validity(s):
    return dict(min_dist_y1=150 * s, max_dist_y1=230 * s, min_dist_y2=110 * s, max_dist_y2=230 * s,
                min_dist_y3=80 * s, max_dist_y3=200 * s, tangent_thresh=0.25)


def _check_process(bt, res, out, s, o, want, tag, edge=0):
    att = o.trace["attempts"]
    last = att[-1]
    assert int(res["counter"]) == o.counter, tag
    assert int(res["success"]) == o.success, tag
    assert int(res["attempts"]) == len(att), tag
    assert int(res["search_mode"]) == (1 if last["mode"] == "bs" else 0), tag
    assert bool(res["detected_pixels"]) == bool(o.detected_pixels), tag
    assert bool(res["valid_lane_lines"]) == bool(o.valid_lane_lines), tag
    assert int(res["last_detection"]) == o.last_detection, tag
    assert bool(res["first_detected"]) == bool(att[0]["detected"]), tag
    assert bool(res["first_valid"]) == bool(att[0]["valid"]), tag
    assert not _mism(bt.debug_read("mask", s), last["mask"]), (tag, _mism(bt.debug_read("mask", s), last["mask"]))
    if last["detected"]:
        sides, _ = bt.read_capture(s, len(att) - 1)
        assert np.array_equal(sides[0][0], last["left_y"]) and np.array_equal(sides[0][1], last["left_x"]), tag
        assert np.array_equal(sides[1][0], last["right_y"]) and np.array_equal(sides[1][1], last["right_x"]), tag
        np.testing.assert_allclose(res["left_fit"], last["left_fit"], rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_fit"], last["right_fit"], rtol=FIT_RTOL, err_msg=str(tag))
    if o.valid_lane_lines:
        assert int(res["average_curve_radius"]) == int(o.average_curve_radius), tag
        assert float(res["eccentricity"]) == pytest.approx(o.eccentricity, rel=1e-12, abs=1e-15), tag
        np.testing.assert_allclose(res["left_avg"], o.left_avg_coeffs, rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_avg"], o.right_avg_coeffs, rtol=FIT_RTOL, err_msg=str(tag))
    bad = np.argwhere((out != want).any(axis=-1))
    if edge:        # text clipped by the right frame edge (DESIGN.md section 1): its last column, in the text rows
        r0, r1 = bt.text_rows
        bad = bad[(bad[:, 1] < out.shape[1] - edge) | (bad[:, 0] < r0) | (bad[:, 0] >= r1)]
    assert len(bad) == 0, (tag, len(bad), [(tuple(yx), out[tuple(yx)].tolist(), want[tuple(yx)].tolist()) for yx in bad[:6]])


# Road videos whose lane-pixel sets are never exactly straight at that scale.  With lines 2.5 px wide (quarter scale)
# most seeds give some frame whose pixel set fits a straight line exactly: the quadratic coefficient, the curve
# radius (1 / |2a|, some 10^12 m) and an eccentricity of exactly 0 are then fp64 round-off of the least-squares
# solve, in the reference as anywhere else.  (synth.RoadVideo avoids such frames at the shipped scale.)
_SEEDS = {0.5: (30, 31), 0.25: (30, 105)}


@pytest.mark.parametrize("scale", [0.5, 0.25])
def test_process_at_reduced_scale(torch_mod, scale):
    """Three streams, six frames, at a reduced scale with the pixel-valued options and the validity windows scaled:
    two synthetic road videos (sliding-window search, band search, lane polygon, overlay, clipped text) and one stream
    of noise and blank frames that fails every frame and takes the hard-coded second attempt (ignore_sides = 360,
    wider than half the view).  Records, masks, captured pixel sets and annotated frames bit for bit against the cv2
    oracle, annotated frames also against the NumPy oracle."""
    from lane_tracker_b200 import BatchedLaneTracker
    torch = torch_mod
    cal = synth.shipped_calibration(scale)
    opts = _scaled_options(scale)
    V = _scaled_validity(scale)
    T = 6
    plans = [[["synth", seed, t] for t in range(T)] for seed in _SEEDS[scale]]
    plans.append([["noise", 800]] + [["blank", 35 + 20 * t] for t in range(1, T)])
    S = len(plans)
    vd = dict(min_d1=V["min_dist_y1"], max_d1=V["max_dist_y1"], min_d2=V["min_dist_y2"], max_d2=V["max_dist_y2"],
              min_d3=V["min_dist_y3"], max_d3=V["max_dist_y3"], tan=V["tangent_thresh"])
    oracles, np_oracles = [], []
    for _ in range(S):
        o = OracleLaneTracker(**cal, backend="cv2")
        o.validity = dict(vd)
        oracles.append(o)
        o = OracleLaneTracker(**cal)
        o.validity = dict(vd)
        np_oracles.append(o)
    # At quarter scale the text runs past the 320-column frame.  cv2.putText shades the last frame column of a clipped
    # anti-aliased stroke in a way the glyph sprites (of the kernel and of the NumPy oracle) do not model (DESIGN.md
    # section 1): that column of the text rows is compared with the NumPy oracle only.
    edge = 1 if cal["img_size"][0] < 460 else 0
    bt = BatchedLaneTracker(S, **cal)
    bt.set_validity(**V)
    bt.set_capture(True)
    n_valid = n_band = n_retry = 0
    try:
        for t in range(T):
            frames = np.stack([frame_from_spec(plans[s][t], scale) for s in range(S)])
            d = torch.as_tensor(frames).cuda()
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, **opts)
                wants = [oracles[s].process(frames[s].copy(), **opts) for s in range(S)]
                np_wants = [np_oracles[s].process(frames[s].copy(), **opts) for s in range(S)]
            out = out.cpu().numpy()
            for s in range(S):
                o = oracles[s]
                for a in o.trace["attempts"]:       # the data are what the seeds above promise
                    assert not a["detected"] or min(abs(a["left_fit"][0]), abs(a["right_fit"][0])) > 1e-9, (scale, t, s)
                _check_process(bt, res[s], out[s], s, o, wants[s], (scale, t, s), edge)
                assert np.array_equal(out[s], np_wants[s]), (scale, t, s, int((out[s] != np_wants[s]).any(-1).sum()))
                n_valid += bool(o.valid_lane_lines)
                n_band += o.trace["attempts"][-1]["mode"] == "bs"
                n_retry += s == S - 1 and len(o.trace["attempts"]) == 2
    finally:
        bt.close()
    assert n_valid >= 5 and n_band >= 5, (n_valid, n_band)
    assert n_retry == T, n_retry                    # the failing stream took the second attempt on every frame
