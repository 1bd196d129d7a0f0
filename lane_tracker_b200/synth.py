"""Synthetic 1280x720 road video (host-side test/bench data, not on the hot path).

Recipe from SURVEY.md section 8(d): textured pavement with a solid yellow left
line and a dashed white right line 180 px apart in the bird's-eye view, a
slowly varying quadratic lane shape, projected into the camera view with the
shipped homography.  Under the reference's *unmodified* validity thresholds
(lane_tracker.py:588-593) this yields a sliding-window search on frame 0 and
band-search tracking afterwards.

Everything is deterministic in (seed, t): ``rng = default_rng(seed*100003 + t)``.
"""
from __future__ import annotations

import numpy as np

# shipped calibration (cam_calib.p / warp_params.p of the reference, SURVEY.md B.1)
CAM_MATRIX = np.array([[1154.3293544733699, 0.0, 669.68287497444635],
                       [0.0, 1148.4715517793131, 385.86265402405462],
                       [0.0, 0.0, 1.0]])
DIST_COEFFS = np.array([[-0.24180123999440323, -0.047799949862003206, -0.0011385469776010269,
                         -0.00011245666608284012, 0.018317194299296482]])
WARP_M = np.array([[-0.16192154913816159, -1.2786360662302192, 641.41214769155897],
                   [-1.6944778913341452e-14, -3.0195465710372815, 1380.891412308576],
                   [-1.474514954580286e-17, -0.002377623877779378, 1.0]])
WARP_MINV = np.array([[0.53932875397536018, -0.50395955194543518, 349.98140303318553],
                      [8.8817841970012523e-16, -0.3311755511876282, 457.31747460155714],
                      [-3.0357660829594124e-18, -0.00078741089824045977, 1.0]])
IMG_SIZE = (1280, 720)
WARPED_SIZE = (1080, 1100)
MPPV = 0.03048
MPPH = 0.0146304


def shipped_calibration(scale=1.0):
    """Constructor arguments of ``LaneTracker`` for the shipped calibration.

    ``scale`` rescales image and bird's-eye sizes (BASELINE.json config 5):
    ``K' = S K``, ``M' = S M S^-1``, ``Minv' = S Minv S^-1`` (SURVEY.md 8(d)).
    """
    if scale == 1.0:
        return dict(img_size=IMG_SIZE, warped_size=WARPED_SIZE, cam_matrix=CAM_MATRIX.copy(),
                    dist_coeffs=DIST_COEFFS.copy(), warp_matrices=(WARP_M.copy(), WARP_MINV.copy()),
                    mpp_conversion=(MPPV, MPPH))
    S = np.diag([scale, scale, 1.0])
    Si = np.diag([1.0 / scale, 1.0 / scale, 1.0])
    isz = (int(round(IMG_SIZE[0] * scale)), int(round(IMG_SIZE[1] * scale)))
    wsz = (int(round(WARPED_SIZE[0] * scale)), int(round(WARPED_SIZE[1] * scale)))
    return dict(img_size=isz, warped_size=wsz, cam_matrix=S @ CAM_MATRIX,
                dist_coeffs=DIST_COEFFS.copy(), warp_matrices=(S @ WARP_M @ Si, S @ WARP_MINV @ Si),
                mpp_conversion=(MPPV / scale, MPPH / scale))


class RoadVideo:
    """Frame generator for one stream; ``frame(t)`` -> uint8 RGB [h, w, 3]."""

    def __init__(self, seed=0, scale=1.0, separation=180.0, calibration=None):
        """calibration: constructor arguments of ``LaneTracker`` (``shipped_calibration`` form) whose warp ``M`` renders
        the road into the frame, for cameras mounted otherwise (None: ``shipped_calibration(scale)``).  The frames have
        no lens distortion either way."""
        cal = shipped_calibration(scale) if calibration is None else calibration
        self.seed = int(seed)
        self.scale = float(scale)
        self.separation = separation * scale
        self.w, self.h = cal["img_size"]
        self.bw, self.bh = cal["warped_size"]
        M = cal["warp_matrices"][0]
        xs, ys = np.meshgrid(np.arange(self.w, dtype=np.float64), np.arange(self.h, dtype=np.float64))
        d = M[2, 0] * xs + M[2, 1] * ys + M[2, 2]
        d = np.where(np.abs(d) < 1e-9, 1e-9, d)   # the road half of the frame has d < 0
        bx = (M[0, 0] * xs + M[0, 1] * ys + M[0, 2]) / d
        by = (M[1, 0] * xs + M[1, 1] * ys + M[1, 2]) / d
        self._inside = (bx >= 0) & (bx <= self.bw - 1) & (by >= 0) & (by <= self.bh - 1)
        bx = np.clip(bx, 0, self.bw - 1)
        by = np.clip(by, 0, self.bh - 1)
        x0 = np.minimum(bx.astype(np.int64), self.bw - 2)
        y0 = np.minimum(by.astype(np.int64), self.bh - 2)
        self._fx = (bx - x0).astype(np.float32)[..., None]
        self._fy = (by - y0).astype(np.float32)[..., None]
        self._i00 = (y0 * self.bw + x0).ravel()
        # quarter-resolution -> full-resolution bilinear upsample indices
        qh, qw = (self.bh + 3) // 4 + 1, (self.bw + 3) // 4 + 1
        self._q = (qh, qw)
        yy = np.arange(self.bh) / 4.0
        xx = np.arange(self.bw) / 4.0
        self._qy0 = yy.astype(np.int64)
        self._qx0 = xx.astype(np.int64)
        self._qfy = (yy - self._qy0).astype(np.float32)[:, None]
        self._qfx = (xx - self._qx0).astype(np.float32)[None, :]

    def lane_centres(self, t):
        """BV x of the left/right line centre on every BV row (float64 [bh])."""
        s = self.scale
        y = (np.arange(self.bh, dtype=np.float64) - (self.bh - 1)) / s
        a = 6e-5 * np.sin((t + 11.0) / 60.0)      # phase offsets: never an exactly straight line (a = b = 0 makes
        b = -0.05 * np.sin((t + 5.0) / 90.0)      # the reference's curve radius 1/|2a| a pure round-off product)
        c0 = 450.37 + 15.0 * np.sin(t / 45.0)     # never pixel-symmetric: an exactly integral fit makes the
                                                  # int() truncations downstream depend on fp64 round-off
        xl = (a * y * y + b * y + c0) * s
        return xl, xl + self.separation

    def bird_view(self, t):
        rng = np.random.default_rng(self.seed * 100003 + int(t))
        qh, qw = self._q
        q = rng.normal(95.0, 6.0, size=(qh, qw)).astype(np.float32)
        y0, x0 = self._qy0, self._qx0
        top = q[y0][:, x0] * (1 - self._qfx) + q[y0][:, x0 + 1] * self._qfx
        bot = q[y0 + 1][:, x0] * (1 - self._qfx) + q[y0 + 1][:, x0 + 1] * self._qfx
        base = top * (1 - self._qfy) + bot * self._qfy
        base += rng.normal(0.0, 3.0, size=base.shape).astype(np.float32)
        bv = np.stack([base - 2.0, base, base + 4.0], axis=2)
        xl, xr = self.lane_centres(t)
        s = self.scale
        xs = np.arange(self.bw, dtype=np.float64)[None, :]
        left = np.abs(xs - xl[:, None]) <= 5.0 * s
        rows = np.arange(self.bh, dtype=np.float64)[:, None]
        dash_on = np.mod(rows / s + 7.0 * t, 160.0) < 70.0
        right = (np.abs(xs - xr[:, None]) <= 5.0 * s) & dash_on
        bv[left] = (230.0, 200.0, 60.0)
        bv[right] = (240.0, 240.0, 240.0)
        return np.clip(np.rint(bv), 0, 255).astype(np.uint8)

    def frame(self, t):
        bv = self.bird_view(t).reshape(-1, 3).astype(np.float32)
        i = self._i00
        bw = self.bw
        shp = (self.h, self.w, 3)
        p00 = bv[i].reshape(shp)
        p01 = bv[i + 1].reshape(shp)
        p10 = bv[i + bw].reshape(shp)
        p11 = bv[i + bw + 1].reshape(shp)
        fx, fy = self._fx, self._fy
        cam = (p00 * (1 - fx) + p01 * fx) * (1 - fy) + (p10 * (1 - fx) + p11 * fx) * fy
        out = np.clip(np.rint(cam), 0, 255).astype(np.uint8)
        out[~self._inside] = (130, 160, 200)
        return out


def render_streams(n_streams, n_frames, scale=1.0, first_seed=0, workers=None):
    """uint8 array [n_streams, n_frames, h, w, 3]; stream s uses seed first_seed+s."""
    jobs = [(first_seed + s, n_frames, scale) for s in range(n_streams)]
    if workers is None or workers <= 1 or n_streams == 1:
        return np.stack([_render_one(j) for j in jobs])
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(workers, n_streams)) as pool:
        return np.stack(pool.map(_render_one, jobs))


def _render_one(job):
    seed, n_frames, scale = job
    v = RoadVideo(seed, scale)
    return np.stack([v.frame(t) for t in range(n_frames)])


def rgb_to_nv12(frames):
    """RGB frames uint8 [..., H, W, 3] -> NV12 uint8 [..., H * 3 / 2, W] (H and W even): ITU-R BT.601 limited range,
    each chroma sample the mean of its 2x2 block, rounded to nearest -- what a camera or a decoder delivers for road
    video.  (The inverse, cv2.cvtColor(COLOR_YUV2RGB_NV12), is lossy: converting back does not give the input.)"""
    rgb = np.asarray(frames)
    if rgb.dtype != np.uint8 or rgb.ndim < 3 or rgb.shape[-1] != 3 or rgb.shape[-3] % 2 or rgb.shape[-2] % 2:
        raise ValueError("rgb_to_nv12: expected uint8 [..., H, W, 3] with even H and W")
    h, w = rgb.shape[-3], rgb.shape[-2]
    lead = rgb.shape[:-3]
    f = rgb.astype(np.float64)
    r, g, b = f[..., 0], f[..., 1], f[..., 2]
    y = 16 + (65.481 * r + 128.553 * g + 24.966 * b) / 255
    cb = 128 + (-37.797 * r - 74.203 * g + 112.0 * b) / 255
    cr = 128 + (112.0 * r - 93.786 * g - 18.214 * b) / 255
    sub = lambda c: c.reshape(lead + (h // 2, 2, w // 2, 2)).mean(axis=(-3, -1))
    out = np.empty(lead + (h * 3 // 2, w), dtype=np.uint8)
    out[..., :h, :] = np.clip(np.rint(y), 0, 255)
    out[..., h:, :] = np.clip(np.rint(np.stack([sub(cb), sub(cr)], axis=-1)), 0, 255).reshape(lead + (h // 2, w))
    return out
