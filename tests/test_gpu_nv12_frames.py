"""NV12 input frames: lt_set_frame_format, and ``BatchedLaneTracker`` / the pipelines taking the format from the tensor
shape ([n, H * 3 / 2, W] is NV12, [n, H, W, 3] is RGB).

The oracle of every test is a second handle of the same configuration fed ``nv12_to_rgb`` of the same frames through
the RGB path.  The arithmetic is the same, so result records (fits included), final masks, annotated frames, every
stream's state, polylines, cached lane polygon and captured pixel lists must match byte for byte.  Two streams of the
64-stream test are also anchored to the CPU oracle run on ``cvops.yuv2rgb_nv12`` of their frames.  Content differs
per stream: road videos of distinct seeds, the bundled photographs (which take the second attempt), seeded random
NV12 with luma and chroma extremes, and blank frames."""
import ctypes as C
import warnings

import numpy as np
import pytest

import _fixtures as fx
from lane_tracker_b200 import synth

pytestmark = pytest.mark.gpu

PHOTOS = fx.frame_names()
_PHOTO_CACHE = {}


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def _cal(kind="shipped", scale=1.0):
    cal = synth.shipped_calibration(scale)
    if kind == "pincushion":
        # k1 > 0: at the corners of the ROI the undistort samples beyond the frame's left and right edges, so some
        # ROI pixels have 1-3 taps inside the frame (the shipped barrel distortion keeps every tap inside)
        d = cal["dist_coeffs"].copy()
        d[0, 0] = 0.2
        cal["dist_coeffs"] = d
    elif kind == "text_overlap":
        # overlay rows moved up by 400 frame rows, onto the rows of the putText lines: text is drawn under the blend
        M, Minv = cal["warp_matrices"]
        cal["warp_matrices"] = (M, np.array([[1.0, 0, 0], [0, 1.0, -400.0], [0, 0, 1.0]]) @ Minv)
    return cal


def _photo(name):
    if name not in _PHOTO_CACHE:
        _PHOTO_CACHE[name] = synth.rgb_to_nv12(fx.load_frame(name))
    return _PHOTO_CACHE[name]


def _noise(seed, W, H):
    """Seeded random NV12 with luma extremes (0, 255, and the clamp edges 15 / 16 / 235 / 236) and chroma extremes
    (0 / 255 pairs: every channel saturates) across the rows the tracker reads."""
    f = np.random.default_rng(seed).integers(0, 256, (H * 3 // 2, W), dtype=np.uint8)
    r0 = H * 5 // 8
    f[r0:r0 + H // 8:3] = np.resize(np.array([0, 255, 15, 16, 235, 236], np.uint8), W)
    f[H + r0 // 2:H + r0 // 2 + H // 32] = np.resize(np.array([0, 0, 255, 255, 0, 255, 255, 0], np.uint8), W)
    return f


def _content(S, T, scale=1.0, seed0=0):
    """NV12 uint8 [T, S, H * 3 / 2, W]; the kind of stream s cycles through road / photograph / noise / blank."""
    W, H = synth.shipped_calibration(scale)["img_size"]
    pattern = ("road", "photo", "noise", "road", "blank", "road") if scale == 1.0 else ("road", "noise", "road", "blank")
    kinds = [pattern[s % len(pattern)] for s in range(S)]
    roads = [s for s in range(S) if kinds[s] == "road"]
    rv = synth.render_streams(len(roads), T, scale, first_seed=seed0, workers=8)
    out = np.empty((T, S, H * 3 // 2, W), np.uint8)
    for j, s in enumerate(roads):
        out[:, s] = synth.rgb_to_nv12(rv[j])
    for s in range(S):
        for t in range(T):
            if kinds[s] == "photo":
                out[t, s] = _photo(PHOTOS[(s // len(pattern) + t) % len(PHOTOS)])
            elif kinds[s] == "noise":
                out[t, s] = _noise(1000 * seed0 + 10 * s + t, W, H)
            elif kinds[s] == "blank":
                out[t, s, :H] = (30 + 7 * s + t) % 200
                out[t, s, H:] = 128
    return out


def _tracker(S, cal):
    from lane_tracker_b200 import BatchedLaneTracker
    t = BatchedLaneTracker(S, **cal)
    t.set_capture(True)
    return t


def _snapshot(bt, s):
    """Everything a call may change of stream s: state, polylines, cached polygon, captured pixels of both attempts."""
    st, lx, rx = bt.get_state(s)
    snap = [bytes(st), lx.tobytes(), rx.tobytes(), bt.debug_read("lane_rows", s).tobytes()]
    for attempt in (0, 1):
        sides, cents = bt.read_capture(s, attempt)
        snap.append([(y.tobytes(), x.tobytes()) for y, x in sides])
        snap.append(cents)
    return snap


class Twin:
    """Handle `a` fed NV12 frames, handle `b` (same configuration) fed nv12_to_rgb of the same frames."""

    def __init__(self, torch, S, cal):
        self.torch = torch
        self.a, self.b = _tracker(S, cal), _tracker(S, cal)
        self.records = []
        self.mask_pixels = 0            # final masks with a lane pixel: the comparison is not of empty masks

    def close(self):
        self.a.close()
        self.b.close()

    def step(self, nv, overlay=True, ids=None, **kw):
        torch = self.torch
        d = torch.as_tensor(np.ascontiguousarray(nv)).cuda()
        rgb = self.b.nv12_to_rgb(d)
        oa = torch.full(rgb.shape, 77, dtype=torch.uint8, device="cuda") if overlay else None
        ob = torch.empty_like(rgb) if overlay else None
        ra = self.a.process(d, oa, ids=ids, **kw)
        rb = self.b.process(rgb, ob, ids=ids, **kw)
        assert ra.tobytes() == rb.tobytes()
        for i in range(int(d.shape[0])):
            mask = self.a.debug_read("mask", i)
            assert np.array_equal(mask, self.b.debug_read("mask", i)), i
            self.mask_pixels += int(mask.any())
        if overlay:
            assert torch.equal(oa, ob)
        self.records.append(ra)
        return ra, oa

    def check_streams(self, ids):
        for s in ids:
            assert _snapshot(self.a, s) == _snapshot(self.b, s), s


def _tap_cases(bt):
    """(ROI pixels with 1-3 taps inside the frame, taps at odd sx, taps at odd sy) of a handle's undistort."""
    W, H = bt.img_size
    r0, r1 = bt.geometry["roi_rows"]
    m = bt.debug_read("undistort_map")[r0:r1]
    sx, sy = m[..., 0] >> 5, m[..., 1] >> 5
    inside = sum(((sy + dy >= 0) & (sy + dy < H) & (sx + dx >= 0) & (sx + dx < W)).astype(int)
                 for dy in (0, 1) for dx in (0, 1))
    return int(((inside > 0) & (inside < 4)).sum()), int((sx % 2 == 1).sum()), int((sy % 2 == 1).sum())


def _anchor(nv_frames, records, outs, masks, cal):
    """One stream's NV12 frames through the CPU oracle on cvops.yuv2rgb_nv12 of each frame."""
    from oracle import cvops
    from oracle.tracker import OracleLaneTracker
    W, H = cal["img_size"]
    ref = OracleLaneTracker(**cal)
    for t, f in enumerate(nv_frames):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = ref.process(cvops.yuv2rgb_nv12(f, W, H))
        assert np.array_equal(outs[t], want), t
        assert np.array_equal(masks[t], ref.trace["attempts"][-1]["mask"]), t
        assert bool(records[t]["detected_pixels"]) == bool(ref.detected_pixels), t
        assert bool(records[t]["valid_lane_lines"]) == bool(ref.valid_lane_lines), t
        assert int(records[t]["last_detection"]) == ref.last_detection, t


@pytest.mark.parametrize("S,kind", [(64, "shipped"), (17, "pincushion")])
def test_nv12_matches_rgb_path(torch_mod, S, kind):
    """64 streams at the shipped calibration, 17 at one whose undistort samples beyond the frame edges."""
    T = 6
    cal = _cal(kind)
    tw = Twin(torch_mod, S, cal)
    try:
        partial, odd_x, odd_y = _tap_cases(tw.a)
        assert odd_x > 0 and odd_y > 0
        if kind == "pincushion":
            assert partial > 0
        ov0, ov1 = tw.a.geometry["overlay_rows"]
        assert ov0 % 2 or ov1 % 2, (ov0, ov1)       # a chroma row pair split between the overlay and the converter
        nv = _content(S, T, seed0=S)
        anchored = {0: ([], [], []), 1: ([], [], [])} if kind == "shipped" else {}
        for t in range(T):
            res, out = tw.step(nv[t])
            for s, (recs, outs, masks) in anchored.items():
                recs.append(res[s])
                outs.append(out[s].cpu().numpy())
                masks.append(tw.a.debug_read("mask", s))
        tw.check_streams(range(S))
        allr = np.concatenate(tw.records)
        assert allr["valid_lane_lines"].sum() > 0 and allr["drew_lane"].sum() > 0 and (allr["attempts"] == 2).sum() > 0
        for s, (recs, outs, masks) in anchored.items():
            _anchor(nv[:, s], recs, outs, masks, cal)
    finally:
        tw.close()


@pytest.mark.parametrize("scale,S", [(1.5, 5), (3.0, 3)])
def test_nv12_scaled_geometry(torch_mod, scale, S):
    T = 3
    tw = Twin(torch_mod, S, _cal(scale=scale))
    try:
        nv = _content(S, T, scale=scale, seed0=7)
        for t in range(T):
            tw.step(nv[t])
        tw.check_streams(range(S))
        # the reference's pixel-valued constants (window sizes, validity windows) do not scale: the lanes are found
        # but fail validation, so the check is that the masks compared were not empty
        assert tw.mask_pixels > 0
    finally:
        tw.close()


def test_nv12_text_under_blend(torch_mod):
    """Overlay rows that reach the putText rows: the whole frame is converted into out before text and blend."""
    S, T = 6, 4
    tw = Twin(torch_mod, S, _cal("text_overlap"))
    try:
        assert tw.a.text_enabled
        (t0, t1), (o0, o1) = tw.a.text_rows, tw.a.geometry["overlay_rows"]
        assert t0 < o1 and o0 < t1, (tw.a.text_rows, tw.a.geometry["overlay_rows"])
        nv = _content(S, T, seed0=3)
        for t in range(T):
            tw.step(nv[t])
        tw.check_streams(range(S))
        assert np.concatenate(tw.records)["drew_lane"].sum() > 0
    finally:
        tw.close()


def test_nv12_scattered_ids_and_fits_only(torch_mod):
    """Stream-id batches of changing size and order, overlay and fits only; unlisted streams untouched."""
    S = 33
    rng = np.random.default_rng(33)
    rounds = [rng.permutation(S)[:17], np.array([32]), rng.permutation(S)[:9], rng.permutation(S), rng.permutation(S)[:20]]
    nv = _content(S, len(rounds), seed0=11)
    seen = np.zeros(S, int)
    tw = Twin(torch_mod, S, _cal())
    try:
        for r, ids in enumerate(rounds):
            others = sorted(set(range(S)) - set(ids.tolist()))
            before = [_snapshot(tw.a, s) for s in others]
            frames = np.stack([nv[seen[s], s] for s in ids])
            seen[ids] += 1
            tw.step(frames, overlay=(r % 2 == 1), ids=ids)
            assert [_snapshot(tw.a, s) for s in others] == before
        tw.check_streams(range(S))
    finally:
        tw.close()


def _sequential(torch, S, cal, nv, overlay):
    """Reference: sequential process() calls on NV12 frames -> (records, annotated frames) per batch."""
    t = _tracker(S, cal)
    recs, outs = [], []
    try:
        for f in nv:
            d = torch.as_tensor(f).cuda()
            o = torch.empty((S,) + tuple(t.img_size[::-1]) + (3,), dtype=torch.uint8, device="cuda") if overlay else None
            recs.append(t.process(d, o).tobytes())
            outs.append(o.cpu().numpy() if overlay else None)
        snaps = [_snapshot(t, s) for s in range(S)]
    finally:
        t.close()
    return recs, outs, snaps


@pytest.mark.parametrize("overlay", [True, False])
def test_nv12_pipelines(torch_mod, overlay):
    from lane_tracker_b200 import DevicePipeline, GraphedProcess, HostPipeline
    torch = torch_mod
    S, T = 16, 5
    cal = _cal()
    nv = _content(S, T, seed0=21)
    want_recs, want_outs, want_snaps = _sequential(torch, S, cal, nv, overlay)
    W, H = cal["img_size"]

    def finish(t, recs, outs, parts=8):
        """parts: how much of each stream's snapshot to compare (8: all of it, 3: state and polylines)."""
        assert recs == want_recs
        if overlay:
            for o, w in zip(outs, want_outs):
                assert np.array_equal(o, w)
        for s in range(S):
            got, want = _snapshot(t, s), want_snaps[s]
            for k in range(parts):
                assert got[k] == want[k], (s, k)
        t.close()

    # DevicePipeline
    t = _tracker(S, cal)
    pipe = DevicePipeline(t)
    recs, outs = [], []
    dev = [torch.as_tensor(f).cuda() for f in nv]
    for f in dev:
        o = torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda") if overlay else None
        pipe.submit(f, o)
        recs.append(pipe.fetch_results(S).tobytes())
        outs.append(o.cpu().numpy() if overlay else None)
    finish(t, recs, outs)

    # GraphedProcess
    t = _tracker(S, cal)
    g = GraphedProcess(t, S, overlay=overlay, frame_format="nv12")
    assert tuple(g.frames.shape) == (S, H * 3 // 2, W) and (not overlay or tuple(g.out.shape) == (S, H, W, 3))
    recs, outs = [], []
    for f in dev:
        g.frames.copy_(f)
        g.replay()
        recs.append(g.fetch_results().tobytes())
        outs.append(g.out.cpu().numpy() if overlay else None)
    # GraphedProcess runs the chain once before capturing it and restores the tracking state and polylines after that
    # run (set_state); the run's captured pixel lists and cached polygon stay, as for RGB (test_gpu_parity.py)
    finish(t, recs, outs, parts=3)

    # HostPipeline: fits only uploads the source rows and their chroma rows; everything else is poisoned on the host
    t = _tracker(S, cal)
    hp = HostPipeline(t, depth=2, overlay=overlay, frame_format="nv12")
    a, b = t.geometry["source_rows"]
    recs, outs = [], []
    for f in nv:
        h = torch.as_tensor(f.copy()).pin_memory()
        if not overlay:
            assert hp.rows_in == (a, b)
            h[:, :a] = 0xA5
            h[:, b:H] = 0x5A
            h[:, H:H + a // 2] = 0xC3
            h[:, H + (b + 1) // 2:] = 0x3C
        hp.submit(h)
        for o, r in hp.drain():
            recs.append(r.tobytes())
            outs.append(o.numpy().copy() if overlay else None)
    finish(t, recs, outs)


def test_nv12_and_rgb_batches_alternate(torch_mod):
    """NV12 and RGB batches alternating on one handle equal an all-RGB sequence."""
    torch = torch_mod
    S, T = 9, 6
    nv = _content(S, T, seed0=5)
    a, b = _tracker(S, _cal()), _tracker(S, _cal())
    try:
        for t in range(T):
            d = torch.as_tensor(nv[t]).cuda()
            rgb = b.nv12_to_rgb(d)
            oa, ob = torch.empty_like(rgb), torch.empty_like(rgb)
            ra = a.process(d if t % 2 == 0 else rgb, oa)
            rb = b.process(rgb, ob)
            assert ra.tobytes() == rb.tobytes(), t
            assert torch.equal(oa, ob), t
        assert [_snapshot(a, s) for s in range(S)] == [_snapshot(b, s) for s in range(S)]
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("kind", ["shipped", "pincushion"])
def test_nv12_remap(torch_mod, kind):
    torch = torch_mod
    S = 17
    nv = torch.as_tensor(_content(S, 1, seed0=9)[0]).cuda()
    a, b = _tracker(S, _cal(kind)), _tracker(S, _cal(kind))
    try:
        bva = a.remap(nv)
        bvb = b.remap(b.nv12_to_rgb(nv))
        assert torch.equal(bva, bvb)
        for s in range(S):
            for what in ("r_plane", "b_plane"):
                assert np.array_equal(a.debug_read(what, s), b.debug_read(what, s)), (what, s)
    finally:
        a.close()
        b.close()


def test_nv12_refusals(torch_mod):
    from lane_tracker_b200 import BatchedLaneTracker, GraphedProcess, HostPipeline, _lib
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    S = 2
    cal = _cal()
    W, H = cal["img_size"]
    t = BatchedLaneTracker(S, **cal)
    lib = t.lib
    err = lambda: lib.lt_last_error().decode()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    try:
        # unknown formats
        for f in (-1, 2):
            assert lib.lt_set_frame_format(t._h, f) < 0 and "frame format" in err()
        # NV12 and the fused remap variant exclude each other, whichever comes second
        assert lib.lt_set_remap_mode(t._h, 1) == 0
        assert lib.lt_set_frame_format(t._h, 1) < 0 and "remap mode 1" in err()
        assert lib.lt_set_remap_mode(t._h, 0) == 0
        assert lib.lt_set_frame_format(t._h, 1) == 0
        assert lib.lt_set_remap_mode(t._h, 1) < 0 and "NV12" in err()
        # d_out overlapping the NV12 input, a misaligned NV12 buffer: refused before anything is enqueued
        from lane_tracker_b200.tracker import RESULT_DTYPE
        p = make_params()
        res = C.c_void_p(torch.zeros(S * RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda").data_ptr())
        rgb_bytes, nv_bytes = S * H * W * 3, S * H * W * 3 // 2
        buf = torch.zeros(rgb_bytes + nv_bytes + 64, dtype=torch.uint8, device="cuda")
        base = buf.data_ptr()
        call = lambda fr, out: lib.lt_process(t._h, C.c_void_p(fr), C.c_void_p(out), S, C.byref(p), res, stream)
        for fr, out in ((base, base), (base, base + nv_bytes - 4), (base + rgb_bytes - 8, base)):
            assert call(fr, out) < 0 and "overlaps" in err(), (fr - base, out - base)
        ids = (C.c_int32 * S)(1, 0)
        assert lib.lt_process_streams(t._h, C.c_void_p(base), C.c_void_p(base + 8), ids, S, C.byref(p), res,
                                      stream) < 0 and "overlaps" in err()
        assert lib.lt_process_back(t._h, C.c_void_p(base), C.c_void_p(base + nv_bytes - 8), S, C.byref(p), 0, res,
                                   stream) < 0 and "overlaps" in err()
        assert call(base + 2, base + nv_bytes + 8) < 0 and "aligned" in err()
        assert lib.lt_remap(t._h, C.c_void_p(base + 2), None, S, stream) < 0 and "aligned" in err()
        torch.cuda.synchronize()
        for s in range(S):
            assert t.get_state(s)[0].counter == 0
        assert lib.lt_set_frame_format(t._h, 0) == 0         # back to what the Python side last set
        # Python: shapes, dtypes, alignment, out, pipelines
        nv = torch.zeros((S, H * 3 // 2, W), dtype=torch.uint8, device="cuda")
        for bad in (torch.zeros((S, H, W), dtype=torch.uint8, device="cuda"),
                    torch.zeros((S, H * 3 // 2, W, 1), dtype=torch.uint8, device="cuda"),
                    torch.zeros((S, H * 3 // 2, W), dtype=torch.int16, device="cuda"),
                    torch.zeros((S, H * 3 // 2 + 1, W), dtype=torch.uint8, device="cuda"),
                    torch.zeros(S * H * 3 // 2 * W + 2, dtype=torch.uint8, device="cuda")[2:].view(S, H * 3 // 2, W)):
            with pytest.raises(ValueError):
                t.process(bad)
        with pytest.raises(ValueError):
            t.process(nv, torch.zeros((S, H * 3 // 2, W), dtype=torch.uint8, device="cuda"))
        with pytest.raises(ValueError):
            t.remap(nv[:, :H])
        with pytest.raises(ValueError):
            HostPipeline(t, frame_format="nv12", inplace=True)
        with pytest.raises(ValueError):
            HostPipeline(t, frame_format="yuv420")
        with pytest.raises(ValueError):
            GraphedProcess(t, frame_format="i420")
        hp = HostPipeline(t, depth=1, overlay=False, frame_format="nv12")
        with pytest.raises(ValueError):
            hp.submit(torch.zeros((S, H, W, 3), dtype=torch.uint8).pin_memory())
    finally:
        t.close()
    # an odd image height has no NV12 layout
    odd = dict(cal, img_size=(W, H - 1))
    t = BatchedLaneTracker(1, **odd)
    try:
        assert t.lib.lt_set_frame_format(t._h, 1) < 0 and "even" in t.lib.lt_last_error().decode()
        with pytest.raises(ValueError):
            t.process(torch.zeros((1, (H - 1) * 3 // 2, W), dtype=torch.uint8, device="cuda"))
    finally:
        t.close()
