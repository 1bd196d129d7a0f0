"""Launch geometries that only large or unusual batches reach, against the CPU oracle.

Every launcher picks its grid from the number of streams and its kernel variant from the filter options: 288-row
instead of 96-row bands for the vertical threshold and 32-row instead of 8-row bands for the opening from 16 streams
on, TMA / cp.async / unpacked threshold kernels by window size, retry-list launches that loop over a list of failing
streams, the morphology band split chosen (and cached) per stream count, CTAs of 8 streams in groups of 16 for the
undistort.  The tests here run those branches with batches in which every stream has different content (synthetic
road videos of distinct seeds, photographs, seeded noise, blank frames), so that a stream that reads or writes
another stream's slot shows up.  Everything goes through the C ABI; the oracle (tests/_oracle_pool.py) is the
checker: result records, final masks, captured pixel sets and annotated frames bit for bit, fit coefficients within
1e-6 relative.  The last test covers caller frame buffers at addresses that are 4- but not 16-byte aligned, and the
refusal of addresses that are not 4-byte aligned."""
import ctypes as C
import os
import time
import warnings

import numpy as np
import pytest

import _fixtures as fx
import _oracle_pool
from _oracle_pool import frame_from_spec
from lane_tracker_b200 import synth

pytestmark = pytest.mark.gpu

FIT_RTOL = 1e-6
PHOTOS = fx.frame_names()          # the 11 bundled photographs: both attempts, every frame


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)        # the launcher's own band split, not a pinned one


@pytest.fixture(scope="module", autouse=True)
def _oracle_wall_time():
    t0 = time.perf_counter()
    yield
    print("\ntest_gpu_launch_geometry: %.1f s wall in this module (oracle frames: %d)"
          % (time.perf_counter() - t0, _ORACLE_FRAMES[0]))


_ORACLE_FRAMES = [0]


def _oracle(plans, params=None, scale=1.0):
    """Oracle records of independent streams: plans[s] is the list of frame specs stream s sees, in order."""
    _ORACLE_FRAMES[0] += sum(len(p) for p in plans)
    return _oracle_pool.run_jobs([dict(kind="plan", plan=plan, scale=scale) for plan in plans], params)


def _batch(torch, specs, scale=1.0):
    return torch.as_tensor(np.stack([frame_from_spec(sp, scale) for sp in specs])).cuda()


def _check_record(res, want, tag):
    assert int(res["counter"]) == want["counter"], tag
    assert int(res["success"]) == want["success"], tag
    assert int(res["attempts"]) == want["attempts"], tag
    assert int(res["search_mode"]) == (1 if want["mode"] == "bs" else 0), tag
    assert bool(res["detected_pixels"]) == want["detected"], tag
    assert bool(res["valid_lane_lines"]) == want["valid"], tag
    assert int(res["last_detection"]) == want["last_detection"], tag
    assert bool(res["first_detected"]) == want["first_detected"], tag
    assert bool(res["first_valid"]) == want["first_valid"], tag
    if want["detected"]:
        assert int(res["n_left"]) == want["n_left"] and int(res["n_right"]) == want["n_right"], tag
        np.testing.assert_allclose(res["left_fit"], want["left_fit"], rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_fit"], want["right_fit"], rtol=FIT_RTOL, err_msg=str(tag))
    if want["valid"]:
        assert int(res["average_curve_radius"]) == want["radius"], tag
        assert float(res["eccentricity"]) == pytest.approx(want["ecc"], rel=1e-12, abs=1e-15), tag
        np.testing.assert_allclose(res["left_avg"], want["left_avg"], rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_avg"], want["right_avg"], rtol=FIT_RTOL, err_msg=str(tag))


def _check_streams(bt, res, out, wants, tag):
    """wants[s]: the oracle record of stream s for this frame.  Record, final mask, pixel set of the last attempt
    (capture on) and annotated frame of every stream listed."""
    for s, want in wants.items():
        t = (tag, s)
        _check_record(res[s], want, t)
        assert fx.sha(out[s]) == want["out"], t
        assert fx.sha(bt.debug_read("mask", s)) == want["mask"], t
        if want["detected"]:
            sides, _ = bt.read_capture(s, want["attempts"] - 1)
            assert fx.pix_digest(sides[0][0], sides[0][1], sides[1][0], sides[1][1]) == want["pix"], t


def _run_and_check(torch, bt, plans, want, scale=1.0, **kw):
    """Feed frame t of every plan to the handle, compare every stream with the oracle after every frame.
    Returns the retry count (streams that took the second attempt) of every frame."""
    S = len(plans)
    retries = []
    for t in range(len(plans[0])):
        d = _batch(torch, [plans[s][t] for s in range(S)], scale)
        out = torch.empty_like(d)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = bt.process(d, out, **kw)
        _check_streams(bt, res, out.cpu().numpy(), {s: want[s][t] for s in range(S)}, t)
        retries.append(sum(want[s][t]["attempts"] == 2 for s in range(S)))
    return retries


def _failing_frame(s, t, k):
    """Content that fails the first attempt, distinct per (stream, frame): a photograph (the k-th of this frame),
    seeded noise or a blank frame.  Noise only on the first frame: once a stream has valid lanes, the band search
    finds enough pixels of a noise frame along the previous lines, and the frame passes."""
    kinds = ("image", "noise", "blank") if t == 0 else ("image", "blank")
    kind = kinds[(s + t) % len(kinds)]
    if kind == "image":
        return ["image", PHOTOS[(k + t) % len(PHOTOS)]]
    if kind == "noise":
        return ["noise", 1000 * t + s]
    return ["blank", 30 + (7 * s) % 200]


def _failing_frames(t, streams, scale=1.0):
    """{stream: failing content} for the listed streams of frame t; photographs exist at the shipped scale only."""
    out, k = {}, 0
    for s in sorted(streams):
        sp = _failing_frame(s, t, k)
        if sp[0] == "image":
            k += 1
            if scale != 1.0:
                sp = ["noise", 5000 + 1000 * t + s]
        out[s] = sp
    return out


def _plans(S, T, fail, seed0, scale=1.0):
    """plans[s][t]: synthetic road video (seed seed0 + s) except where (s, t) is listed in fail[t].  Photographs
    exist at the shipped scale only."""
    plans = [[None] * T for _ in range(S)]
    for t in range(T):
        bad = _failing_frames(t, fail[t], scale)
        for s in range(S):
            plans[s][t] = bad.get(s, ["synth", seed0 + s, t])
    for t in range(T):      # no two streams of a batch see the same frame
        keys = [tuple(plans[s][t]) for s in range(S)]
        assert len(set(keys)) == S, keys
    return plans


# ---- 1. scattered retry lists ----------------------------------------------------------------------------------

# failing streams per frame: more than 16, exactly 1, at most 8, more than 8; first and last stream included
_SCATTER_FAIL = [
    {0, 2, 3, 5, 8, 9, 11, 14, 15, 16, 19, 20, 22, 24, 25, 27, 28, 30, 31, 32},
    {16},
    {1, 6, 17, 26, 32},
    {0, 4, 7, 10, 12, 13, 18, 21, 23, 29, 31, 32},
]


def test_scattered_retry_lists_33_streams(torch_mod):
    """S = 33 over four frames: the streams that take the second attempt are scattered over the batch and change
    from frame to frame (more than 16, one, at most 8, more than 8; the first and the last stream among them).  The second attempt runs
    on the retry list: box filter, opening and searches over 8 slots that loop over the list."""
    from lane_tracker_b200 import BatchedLaneTracker
    S, T = 33, 4
    plans = _plans(S, T, _SCATTER_FAIL, seed0=100)
    want = _oracle(plans)
    bt = BatchedLaneTracker(S, **synth.shipped_calibration())
    bt.set_capture(True)
    try:
        retries = _run_and_check(torch_mod, bt, plans, want)
        lists = [sorted(s for s in range(S) if want[s][t]["attempts"] == 2) for t in range(T)]
    finally:
        bt.close()
    assert retries[0] > 16 and retries[1] == 1 and 1 < retries[2] <= 8 and 8 < retries[3] <= 16, retries
    assert any(0 in l for l in lists) and any(S - 1 in l for l in lists), lists
    assert lists[0] != lists[3] and lists[1] != lists[2], lists


# ---- 2. filter options with 16 or more streams ------------------------------------------------------------------

# (k on each side of LT_HALO_Y - 16 = 40 selects the row-padded TMA / cp.async vertical threshold; a pair on both
# sides splits into two launches; k*255 + C*k >= 2^15 the unpacked kernels; k > 127 the prefix-sum row kernel)
_OPTION_ROWS = {
    "k40_k41_noise20": dict(ksize_r=40, ksize_b=41, mask_noise=True, ksize_noise=20),
    "k40_k40_ntries1": dict(ksize_r=40, ksize_b=40, n_tries=1),
    "k41_k41_partial": dict(ksize_r=41, ksize_b=41, partial=0.5),
    "wide_unpacked_noise65": dict(ksize_r=130, C_r=2, ksize_b=100, C_b=80, mask_noise=True, ksize_noise=65),
    "neighborhood_bw40": dict(filter_type="neighborhood", bandwidth=40),
}
_OPTION_FAIL_17 = [{2, 9, 13}, {0, 6, 11, 16}]
assert {40, 41} <= {kw.get(k) for kw in _OPTION_ROWS.values() for k in ("ksize_r", "ksize_b")}


@pytest.mark.parametrize("S,row", [(17, r) for r in _OPTION_ROWS] + [(64, "k40_k41_noise20")])
def test_filter_options_with_many_streams(torch_mod, S, row):
    """Non-default filter options with a batch of >= 16 streams (288-row bands of the vertical threshold, 32-row
    bands of the opening): each row of the table selects another kernel variant; two frames per stream."""
    from lane_tracker_b200 import BatchedLaneTracker
    kw = _OPTION_ROWS[row]
    assert S >= 16
    fail = _OPTION_FAIL_17 if S == 17 else [{2, 9, 13, 20, 31, 40, 47, 63}, {0, 6, 11, 16, 27, 38, 52, 59}]
    plans = _plans(S, 2, fail, seed0=200 + 100 * (S == 64))
    want = _oracle(plans, kw)
    bt = BatchedLaneTracker(S, **synth.shipped_calibration())
    bt.set_capture(True)
    if kw.get("bandwidth", 25) > 32:
        bt.set_pixel_capacity((2 * kw["bandwidth"] - 1) * 1100)
    try:
        retries = _run_and_check(torch_mod, bt, plans, want, **kw)
    finally:
        bt.close()
    if kw.get("n_tries", 2) == 1:
        assert retries == [0, 0]
    else:
        assert all(r > 0 for r in retries), retries          # the retry-list launches ran


# ---- 3. partial batches ------------------------------------------------------------------------------------------

def test_partial_batches_across_the_branch_points(torch_mod):
    """One handle of 64 streams called with 15, 16, 17, 8 and 9 frames: the launch geometry (bands, slot counts,
    the cached morphology band split) follows the number of frames, not the handle size.  Streams below n match the
    oracle; the state of the streams at n and above is left byte for byte as it was."""
    from lane_tracker_b200 import BatchedLaneTracker
    S, calls = 64, [15, 16, 17, 8, 9]
    fail = {0: {3, 12}, 1: {0, 15}, 2: {5, 16}, 3: {7}, 4: {1, 8}}
    plans = [[] for _ in range(S)]
    for c, n in enumerate(calls):
        bad = _failing_frames(c, fail[c])
        for s in range(n):
            plans[s].append(bad.get(s, ["synth", 400 + s, c]))
    want = _oracle([p for p in plans if p])
    cal = synth.shipped_calibration()
    bt = BatchedLaneTracker(S, **cal)
    bt.set_capture(True)

    def state(s):
        st, lx, rx = bt.get_state(s)
        return bytes(st), lx.tobytes(), rx.tobytes()

    bands = []
    try:
        seen = [0] * S
        for c, n in enumerate(calls):
            before = {s: state(s) for s in range(n, S)}
            d = _batch(torch_mod, [plans[s][seen[s]] for s in range(n)])
            out = torch_mod.empty_like(d)
            res = bt.process(d, out)
            assert len(res) == n
            _check_streams(bt, res, out.cpu().numpy(), {s: want[s][seen[s]] for s in range(n)}, (c, n))
            for s in range(n, S):
                assert state(s) == before[s], (c, n, s)
            for s in range(n):
                seen[s] += 1
            bands.append(bt.morph_bands())
    finally:
        bt.close()
    # the band split of each call is the one a fresh handle picks for that many streams (the cache follows n)
    for n, b in zip(calls, bands):
        fresh = BatchedLaneTracker(n, **cal)
        try:
            fresh.remap(_batch(torch_mod, [["blank", 90]] * n), want_bv=False)
            fresh.filter_lane_points(None, "bilateral", 15, 8, 35, 5)
            assert fresh.morph_bands() == b, (n, b)
        finally:
            fresh.close()
    assert len(set(bands)) >= 2, bands


# ---- 4. permutation invariance -----------------------------------------------------------------------------------

@pytest.mark.parametrize("S", [33, 18, 21])
def test_stream_permutation_invariance(torch_mod, S):
    """The same S streams in order in one handle and permuted in another, three frames of state: every stream's
    record, mask and annotated frame are the same bytes.  An index error that maps stream s to s +- 4, 8, 16 (chunk,
    CTA and group strides of the undistort layout) or anything else breaks this (no oracle needed)."""
    from lane_tracker_b200 import BatchedLaneTracker
    torch = torch_mod
    T = 3
    fail = [set(range(1, S, 5)) | {S - 1}, set(range(3, S, 7)), set(range(0, S, 4))]
    plans = _plans(S, T, fail, seed0=500)
    perm = np.random.default_rng(S).permutation(S)
    assert (perm != np.arange(S)).sum() >= S - 2
    cal = synth.shipped_calibration()
    a, b = BatchedLaneTracker(S, **cal), BatchedLaneTracker(S, **cal)
    try:
        for t in range(T):
            d = _batch(torch, [plans[s][t] for s in range(S)])
            dp = d[torch.as_tensor(perm, device=d.device)].contiguous()
            oa, ob = torch.empty_like(d), torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ra = a.process(d, oa)
                rb = b.process(dp, ob)
            oa, ob = oa.cpu().numpy(), ob.cpu().numpy()
            for i in range(S):
                s = int(perm[i])
                assert rb[i].tobytes() == ra[s].tobytes(), (S, t, i, s)
                assert np.array_equal(ob[i], oa[s]), (S, t, i, s)
                assert np.array_equal(b.debug_read("mask", i), a.debug_read("mask", s)), (S, t, i, s)
            assert 0 < int((ra["attempts"] == 2).sum()) < S
    finally:
        a.close()
        b.close()


# ---- 5. scaled geometry at batch size ------------------------------------------------------------------------------

@pytest.mark.parametrize("scale,S,T", [(1.5, 17, 2), (3.0, 8, 1)])
def test_scaled_geometry_batches(torch_mod, scale, S, T):
    """1920x1080 frames with 17 streams (two frames, n_tries = 2) and 3840x2160 frames with 8 streams: the rescaled
    calibration changes every plane, band and tile count; every stream against the oracle."""
    from lane_tracker_b200 import BatchedLaneTracker
    fail = [{1, 6, 12}, {0, 9, 16}][:T] if S == 17 else [{2, 5}]
    plans = _plans(S, T, fail, seed0=600, scale=scale)
    want = _oracle(plans, dict(n_tries=2), scale=scale)
    bt = BatchedLaneTracker(S, **synth.shipped_calibration(scale))
    bt.set_capture(True)
    try:
        retries = _run_and_check(torch_mod, bt, plans, want, scale=scale, n_tries=2)
    finally:
        bt.close()
    assert all(r >= 1 for r in retries), retries


# ---- 6. frame buffer alignment ------------------------------------------------------------------------------------

def _view_at(torch, nbytes, offset, shape):
    """A contiguous uint8 view of `nbytes` bytes that starts `offset` bytes into a 256-byte aligned allocation."""
    buf = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    assert buf.data_ptr() % 256 == 0
    return buf[offset:offset + nbytes].view(*shape)


def test_frame_buffers_at_unaligned_offsets(torch_mod):
    """Frames and out that start 4, 8 or 12 bytes into an allocation (4- but not 16-byte aligned: the overlay
    copies every row itself instead of the vector row copy), out of place and in place: the same results and frames
    as with aligned buffers.  Offsets 1-3 are refused -- ValueError from the Python classes, an error from every
    ABI entry that takes a frame buffer -- before any kernel is launched."""
    from lane_tracker_b200 import BatchedLaneTracker, _lib
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    S, T = 3, 2
    plans = _plans(S, T, [{1}, {2}], seed0=700)
    cal = synth.shipped_calibration()
    batches = [_batch(torch, [plans[s][t] for s in range(S)]) for t in range(T)]
    shape, nbytes = tuple(batches[0].shape), batches[0].numel()

    ref = BatchedLaneTracker(S, **cal)
    want = []
    for d in batches:
        o = torch.empty_like(d)
        r = ref.process(d, o)
        want.append((r.tobytes(), o.cpu().numpy()))
    ref.close()
    assert any((w[1] != d.cpu().numpy()).any() for w, d in zip(want, batches))     # the overlay changed pixels

    for off in (4, 8, 12):
        a, b = BatchedLaneTracker(S, **cal), BatchedLaneTracker(S, **cal)
        try:
            for t, d in enumerate(batches):
                fr = _view_at(torch, nbytes, off, shape)
                out = _view_at(torch, nbytes, 16 - off, shape)
                fr.copy_(d)
                ra = a.process(fr, out)                   # out of place, both buffers misaligned by 16
                assert ra.tobytes() == want[t][0], (off, t)
                assert np.array_equal(out.cpu().numpy(), want[t][1]), (off, t)
                assert torch.equal(fr, d), (off, t)       # the input is untouched
                rb = b.process(fr, fr)                    # in place
                assert rb.tobytes() == want[t][0], (off, t)
                assert np.array_equal(fr.cpu().numpy(), want[t][1]), (off, t)
        finally:
            a.close()
            b.close()

    lib = _lib.load()
    bt = BatchedLaneTracker(S, **cal)
    try:
        good = batches[0]
        good_out = torch.empty_like(good)
        p = make_params()
        res = bt._results_dev
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        xs = torch.zeros((S, 2, cal["warped_size"][1]), dtype=torch.int32, device="cuda")
        cnt = torch.zeros((S, 2), dtype=torch.int32, device="cuda")
        bv = torch.empty((S, cal["warped_size"][1], cal["warped_size"][0], 3), dtype=torch.uint8, device="cuda")
        kinds = (C.c_int32 * S)(*[1] * S)
        counters = (C.c_int32 * S)(*[0] * S)
        for off in (1, 2, 3):
            fr = _view_at(torch, nbytes, off, shape)
            fr.copy_(good)
            n0 = lib.lt_launch_count()
            with pytest.raises(ValueError, match="aligned"):
                bt.process(fr)
            with pytest.raises(ValueError, match="aligned"):
                bt.process(good, fr)
            with pytest.raises(ValueError, match="aligned"):
                bt.process_front_async(fr, 0)
            with pytest.raises(ValueError, match="aligned"):
                bt.process_back_async(good, fr, 0)
            with pytest.raises(ValueError, match="aligned"):
                bt.remap(fr)
            with pytest.raises(ValueError, match="aligned"):
                bt.warp_frame(fr)
            with pytest.raises(ValueError, match="aligned"):
                bt.draw_lane(fr, xs, cnt)
            with pytest.raises(ValueError, match="aligned"):
                bt.draw_text(fr, [1] * S)
            # the ABI itself, called with handmade pointers
            g, bad = good.data_ptr(), good.data_ptr() + off
            P = C.c_void_p
            calls = [
                lambda: lib.lt_process(bt._h, P(bad), P(good_out.data_ptr()), S, C.byref(p), P(res.data_ptr()), st),
                lambda: lib.lt_process(bt._h, P(g), P(bad), S, C.byref(p), P(res.data_ptr()), st),
                lambda: lib.lt_process_front(bt._h, P(bad), S, C.byref(p), 0, st),
                lambda: lib.lt_process_back(bt._h, P(bad), P(good_out.data_ptr()), S, C.byref(p), 0, P(res.data_ptr()), st),
                lambda: lib.lt_process_back(bt._h, P(g), P(bad), S, C.byref(p), 0, P(res.data_ptr()), st),
                lambda: lib.lt_remap(bt._h, P(bad), P(bv.data_ptr()), S, st),
                lambda: lib.lt_warp_frame(bt._h, P(bad), S, P(bv.data_ptr()), st),
                lambda: lib.lt_draw_lane(bt._h, P(bad), P(good_out.data_ptr()), S, P(xs.data_ptr()), P(cnt.data_ptr()), st),
                lambda: lib.lt_draw_lane(bt._h, P(g), P(bad), S, P(xs.data_ptr()), P(cnt.data_ptr()), st),
                lambda: lib.lt_draw_text(bt._h, P(bad), S, kinds, None, None, counters, st),
            ]
            for i, call in enumerate(calls):
                with pytest.raises(_lib.LaneTrackerError, match="4-byte aligned"):
                    _lib.check(call())
            torch.cuda.synchronize()
            assert lib.lt_launch_count() == n0, off          # nothing was launched
            assert torch.equal(fr, good)
        # the handle is intact: an aligned call afterwards gives the reference results
        bt.reset()
        r = bt.process(good, good_out)
        assert r.tobytes() == want[0][0] and np.array_equal(good_out.cpu().numpy(), want[0][1])
    finally:
        bt.close()
