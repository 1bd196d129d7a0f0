"""Batches of any subset of streams, in any order: ``ids`` of ``BatchedLaneTracker.process`` and of the pipelines
(C ABI: lt_process_streams / lt_process_back_streams).

Frame i of a batch belongs to stream ids[i].  Frames, out frames, result records and masks are indexed by batch
position; tracking state, averaged polylines, the cached lane polygon and the captured pixel lists by stream id.  Every
stream here carries distinct content (road videos of distinct seeds, the bundled photographs, which take the second
attempt, seeded noise and blank frames), so that a kernel that reads or writes another stream's slot shows up.  The
oracle (tests/_oracle_pool.py, or tests/_oracle_pool_counted.py where the frame counter is drawn) runs, per stream,
exactly the frames that stream received, in order: result records, final masks, captured pixel sets and annotated
frames bit for bit, fit coefficients within 1e-6 relative."""
import ctypes as C
import os
import time
import warnings

import numpy as np
import pytest

import _fixtures as fx
import _oracle_pool
import _oracle_pool_counted
from _oracle_pool import frame_from_spec
from lane_tracker_b200 import synth

pytestmark = pytest.mark.gpu

FIT_RTOL = 1e-6
PHOTOS = fx.frame_names()
_ORACLE_FRAMES = [0]


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)


@pytest.fixture(scope="module", autouse=True)
def _oracle_wall_time():
    t0 = time.perf_counter()
    yield
    print("\ntest_gpu_stream_ids: %.1f s wall in this module (oracle frames: %d)"
          % (time.perf_counter() - t0, _ORACLE_FRAMES[0]))


def _tracker(S, **kw):
    from lane_tracker_b200 import BatchedLaneTracker
    return BatchedLaneTracker(S, **synth.shipped_calibration(), **kw)


def _batch(torch, specs):
    return torch.as_tensor(np.stack([frame_from_spec(sp) for sp in specs])).cuda()


def _oracle(plans, print_frame_count=False):
    """plans: {stream: [frame spec, ...]} -> {stream: [oracle record per frame]}."""
    keys = sorted(plans)
    _ORACLE_FRAMES[0] += sum(len(plans[s]) for s in keys)
    pool = _oracle_pool_counted if print_frame_count else _oracle_pool
    res = pool.run_jobs([dict(kind="plan", plan=plans[s]) for s in keys])
    return dict(zip(keys, res))


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


def _failing(s, r, k):
    """Content that fails the first attempt, distinct per stream within a round: the k-th photograph of the round,
    seeded noise or a blank frame."""
    kind = ("image", "blank", "noise", "image")[(s + r) % 4]
    if kind == "image":
        return ["image", PHOTOS[(k + r) % len(PHOTOS)]]
    if kind == "noise":
        return ["noise", 7000 + 100 * r + s]
    return ["blank", 30 + (7 * s) % 200]


def _round_specs(ids, r, seen, fail, seed0):
    """Frame specs of one round: stream s gets frame seen[s] of its road video unless it is in `fail`."""
    specs, k = [], 0
    for s in ids:
        if s in fail:
            specs.append(_failing(s, r, k))
            k += int(specs[-1][0] == "image")
        else:
            specs.append(["synth", seed0 + s, seen[s]])
    keys = [tuple(sp) for sp in specs]
    assert len(set(keys)) == len(keys), keys
    return specs


def _state(bt, s):
    """Tracking state, averaged polylines and cached lane polygon of stream s, as bytes."""
    st, lx, rx = bt.get_state(s)
    return [bytes(st), lx.tobytes(), rx.tobytes(), bt.debug_read("lane_rows", s).tobytes()]


def _snapshot(bt, s):
    """Everything a call may change of stream s: _state and the captures of both attempts (capture on)."""
    snap = _state(bt, s)
    for attempt in (0, 1):
        sides, cents = bt.read_capture(s, attempt)
        snap.append([(y.tobytes(), x.tobytes()) for y, x in sides])
        snap.append(cents)
    return snap


def _plan_rounds(S, rounds, seed0, fail_rate, rng):
    """-> (specs per round, oracle plans per stream)."""
    seen = [0] * S
    all_specs, plans = [], {}
    for r, ids in enumerate(rounds):
        fail = {int(s) for s in ids if rng.random() < fail_rate}
        specs = _round_specs([int(s) for s in ids], r, seen, fail, seed0)
        for s, sp in zip(ids, specs):
            plans.setdefault(int(s), []).append(sp)
            seen[int(s)] += 1
        all_specs.append(specs)
    return all_specs, plans


# ---- 1. identity ids equal the prefix path -------------------------------------------------------------------------

def test_identity_ids_equal_prefix_calls(torch_mod):
    """Two 64-stream handles fed the same frames, five calls at n = 64, 17, 9, 64, 17: one with process(frames),
    the other with process(frames, ids=range(n)).  Records, out frames, every stream's state, polylines and cached
    polygon are the same bytes (no oracle)."""
    torch = torch_mod
    S, calls = 64, [64, 17, 9, 64, 17]
    a, b = _tracker(S), _tracker(S)
    seen = [0] * S
    try:
        for r, n in enumerate(calls):
            fail = set(range(r % 3, n, 5))
            specs = _round_specs(list(range(n)), r, seen, fail, seed0=1000)
            for s in range(n):
                seen[s] += 1
            d = _batch(torch, specs)
            oa, ob = torch.empty_like(d), torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ra = a.process(d, oa)
                rb = b.process(d, ob, ids=range(n))
            assert ra.tobytes() == rb.tobytes(), (r, n)
            assert torch.equal(oa, ob), (r, n)
            for s in range(S):
                sa, la, xa = a.get_state(s)
                sb, lb, xb = b.get_state(s)
                assert bytes(sa) == bytes(sb) and np.array_equal(la, lb) and np.array_equal(xa, xb), (r, n, s)
                assert np.array_equal(a.debug_read("lane_rows", s), b.debug_read("lane_rows", s)), (r, n, s)
            assert 0 < int((ra["attempts"] == 2).sum()) < n
    finally:
        a.close()
        b.close()


# ---- 2. scattered arrival against the oracle ------------------------------------------------------------------------

def _scatter_rounds(S):
    rng = np.random.default_rng(33)
    rounds = [rng.permutation(S)[:m] for m in (33, 17, 16, 9, 1)]
    rounds.append(1 + rng.permutation(S - 2))                 # every stream but 0 and S - 1
    rounds += [rng.permutation(S)[:m] for m in (24, 12)]
    return rounds


def test_scattered_arrival_matches_oracle(torch_mod):
    """33 streams (more than one undistort group of 16), capture on, text on with the frame counter: eight rounds,
    each a random subset in random order (33, 17, 16, 9, 1, 31 without streams 0 and 32, 24, 12 streams).  Each
    stream matches the oracle run over exactly the frames it received."""
    torch = torch_mod
    S = 33
    rounds = _scatter_rounds(S)
    assert 0 not in rounds[5] and S - 1 not in rounds[5] and len(rounds[5]) == S - 2
    # seed 6: every oracle fit of this plan is well conditioned.  A pixel set that lies in one column on every row
    # (x = 661, met with other seeds where a photograph follows tracked frames) has a fit whose a and b are zero up
    # to rounding, and the moment-based fit rounds them differently from np.polyfit by more than FIT_RTOL.
    specs, plans = _plan_rounds(S, rounds, seed0=1200, fail_rate=0.25, rng=np.random.default_rng(6))
    want = _oracle(plans, print_frame_count=True)
    bt = _tracker(S, print_frame_count=True)
    assert bt.text_enabled
    bt.set_capture(True)
    seen = [0] * S
    modes, retries = set(), 0
    try:
        for r, (ids, sp) in enumerate(zip(rounds, specs)):
            d = _batch(torch, sp)
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, ids=ids)
            assert len(res) == len(ids)
            out = out.cpu().numpy()
            for i, s in enumerate(int(v) for v in ids):
                w, tag = want[s][seen[s]], (r, i, s)
                _check_record(res[i], w, tag)
                assert fx.sha(out[i]) == w["out"], tag
                assert fx.sha(bt.debug_read("mask", i)) == w["mask"], tag
                if w["detected"]:
                    sides, _ = bt.read_capture(s, w["attempts"] - 1)
                    assert fx.pix_digest(sides[0][0], sides[0][1], sides[1][0], sides[1][1]) == w["pix"], tag
                seen[s] += 1
                modes.add(int(res[i]["search_mode"]))
                retries += int(res[i]["attempts"] == 2)
    finally:
        bt.close()
    assert modes == {0, 1} and retries > 0, (modes, retries)


# ---- 3. a failing frame redraws its own stream's polygon ------------------------------------------------------------

def test_failing_frame_redraws_its_own_polygon(torch_mod):
    """Eight streams track their own road (one permuted batch), then streams 2 and 6 get a blank frame at batch
    positions 0 and 1, which streams 5 and 0 held in the first round.  Each must re-draw its own cached lane polygon
    (annotated frame against the oracle)."""
    torch = torch_mod
    S = 8
    first = [5, 0, 7, 3, 1, 6, 4, 2]
    rounds = [first, [2, 6]]
    seen = [0] * S
    specs = [_round_specs(first, 0, seen, set(), seed0=1400)]
    for s in first:
        seen[s] += 1
    specs.append([["blank", 60], ["blank", 140]])
    plans = {s: [specs[0][first.index(s)]] for s in range(S)}
    plans[2].append(specs[1][0])
    plans[6].append(specs[1][1])
    want = _oracle(plans)
    bt = _tracker(S)
    try:
        for r, (ids, sp) in enumerate(zip(rounds, specs)):
            d = _batch(torch, sp)
            out = torch.empty_like(d)
            res = bt.process(d, out, ids=ids)
            out = out.cpu().numpy()
            for i, s in enumerate(ids):
                w = want[s][r]
                _check_record(res[i], w, (r, i, s))
                assert fx.sha(out[i]) == w["out"], (r, i, s)
            if r == 0:
                assert all(res[first.index(s)]["valid_lane_lines"] for s in (0, 2, 5, 6))
            else:
                assert not res["valid_lane_lines"].any() and res["drew_lane"].all()
                assert not np.array_equal(out, d.cpu().numpy())      # the cached polygons were blended
    finally:
        bt.close()


# ---- 4. unlisted streams are untouched ------------------------------------------------------------------------------

def test_unlisted_streams_are_untouched(torch_mod):
    """24 streams with capture on: one full batch, then five partial batches whose ids are never a prefix (valid
    frames and photographs that take the second attempt).  After every call, each stream that was not listed has
    the same state, polylines, cached polygon and captured pixel lists of both attempts as before it."""
    torch = torch_mod
    S = 24
    rng = np.random.default_rng(24)
    rounds = [rng.permutation(S)] + [np.sort(rng.permutation(np.arange(1, S))[:m])[::-1] for m in (7, 12, 3, 16, 1)]
    specs, _ = _plan_rounds(S, rounds, seed0=1600, fail_rate=0.3, rng=rng)
    bt = _tracker(S)
    bt.set_capture(True)
    try:
        for r, (ids, sp) in enumerate(zip(rounds, specs)):
            listed = {int(s) for s in ids}
            before = {s: _snapshot(bt, s) for s in range(S) if s not in listed}
            d = _batch(torch, sp)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, torch.empty_like(d), ids=ids)
            if r:
                assert res["valid_lane_lines"].any(), r
            for s, snap in before.items():
                assert _snapshot(bt, s) == snap, (r, s)
        assert 0 not in {int(s) for ids in rounds[1:] for s in ids}
    finally:
        bt.close()


# ---- 5. permutation invariance ---------------------------------------------------------------------------------------

def test_subset_order_does_not_matter(torch_mod):
    """The same 20 of 33 streams in two orders on two handles, three rounds: every stream gets the same record,
    mask and out frame (no oracle)."""
    torch = torch_mod
    S = 33
    rng = np.random.default_rng(7)
    sub = rng.permutation(S)[:20]
    seen = [0] * S
    a, b = _tracker(S), _tracker(S)
    try:
        for r in range(3):
            ids_a = np.sort(sub)
            ids_b = rng.permutation(sub)
            fail = {int(s) for s in sub[r::4]}
            sp = dict(zip((int(s) for s in ids_a), _round_specs([int(s) for s in ids_a], r, seen, fail, seed0=1800)))
            for s in sub:
                seen[int(s)] += 1
            da = _batch(torch, [sp[int(s)] for s in ids_a])
            db = _batch(torch, [sp[int(s)] for s in ids_b])
            oa, ob = torch.empty_like(da), torch.empty_like(db)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ra = a.process(da, oa, ids=ids_a)
                rb = b.process(db, ob, ids=torch.as_tensor(ids_b))
            oa, ob = oa.cpu().numpy(), ob.cpu().numpy()
            pos_a = {int(s): i for i, s in enumerate(ids_a)}
            for j, s in enumerate(int(v) for v in ids_b):
                i = pos_a[s]
                assert rb[j].tobytes() == ra[i].tobytes(), (r, s)
                assert np.array_equal(ob[j], oa[i]), (r, s)
                assert np.array_equal(b.debug_read("mask", j), a.debug_read("mask", i)), (r, s)
            assert 0 < int((ra["attempts"] == 2).sum()) < len(sub)
    finally:
        a.close()
        b.close()


# ---- 6. two batches in flight -----------------------------------------------------------------------------------------

def test_pipelines_with_ids_equal_sequential_calls(torch_mod):
    """DevicePipeline over eight batches of alternating, overlapping subsets of 24 streams (all eight enqueued
    before the device starts on the first) gives the same out frames, final records and stream states as sequential process(..., ids=...);
    HostPipeline(inplace=True) does the same over four batches."""
    from lane_tracker_b200 import DevicePipeline, HostPipeline
    torch = torch_mod
    S = 24
    rng = np.random.default_rng(66)
    rounds = [rng.permutation(S)[:16] if k % 2 == 0 else rng.permutation(S)[:12] for k in range(8)]
    specs, _ = _plan_rounds(S, rounds, seed0=2000, fail_rate=0.25, rng=rng)
    batches = [_batch(torch, sp) for sp in specs]

    ref = _tracker(S, print_frame_count=True)
    want_out, want_res = [], []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for ids, d in zip(rounds, batches):
            o = torch.empty_like(d)
            want_res.append(ref.process(d, o, ids=ids).tobytes())
            want_out.append(o)
    want_state = [_state(ref, s) for s in range(S)]
    ref.close()

    bt = _tracker(S, print_frame_count=True)
    try:
        pipe = DevicePipeline(bt)
        outs = [torch.empty_like(d) for d in batches]
        torch.cuda.synchronize()
        # hold the device back (~25 ms on the current stream, which every submit waits for) so that all eight
        # batches are enqueued before the first one runs: the ids of batch k+1 are then handed over while the back
        # half of batch k has not read its own yet
        torch.cuda._sleep(50_000_000)
        for ids, d, o in zip(rounds, batches, outs):
            pipe.submit(d, o, ids=ids)
        res = pipe.fetch_results(len(rounds[-1]))
        for k, (o, w) in enumerate(zip(outs, want_out)):
            assert torch.equal(o, w), k
        assert res.tobytes() == want_res[-1]
        for s in range(S):
            assert _state(bt, s) == want_state[s], s
    finally:
        bt.close()

    T = 4
    bt = _tracker(S, print_frame_count=True)
    try:
        pipe = HostPipeline(bt, depth=3, inplace=True)
        hosts = [batches[k].cpu().pin_memory() for k in range(T)]
        got = []
        for k in range(T):
            pipe.submit(hosts[k], ids=rounds[k])
            got += [(o, r.copy()) for o, r in pipe.ready()]
        got += [(o, r.copy()) for o, r in pipe.drain()]
        assert len(got) == T
        for k, (o, r) in enumerate(got):
            assert r.tobytes() == want_res[k], k
            assert torch.equal(o, want_out[k].cpu()), k
    finally:
        bt.close()


# ---- 7. refusals --------------------------------------------------------------------------------------------------------

def test_bad_ids_are_refused(torch_mod):
    """A repeated id, id = S, id = -1, a wrong number of ids, more frames than streams, a CUDA tensor of ids:
    ValueError from Python; the C entry points refuse the same (and a null id list) with the id in lt_last_error,
    launch nothing, and every stream's state is unchanged."""
    from lane_tracker_b200 import DevicePipeline, _lib
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    S = 6
    bt = _tracker(S)
    lib = _lib.load()
    try:
        d = _batch(torch, [["synth", 2200 + s, 0] for s in range(4)])
        out = torch.empty_like(d)
        bt.process(d, out, ids=[3, 0, 5, 1])
        before = [_state(bt, s) for s in range(S)]
        n0 = lib.lt_launch_count()
        bad = {"appears more than once": [3, 0, 3, 1], "stream id 6 outside": [3, 0, 6, 1],
               "stream id -1 outside": [3, -1, 5, 1], "3 stream ids for 4 frames": [3, 0, 5]}
        for msg, ids in bad.items():
            with pytest.raises(ValueError, match=msg):
                bt.process(d, out, ids=ids)
            with pytest.raises(ValueError, match=msg):
                bt.process_back_async(d, out, 0, ids=np.asarray(ids))
            with pytest.raises(ValueError, match=msg):
                DevicePipeline(bt).submit(d, out, ids=torch.as_tensor(ids))
        with pytest.raises(ValueError, match="CUDA tensor"):
            bt.process(d, out, ids=torch.tensor([3, 0, 5, 1], device="cuda"))
        big = _batch(torch, [["blank", 10 + s] for s in range(S + 1)])
        with pytest.raises(ValueError, match="frames for"):
            bt.process(big, ids=list(range(S + 1)))

        p = make_params()
        res = bt._results_dev
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        P = C.c_void_p
        for ids, n, msg in [([3, 0, 3, 1], 4, "stream id 3 appears twice"), ([3, 0, 6, 1], 4, "stream id 6 at"),
                            ([3, -1, 5, 1], 4, "stream id -1 at"), (list(range(S + 1)), S + 1, "n_streams 7 outside"),
                            (None, 4, "null stream id list")]:
            arr = (C.c_int32 * len(ids))(*ids) if ids is not None else None
            src = big if n > 4 else d
            for call in (lambda: lib.lt_process_streams(bt._h, P(src.data_ptr()), P(src.data_ptr()), arr, n, C.byref(p),
                                                        P(res.data_ptr()), st),
                         lambda: lib.lt_process_back_streams(bt._h, P(src.data_ptr()), P(src.data_ptr()), arr, n,
                                                             C.byref(p), 0, P(res.data_ptr()), st)):
                rc = call()
                assert rc < 0, (ids, n)
                assert msg in lib.lt_last_error().decode(), (msg, lib.lt_last_error())
        torch.cuda.synchronize()
        assert lib.lt_launch_count() == n0
        for s in range(S):
            assert _state(bt, s) == before[s], s
    finally:
        bt.close()
