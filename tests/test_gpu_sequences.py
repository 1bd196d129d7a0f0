"""Frame sequences: ``sequence=True`` of ``BatchedLaneTracker.process`` and of the pipelines (C ABI:
lt_process_sequence / lt_process_back_sequence).

Stream ids may repeat in a sequence batch: the frames of one stream are consecutive frames of that stream, in batch
order.  The reference is a second handle fed the same frames one at a time through ``process(frame, ids=[s])``.
Result records, annotated frames and final masks per position, and every stream's state, polylines, cached polygon
and captured pixel lists after the batch must be the same bytes.  Streams mix road videos with photographs (which
take the second attempt), blank and noise frames, so that cached-polygon frames and the n_fail / n_reset fallback
to the sliding window happen inside one batch.  Two streams also run through the CPU oracle."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

import _fixtures as fx
import _oracle_pool_counted
from _oracle_pool import frame_from_spec
from lane_tracker_b200 import synth

pytestmark = pytest.mark.gpu

PHOTOS = fx.frame_names()
FIT_RTOL = 1e-6


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)


def _tracker(S, cal=None, **kw):
    from lane_tracker_b200 import BatchedLaneTracker
    return BatchedLaneTracker(S, **(cal or synth.shipped_calibration()), **kw)


def _spec(s, t, fail):
    """Frame t of stream s: its road video, or a photograph, a blank or a noise frame when t lies in a failing run."""
    if not any(a <= t < b for a, b in fail):
        return ["synth", 3000 + s, t]
    kind = ("image", "blank", "noise", "image")[(s + t) % 4]
    if kind == "image":
        return ["image", PHOTOS[(s + t) % len(PHOTOS)]]
    if kind == "noise":
        return ["noise", 9000 + 100 * t + s]
    return ["blank", 30 + (7 * s + t) % 200]


# failing runs: short ones (cached polygon redrawn), and a long one (beyond n_fail = 8 and n_reset = 4)
FAIL = [(5, 8), (19, 31), (40, 42), (55, 57)]


def _frames(torch, specs, nv12=False):
    a = np.stack([frame_from_spec(sp) for sp in specs])
    return torch.as_tensor(synth.rgb_to_nv12(a) if nv12 else a).cuda()


def _snapshot(bt, s, capture):
    """Everything a call may change of stream s: state, polylines, cached polygon, and (capture on) the captured
    pixel lists of both attempts."""
    st, lx, rx = bt.get_state(s)
    snap = [bytes(st), lx.tobytes(), rx.tobytes(), bt.debug_read("lane_rows", s).tobytes()]
    if capture:
        for attempt in (0, 1):
            sides, cents = bt.read_capture(s, attempt)
            snap.append([(y.tobytes(), x.tobytes()) for y, x in sides])
            snap.append(cents)
    return snap


class Pair:
    """A handle fed sequence batches and a reference handle fed the same frames one at a time."""

    def __init__(self, torch, S, cal=None, capture=False, **kw):
        self.torch, self.S, self.capture = torch, S, capture
        self.a, self.b = _tracker(S, cal, **kw), _tracker(S, cal, **kw)
        if capture:
            self.a.set_capture(True)
            self.b.set_capture(True)

    def close(self):
        self.a.close()
        self.b.close()

    def reference(self, frames, ids, overlay=True, inplace=False, params=None):
        """Per-frame results of the reference: (records, out frames or None, masks)."""
        torch, b = self.torch, self.b
        recs, outs, masks = [], [], []
        w, h = b.img_size
        for i, s in enumerate(int(v) for v in ids):
            f = frames[i:i + 1].clone() if inplace else frames[i:i + 1]
            out = f if inplace else (torch.empty((1, h, w, 3), dtype=torch.uint8, device="cuda") if overlay else None)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                recs.append(b.process(f, out, ids=[s], params=params))
            masks.append(b.debug_read("mask", 0))
            outs.append(out[0].cpu().numpy() if out is not None else None)
        return np.concatenate(recs), outs, masks

    def check(self, res, outs, frames, ids, overlay=True, inplace=False, params=None, tag=""):
        """res / outs: the sequence handle's records and out frames ([n, H, W, 3] NumPy or None) of this batch."""
        want, wout, wmask = self.reference(frames, ids, overlay, inplace, params)
        assert len(res) == len(ids)
        for i in range(len(ids)):
            assert res[i].tobytes() == want[i].tobytes(), (tag, i, int(ids[i]))
            assert np.array_equal(self.a.debug_read("mask", i), wmask[i]), (tag, i)
            if overlay:
                assert np.array_equal(outs[i], wout[i]), (tag, i)
        for s in range(self.S):
            assert _snapshot(self.a, s, self.capture) == _snapshot(self.b, s, self.capture), (tag, s)
        return want

    def step(self, frames, ids, overlay=True, inplace=False, params=None, tag=""):
        """One sequence batch on the first handle, checked against the reference."""
        torch = self.torch
        w, h = self.a.img_size
        src = frames.clone() if inplace else frames
        out = src if inplace else (torch.empty((len(ids), h, w, 3), dtype=torch.uint8, device="cuda")
                                   if overlay else None)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = self.a.process(src, out, ids=ids, sequence=True, params=params)
        return res, self.check(res, out.cpu().numpy() if overlay else None, frames, ids, overlay, inplace, params, tag)


# ---- one stream, many frames ------------------------------------------------------------------------------------------

def test_one_stream_64_frames(torch_mod):
    """One stream, 64 frames in one batch and then 40 more, with failing runs, capture on and the frame counter drawn.
    The retry selection must compact the round's positions, not 0..n-1."""
    torch = torch_mod
    pr = Pair(torch, 64, capture=True, print_frame_count=True)
    try:
        assert pr.a.text_enabled
        allres = []
        for t0, n in ((0, 64), (64, 40)):
            specs = [_spec(0, t, [(a + 40, b + 40) for a, b in FAIL] if t0 else FAIL) for t in range(t0, t0 + n)]
            res, _ = pr.step(_frames(torch, specs), [0] * n, tag=t0)
            allres.append(res)
        res = np.concatenate(allres)
        assert list(res["counter"]) == list(range(1, 105))
        assert (res["attempts"] == 2).any() and res["valid_lane_lines"].any()
        assert set(res["search_mode"]) == {0, 1}
        assert ((res["drew_lane"] != 0) & (res["valid_lane_lines"] == 0)).any()     # cached polygon redrawn
    finally:
        pr.close()


# ---- layouts and multiplicities -----------------------------------------------------------------------------------------

def _layout_ids(kind, k, m, rng):
    if kind == "stream-major":
        return [s for s in range(k) for _ in range(m)]
    if kind == "round-major":
        return [s for _ in range(m) for s in range(k)]
    ids = [s for s in range(k) for _ in range(m)]
    return list(rng.permutation(ids))       # any interleaving keeps each stream's frames in time order


@pytest.mark.parametrize("k,m", [(4, 16), (8, 8), (16, 4)])
def test_layouts(torch_mod, k, m):
    """k streams x m frames in stream-major, round-major and a shuffled time-ordered layout: each stream's frames go
    to consecutive frames of that stream whatever the layout (rounds built by occurrence, not by position)."""
    torch = torch_mod
    rng = np.random.default_rng(k)
    fail = [(3, 5), (9, 12)]
    for kind in ("stream-major", "round-major", "shuffled"):
        ids = _layout_ids(kind, k, m, rng)
        seen = [0] * k
        specs = []
        for s in ids:
            specs.append(_spec(s, seen[s], fail if s % 2 else []))
            seen[s] += 1
        pr = Pair(torch, 64, capture=True)
        try:
            res, _ = pr.step(_frames(torch, specs), ids, tag=kind)
            assert (res["attempts"] == 2).any(), kind
        finally:
            pr.close()


def test_multiplicities_and_untouched_streams(torch_mod):
    """A batch over all 64 streams, then 7 streams with 1 to 20 frames each (64 frames, shuffled in time order): the
    57 others keep their state, polylines, cached polygon and captured pixel lists byte for byte."""
    torch = torch_mod
    S = 64
    pr = Pair(torch, S, capture=True)
    try:
        pr.step(_frames(torch, [_spec(s, 0, [(0, 1)] if s % 5 == 0 else []) for s in range(S)]), list(range(S)),
                tag="all")
        mult = {3: 1, 11: 20, 17: 2, 22: 7, 29: 12, 44: 3, 63: 19}
        assert sum(mult.values()) == S
        ids = [int(v) for v in np.random.default_rng(5).permutation([s for s, c in mult.items() for _ in range(c)])]
        seen = {s: 1 for s in mult}
        specs = []
        for s in ids:
            specs.append(_spec(s, seen[s], [(4, 6), (9, 17)]))
            seen[s] += 1
        others = [s for s in range(S) if s not in mult]
        before = {s: _snapshot(pr.a, s, True) for s in others}
        res, _ = pr.step(_frames(torch, specs), ids, tag="seq")
        for s in others:
            assert _snapshot(pr.a, s, True) == before[s], s
        assert (res["attempts"] == 2).any()
    finally:
        pr.close()


# ---- overlay and text from the position's snapshot ---------------------------------------------------------------------

def _two_streams(n, t0=0):
    """n frames of streams 5 and 2, interleaved unevenly, with failing runs: (ids, specs)."""
    ids = [5 if (i % 3) else 2 for i in range(n)]
    seen = {5: t0, 2: t0}
    specs = []
    for s in ids:
        specs.append(_spec(s, seen[s], [(3, 5), (8, 11), (14, 16), (20, 22)]))
        seen[s] += 1
    return ids, specs


@pytest.mark.parametrize("mode", ["counter", "inplace", "nv12", "fits_only", "text_under_blend"])
def test_overlay_reads_the_position_snapshot(torch_mod, mode):
    """Every out frame is drawn with its own frame's polygon and text (not the stream's last): the frame counter
    drawn, in place, NV12 input, fits only, and a calibration whose overlay rows reach the text rows."""
    torch = torch_mod
    cal, kw = None, {}
    if mode == "counter":
        kw["print_frame_count"] = True
    if mode == "text_under_blend":
        cal = synth.shipped_calibration()
        M, Minv = cal["warp_matrices"]
        cal["warp_matrices"] = (M, np.array([[1.0, 0, 0], [0, 1.0, -400.0], [0, 0, 1.0]]) @ Minv)
    pr = Pair(torch, 24, cal=cal, **kw)
    try:
        if mode == "text_under_blend":
            (t0, t1), (o0, o1) = pr.a.text_rows, pr.a.geometry["overlay_rows"]
            assert t0 < o1 and o0 < t1
        for r in range(2):
            ids, specs = _two_streams(24 - 5 * r, t0=12 * r)
            frames = _frames(torch, specs, nv12=mode == "nv12")
            res, _ = pr.step(frames, ids, overlay=mode != "fits_only", inplace=mode == "inplace", tag=(mode, r))
            assert res["drew_lane"].any() and (res["attempts"] == 2).any()
    finally:
        pr.close()


# ---- no repeats, one attempt ------------------------------------------------------------------------------------------

def test_no_repeats_equals_streams_call(torch_mod):
    """A sequence batch without a repeated id is lt_process_streams: the same records, out frames and states, and
    the same number of launches."""
    from lane_tracker_b200 import _lib
    torch = torch_mod
    lib = _lib.load()
    S = 24
    a, b = _tracker(S), _tracker(S)
    try:
        rng = np.random.default_rng(9)
        for r in range(3):
            ids = [int(v) for v in rng.permutation(S)[:S - 4 * r]]
            d = _frames(torch, [_spec(s, r, [(1, 2)] if s % 3 == 0 else []) for s in ids])
            oa, ob = torch.empty_like(d), torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                c0 = lib.lt_launch_count()
                ra = a.process(d, oa, ids=ids, sequence=True)
                c1 = lib.lt_launch_count()
                rb = b.process(d, ob, ids=ids)
                c2 = lib.lt_launch_count()
            assert c1 - c0 == c2 - c1, r
            assert ra.tobytes() == rb.tobytes() and torch.equal(oa, ob), r
            for s in range(S):
                assert _snapshot(a, s, False) == _snapshot(b, s, False), (r, s)
    finally:
        a.close()
        b.close()


def test_one_attempt(torch_mod):
    """n_tries = 1: no retry selection, rounds of search and update only."""
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    p = make_params(n_tries=1)
    pr = Pair(torch, 32)
    try:
        ids, specs = _two_streams(32)
        res, _ = pr.step(_frames(torch, specs), ids, params=p)
        assert (res["attempts"] == 1).all() and not res["valid_lane_lines"].all()
    finally:
        pr.close()


# ---- the pipelines -------------------------------------------------------------------------------------------------------

def test_device_pipeline(torch_mod):
    """DevicePipeline over four sequence batches (state carried across batches) against the reference."""
    from lane_tracker_b200 import DevicePipeline
    torch = torch_mod
    pr = Pair(torch, 32, print_frame_count=True)
    try:
        pipe = DevicePipeline(pr.a)
        t = {0: 0, 1: 0}
        for r, n in enumerate((32, 20, 32, 7)):
            ids = [int(v) for v in np.random.default_rng(r).integers(0, 2, n)]
            specs = []
            for s in ids:
                specs.append(_spec(s, t[s], [(6, 9), (30, 34)]))
                t[s] += 1
            d = _frames(torch, specs)
            out = torch.empty_like(d)
            pipe.submit(d, out, ids=ids, sequence=True)
            res = pipe.fetch_results(n)
            pr.check(res, out.cpu().numpy(), d, ids, tag=r)
    finally:
        pr.close()


def test_host_pipeline_inplace(torch_mod):
    """HostPipeline(inplace=True) over three sequence batches: the pinned frames come back annotated as the
    reference annotates them one at a time."""
    from lane_tracker_b200 import HostPipeline
    torch = torch_mod
    pr = Pair(torch, 16)
    try:
        pipe = HostPipeline(pr.a, depth=2, inplace=True)
        batches = []
        t = 0
        for r in range(3):
            specs = [_spec(1, t + i, [(5, 8), (20, 22)]) for i in range(16)]
            t += 16
            host = torch.as_tensor(np.stack([frame_from_spec(sp) for sp in specs])).pin_memory()
            batches.append((host.clone(), [1] * 16))
            pipe.submit(host, ids=[1] * 16, sequence=True)
            got = list(pipe.drain())
            assert len(got) == 1
            out, res = got[0]
            frames, ids = batches[-1]
            pr.check(res.copy(), out.numpy(), frames.cuda(), ids, inplace=True, tag=r)
    finally:
        pr.close()


# ---- capture, graphs, stage timing ----------------------------------------------------------------------------------------

def test_capture_holds_the_last_frame(torch_mod):
    """Capture on: after a sequence batch, read_capture of a stream equals the reference's after its last frame
    (checked by Pair), and differs from the lists of an earlier frame of the batch."""
    torch = torch_mod
    pr = Pair(torch, 16, capture=True)
    try:
        ids = [4] * 6
        specs = [_spec(4, t, []) for t in range(6)]
        pr.step(_frames(torch, specs), ids)
        last = pr.a.read_capture(4, 0)[0]
        b = _tracker(16)
        b.set_capture(True)
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                b.process(_frames(torch, specs[:1]), ids=[4])
            first = b.read_capture(4, 0)[0]
        finally:
            b.close()
        assert [(y.tobytes(), x.tobytes()) for y, x in last] != [(y.tobytes(), x.tobytes()) for y, x in first]
    finally:
        pr.close()


def test_cuda_graph_capture(torch_mod):
    """A sequence call captured once with torch.cuda.graph and replayed over three batches."""
    from lane_tracker_b200.tracker import RESULT_DTYPE
    torch = torch_mod
    n = 16
    ids = [0, 1, 1, 0, 2, 2, 2, 0, 1, 0, 0, 1, 2, 0, 1, 2]
    pr = Pair(torch, n, print_frame_count=True)
    try:
        t = {0: 0, 1: 0, 2: 0}

        def batch():
            specs = []
            for s in ids:
                specs.append(_spec(s, t[s], [(4, 7)]))
                t[s] += 1
            return _frames(torch, specs)

        static = batch()
        out = torch.empty_like(static)
        resd = torch.zeros(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            pr.a.process_async(static, out, ids=ids, sequence=True, results_dev=resd)     # warm-up: first use allocates
            torch.cuda.synchronize()
            pr.check(pr.a.fetch_results(n, resd), out.cpu().numpy(), static, ids, tag="warm-up")
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                pr.a.process_async(static, out, ids=ids, sequence=True, results_dev=resd)
        for r in range(3):
            d = batch()
            static.copy_(d)
            g.replay()
            torch.cuda.synchronize()
            pr.check(pr.a.fetch_results(n, resd), out.cpu().numpy(), d, ids, tag=r)
    finally:
        pr.close()


def test_stage_timing_of_64_rounds(torch_mod):
    """profile_begin(1) over a 64-round call: every round's marks fit, so the overlay (the last stage) is timed."""
    torch = torch_mod
    bt = _tracker(64)
    try:
        d = _frames(torch, [_spec(0, t, [(10, 14)]) for t in range(64)])
        out = torch.empty_like(d)
        bt.profile_begin(1)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            bt.process(d, out, ids=[0] * 64, sequence=True)
        ms, calls = bt.profile_read()
        assert calls == 1
        assert ms["overlay"] > 0 and ms["search"] > 0 and ms["update_state"] > 0, ms
    finally:
        bt.close()


# ---- the CPU oracle ------------------------------------------------------------------------------------------------------

def test_two_streams_against_oracle(torch_mod):
    """Streams 5 and 2, 24 frames interleaved in one batch with failing runs, frame counter drawn: records, out
    frames and masks against the CPU oracle run over each stream's frames; captured pixels of the last frames."""
    torch = torch_mod
    ids, specs = _two_streams(24)
    plans = {}
    for s, sp in zip(ids, specs):
        plans.setdefault(s, []).append(sp)
    keys = sorted(plans)
    want = dict(zip(keys, _oracle_pool_counted.run_jobs([dict(kind="plan", plan=plans[s]) for s in keys])))
    bt = _tracker(24, print_frame_count=True)
    bt.set_capture(True)
    try:
        d = _frames(torch, specs)
        out = torch.empty_like(d)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = bt.process(d, out, ids=ids, sequence=True)
        out = out.cpu().numpy()
        seen = {s: 0 for s in keys}
        for i, s in enumerate(ids):
            w, tag = want[s][seen[s]], (i, s)
            seen[s] += 1
            assert int(res[i]["counter"]) == w["counter"] and int(res[i]["attempts"]) == w["attempts"], tag
            assert bool(res[i]["valid_lane_lines"]) == w["valid"], tag
            assert int(res[i]["last_detection"]) == w["last_detection"], tag
            assert bool(res[i]["detected_pixels"]) == w["detected"], tag
            if w["detected"]:
                np.testing.assert_allclose(res[i]["left_fit"], w["left_fit"], rtol=FIT_RTOL, err_msg=str(tag))
                np.testing.assert_allclose(res[i]["right_fit"], w["right_fit"], rtol=FIT_RTOL, err_msg=str(tag))
            assert fx.sha(out[i]) == w["out"], tag
            assert fx.sha(bt.debug_read("mask", i)) == w["mask"], tag
        for s in keys:
            w = want[s][-1]
            if w["detected"]:
                sides, _ = bt.read_capture(s, w["attempts"] - 1)
                assert fx.pix_digest(sides[0][0], sides[0][1], sides[1][0], sides[1][1]) == w["pix"], s
        assert (res["attempts"] == 2).any() and res["valid_lane_lines"].any()
    finally:
        bt.close()


# ---- refusals ------------------------------------------------------------------------------------------------------------

def test_refusals(torch_mod):
    """Python: sequence=True without ids, with profiles or cameras, an id out of range, more frames than streams;
    repeated ids without sequence=True as before.  C: a null id list, n outside [1, S], an id out of range (naming
    the position).  Nothing is launched and no state changes."""
    from lane_tracker_b200 import DevicePipeline, HostPipeline, _lib
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    S = 6
    bt = _tracker(S)
    lib = _lib.load()
    try:
        bt.set_profile(0, make_params())
        d = _frames(torch, [_spec(s, 0, []) for s in (3, 3, 1, 3)])
        out = torch.empty_like(d)
        bt.process(d, out, ids=[3, 3, 1, 3], sequence=True)
        before = [_snapshot(bt, s, False) for s in range(S)]
        host = d.cpu().pin_memory()
        n0 = lib.lt_launch_count()
        cases = [(dict(sequence=True), "needs ids"),
                 (dict(ids=[3, 3, 1, 3], sequence=True, profiles=[0] * 4), "neither profiles nor cameras"),
                 (dict(ids=[3, 3, 1, 3], sequence=True, cameras=[0] * 4), "neither profiles nor cameras"),
                 (dict(ids=[3, 3, 6, 3], sequence=True), "stream id 6 outside"),
                 (dict(ids=[3, 3, 1], sequence=True), "3 stream ids for 4 frames"),
                 (dict(ids=[3, 3, 1, 3]), "appears more than once")]
        for kw, msg in cases:
            with pytest.raises(ValueError, match=msg):
                bt.process(d, out, **kw)
            with pytest.raises(ValueError, match=msg):
                bt.process_back_async(d, out, 0, **kw)
            with pytest.raises(ValueError, match=msg):
                DevicePipeline(bt).submit(d, out, **kw)
            with pytest.raises(ValueError, match=msg):
                HostPipeline(bt, depth=1).submit(host, **kw)
        big = _frames(torch, [["blank", 10 + s] for s in range(S + 1)])
        with pytest.raises(ValueError, match="frames for"):
            bt.process(big, ids=[0] * (S + 1), sequence=True)

        p = make_params()
        res = bt._results_dev
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        P = C.c_void_p
        for ids, n, msg in [([3, 3, 6, 1], 4, "stream id 6 at batch position 2"),
                            ([3, -1, 3, 1], 4, "stream id -1 at batch position 1"),
                            ([0] * (S + 1), S + 1, "n_streams 7 outside"), ([0], 0, "n_streams 0 outside"),
                            (None, 4, "null stream id list")]:
            arr = (C.c_int32 * len(ids))(*ids) if ids is not None else None
            src = big if n > 4 else d
            for call in (lambda: lib.lt_process_sequence(bt._h, P(src.data_ptr()), P(src.data_ptr()), arr, n,
                                                         C.byref(p), P(res.data_ptr()), st),
                         lambda: lib.lt_process_back_sequence(bt._h, P(src.data_ptr()), P(src.data_ptr()), arr, n,
                                                              C.byref(p), 0, P(res.data_ptr()), st)):
                assert call() < 0, (ids, n)
                assert msg in lib.lt_last_error().decode(), (msg, lib.lt_last_error())
        # the other checks of lt_process_streams apply: a misaligned d_out, a null d_results
        arr = (C.c_int32 * 4)(3, 3, 1, 3)
        assert lib.lt_process_sequence(bt._h, P(d.data_ptr()), P(out.data_ptr() + 1), arr, 4, C.byref(p),
                                       P(res.data_ptr()), st) < 0
        assert "d_out must be 4-byte aligned" in lib.lt_last_error().decode()
        assert lib.lt_process_sequence(bt._h, P(d.data_ptr()), P(out.data_ptr()), arr, 4, C.byref(p), None, st) < 0
        torch.cuda.synchronize()
        assert lib.lt_launch_count() == n0
        for s in range(S):
            assert _snapshot(bt, s, False) == before[s], s
    finally:
        bt.close()
