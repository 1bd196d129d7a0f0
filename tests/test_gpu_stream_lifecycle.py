"""Stream starts and state records: ``starts=`` of the process calls and the pipelines, ``reset_async``,
``export_states`` / ``import_states`` (C ABI: lt_reset_async, lt_state_record_bytes, lt_export_states,
lt_import_states).

The reference for a start is a second handle fed the same batches one call at a time, with a synchronous ``reset`` of
the started streams before the batch that carries their first new frame.  Result records, annotated frames and masks,
and every stream's state, polylines, cached polygon and captured pixel lists must be the same bytes.  A started
stream must also match a fresh handle fed only its new video, and one started stream runs through the CPU oracle."""
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


def _spec(video, t, fail=()):
    """Frame t of synthetic video `video`, or a photograph, a blank or a noise frame when t lies in a failing run."""
    if not any(a <= t < b for a, b in fail):
        return ["synth", video, t]
    kind = ("image", "blank", "noise", "image")[(video + t) % 4]
    if kind == "image":
        return ["image", PHOTOS[(video + t) % len(PHOTOS)]]
    if kind == "noise":
        return ["noise", 9000 + 100 * t + video % 100]
    return ["blank", 30 + (7 * video + t) % 200]


def _frames(torch, specs, nv12=False, device="cuda"):
    a = np.stack([frame_from_spec(sp) for sp in specs])
    return torch.as_tensor(synth.rgb_to_nv12(a) if nv12 else a).to(device)


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


class Plan:
    """Which video each stream plays: stream s plays video 3000 + s until it starts video `new` at batch b; t counts
    the frames of the current video."""

    def __init__(self, S, fail=()):
        self.video = {s: 3000 + s for s in range(S)}
        self.t = {s: 0 for s in range(S)}
        self.fail = fail

    def batch(self, ids, starts=None):
        specs = []
        for i, s in enumerate(ids):
            if starts is not None and starts[i]:
                self.video[s] = 5000 + 17 * s + self.video[s] % 7
                self.t[s] = 0
            specs.append(_spec(self.video[s], self.t[s], self.fail if s % 3 == 1 else ()))
            self.t[s] += 1
        return specs


def _reference(torch, b, frames, ids, starts, nv12=False, **kw):
    """The reference step: a synchronous reset of the started streams, then one process call -> (records, out)."""
    torch.cuda.synchronize()
    if starts is not None and any(starts):
        b.reset([int(s) for s, v in zip(ids, starts) if v])
    w, h = b.img_size
    out = torch.empty((len(ids), h, w, 3), dtype=torch.uint8, device="cuda")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = b.process(frames, out, ids=list(ids), **kw)
    return res, out.cpu().numpy()


def _same_streams(a, b, S, capture, tag=""):
    for s in range(S):
        assert _snapshot(a, s, capture) == _snapshot(b, s, capture), (tag, s)


# ---- starts inside a DevicePipeline ----------------------------------------------------------------------------------

def test_starts_in_device_pipeline(torch_mod):
    """16 streams, 12 batches through DevicePipeline with both buffer sets in flight.  At batch 5 streams 2 and 9
    start new videos; at batch 8 stream 4 starts in a batch that also carries failing frames.  Against the reference
    handle batch by batch; the started streams against fresh handles fed only their new videos, stream 2 against the
    CPU oracle."""
    from lane_tracker_b200 import DevicePipeline
    torch = torch_mod
    S = 16
    a = _tracker(S, print_frame_count=True)
    b = _tracker(S, print_frame_count=True)
    a.set_capture(True)
    b.set_capture(True)
    plan = Plan(S, fail=[(6, 9), (10, 11)])
    start_at = {5: (2, 9), 8: (4,)}
    started = {s: k for k, ss in start_at.items() for s in ss}
    new_specs = {s: [] for s in started}
    try:
        pipe = DevicePipeline(a)
        pending = None
        outs, recs, refs = [], [], []
        for k in range(12):
            ids = [int(v) for v in np.random.default_rng(k).permutation(S)]
            starts = [s in start_at.get(k, ()) for s in ids]
            specs = plan.batch(ids, starts)
            for i, s in enumerate(ids):
                if s in started and k >= started[s]:
                    new_specs[s].append((k, i, specs[i]))
            d = _frames(torch, specs)
            out = torch.empty_like(d)
            done = pipe.submit(d, out, ids=ids, starts=starts if any(starts) else None)
            if pending is not None:           # batch k-1, while batch k is in flight
                pd, pout, pk, pdone = pending
                pdone.synchronize()
                recs.append(a.fetch_results(pd, pipe.results_dev[pk & 1]))
                outs.append(pout.cpu().numpy())
            pending = (len(ids), out, k, done)
            refs.append(_reference(torch, b, d, ids, starts))
        pipe.join()
        pd, pout, pk, _ = pending
        recs.append(a.fetch_results(pd, pipe.results_dev[pk & 1]))
        outs.append(pout.cpu().numpy())
        for k in range(12):
            assert recs[k].tobytes() == refs[k][0].tobytes(), k
            assert np.array_equal(outs[k], refs[k][1]), k
        for i in range(S):
            assert np.array_equal(a.debug_read("mask", i), b.debug_read("mask", i)), i
        _same_streams(a, b, S, True)
        assert (np.concatenate(recs)["attempts"] == 2).any()
        # the started streams equal fresh handles fed only their new videos
        for s, items in new_specs.items():
            c = _tracker(S, print_frame_count=True)
            try:
                for k, i, sp in items:
                    res, out = _reference(torch, c, _frames(torch, [sp]), [s], None)
                    assert res[0].tobytes() == recs[k][i].tobytes(), (s, k)
                    assert np.array_equal(out[0], outs[k][i]), (s, k)
            finally:
                c.close()
        # stream 2 against the CPU oracle
        want = _oracle_pool_counted.run_jobs([dict(kind="plan", plan=[sp for _, _, sp in new_specs[2]])])[0]
        for (k, i, _), w in zip(new_specs[2], want):
            r = recs[k][i]
            assert int(r["counter"]) == w["counter"] and int(r["attempts"]) == w["attempts"], k
            assert bool(r["valid_lane_lines"]) == w["valid"] and int(r["last_detection"]) == w["last_detection"], k
            if w["detected"]:
                np.testing.assert_allclose(r["left_fit"], w["left_fit"], rtol=FIT_RTOL)
                np.testing.assert_allclose(r["right_fit"], w["right_fit"], rtol=FIT_RTOL)
            assert fx.sha(outs[k][i]) == w["out"], k
    finally:
        a.close()
        b.close()


# ---- starts in the other call forms ----------------------------------------------------------------------------------

def _camera1():
    """A camera mounted to see further ahead (rows of the bird's-eye view scaled by 0.8 about the bottom row)."""
    cal = synth.shipped_calibration()
    bh = synth.WARPED_SIZE[1]
    M = np.array([[1, 0, 0], [0, 0.8, 0.2 * (bh - 1)], [0, 0, 1.0]]) @ cal["warp_matrices"][0]
    cal["warp_matrices"] = (M, np.linalg.inv(M))
    cal["mpp_conversion"] = (synth.MPPV * 1.25, synth.MPPH)
    return cal


@pytest.mark.parametrize("form", ["host", "host_inplace", "nv12", "profiles", "cameras", "sequence", "remount"])
def test_starts_in_call_forms(torch_mod, form):
    """Four batches of 8 streams with starts in batches 1 and 2, through HostPipeline (in place or not), NV12 frames,
    profiles, cameras, a sequence batch (start at a stream's first position) and a stream re-mounted to another
    camera and started in the same batch; against the reference handle with synchronous resets."""
    from lane_tracker_b200 import HostPipeline
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    S = 8
    a, b = _tracker(S), _tracker(S)
    try:
        for t in (a, b):
            if form in ("cameras", "remount"):
                c = _camera1()
                t.set_camera(1, c["cam_matrix"], c["dist_coeffs"], c["warp_matrices"], c["mpp_conversion"])
            if form == "profiles":
                t.set_profile(0, make_params())
                t.set_profile(1, make_params(C_r=6, bandwidth=30))
        pipe = HostPipeline(a, depth=2, inplace=form == "host_inplace") if form.startswith("host") else None
        plan = Plan(S, fail=[(1, 3)])
        cam_of = {s: 0 for s in range(S)}
        for k in range(4):
            if form == "sequence":
                ids = [1, 1, 5, 1, 5, 2, 2, 6]
                starts = [k == 1 and i == 0, False, k == 2 and i == 2, False, False, k == 1 and i == 5, False, False]
                starts = [bool(v) for v in starts]
            else:
                ids = [int(v) for v in np.random.default_rng(10 + k).permutation(S)]
                starts = [(k == 1 and s in (0, 3)) or (k == 2 and s == 6) for s in ids]
            if form == "remount" and k == 2:
                cam_of[6] = 1                  # stream 6 re-mounted and started in the same batch
            kw = {}
            if form == "profiles":
                kw["profiles"] = [s % 2 for s in ids]
            if form == "cameras":
                kw["cameras"] = [s % 2 for s in ids]
            if form == "remount":
                kw["cameras"] = [cam_of[s] for s in ids]
            if form == "sequence":
                kw["sequence"] = True
            specs = plan.batch(ids, starts)
            d = _frames(torch, specs, nv12=form == "nv12")
            want, wout = _reference(torch, b, d, ids, starts, **kw)
            if pipe is not None:
                host = torch.as_tensor(np.stack([frame_from_spec(sp) for sp in specs])).pin_memory()
                pipe.submit(host, ids=ids, starts=starts, **kw)
                (out, res), = list(pipe.drain())
                res, out = res.copy(), out.numpy()
            else:
                w, h = a.img_size
                o = torch.empty((len(ids), h, w, 3), dtype=torch.uint8, device="cuda")
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    res = a.process(d, o, ids=ids, starts=starts, **kw)
                out = o.cpu().numpy()
                for i in range(len(ids)):
                    assert np.array_equal(a.debug_read("mask", i), b.debug_read("mask", i)), (form, k, i)
            assert res.tobytes() == want.tobytes(), (form, k)
            assert np.array_equal(out, wout), (form, k)
            _same_streams(a, b, S, False, (form, k))
    finally:
        a.close()
        b.close()


# ---- launch counts ----------------------------------------------------------------------------------------------------

def test_launch_counts(torch_mod):
    """Every call form enqueues the same launches with starts=None and with all-False starts, and exactly one more
    with starts (one k_reset_states launch per 1000 flagged streams).  That the no-starts path enqueues what the
    parent commit enqueued is not measured here: that path is unchanged code."""
    from lane_tracker_b200 import _lib
    from lane_tracker_b200.tracker import make_params
    torch = torch_mod
    lib = _lib.load()
    S = 8
    bt = _tracker(S)
    try:
        bt.set_profile(0, make_params())
        c = _camera1()
        bt.set_camera(1, c["cam_matrix"], c["dist_coeffs"], c["warp_matrices"], c["mpp_conversion"])
        d = _frames(torch, [_spec(3000 + s, 0) for s in range(S)])
        out = torch.empty_like(d)
        ids = [7, 2, 5, 0, 1, 3, 4, 6]
        forms = [dict(), dict(ids=ids), dict(ids=ids, profiles=[0] * S), dict(ids=ids, cameras=[0, 1] * 4),
                 dict(ids=[1, 1, 2, 2, 3, 3, 4, 4], sequence=True)]

        def count(fn):
            torch.cuda.synchronize()
            c0 = lib.lt_launch_count()
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                fn()
            return lib.lt_launch_count() - c0

        for kw in forms:
            for back in (False, True):
                def call(starts):
                    if back:
                        bt.process_front_async(d, 1, profiles=kw.get("profiles"), cameras=kw.get("cameras"))
                        bt.process_back_async(d, out, 1, starts=starts, **kw)
                    else:
                        bt.process_async(d, out, starts=starts, **kw)
                n0 = count(lambda: call(None))
                assert count(lambda: call([False] * S)) == n0, kw
                one = [i in (0, 4) for i in range(S)] if not kw.get("sequence") else [i in (0, 2) for i in range(S)]
                assert count(lambda: call(one)) == n0 + 1, kw
        assert count(lambda: bt.reset_async()) == 1
        assert count(lambda: bt.reset_async([3, 1])) == 1
    finally:
        bt.close()


# ---- graph capture ------------------------------------------------------------------------------------------------------

def test_cuda_graph_capture(torch_mod):
    """reset_async + process_async + export_states captured once in torch.cuda.graph and replayed over three batches:
    the same records, frames and state records as the same calls made eagerly on a second handle."""
    from lane_tracker_b200.tracker import RESULT_DTYPE
    torch = torch_mod
    S, n = 8, 8
    a, b = _tracker(S), _tracker(S)
    try:
        plan = Plan(S)
        ids = list(range(n))
        static = _frames(torch, plan.batch(ids))
        out = torch.empty_like(static)
        resd = torch.zeros(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        rec = torch.empty((2, a.record_bytes), dtype=torch.uint8, device="cuda")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for t in (a, b):                  # warm-up of both handles (first launches load the kernels)
                t.process_async(static, out, results_dev=resd)
                t.reset_async([0])
                t.export_states([0])
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                a.reset_async([3, 6])
                a.process_async(static, out, results_dev=resd)
                a.export_states([3, 6], out=rec)
            for r in range(3):
                d = _frames(torch, plan.batch(ids))
                static.copy_(d)
                g.replay()
                torch.cuda.synchronize()
                got, gout, grec = a.fetch_results(n, resd), out.cpu().numpy(), rec.cpu().numpy()
                b.reset_async([3, 6])
                wout = torch.empty_like(d)
                want = b.process(d, wout)
                wrec = b.export_states([3, 6]).cpu().numpy()
                assert got.tobytes() == want.tobytes(), r
                assert np.array_equal(gout, wout.cpu().numpy()), r
                assert np.array_equal(grec, wrec), r
                _same_streams(a, b, S, False, r)
    finally:
        a.close()
        b.close()


# ---- state records ------------------------------------------------------------------------------------------------------

def _run(torch, t, frames, ids):
    w, h = t.img_size
    out = torch.empty((len(ids), h, w, 3), dtype=torch.uint8, device=frames.device)
    with torch.cuda.device(frames.device), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = t.process(frames, out, ids=ids)
    return res, out.cpu().numpy()


def test_state_records_move_streams(torch_mod):
    """Handle A runs 8 batches through DevicePipeline; streams 3 and 5 are exported while its last batch is in flight
    and imported into slots 0 and 1 of handle B (and of a handle on cuda:1 when there is one).  Then A (streams 3, 5)
    and B (slots 0, 1) run the same 8 frames: identical records, frames and state bytes.  Export -> import -> export
    gives identical bytes."""
    from lane_tracker_b200 import DevicePipeline
    torch = torch_mod
    S = 8
    a, b = _tracker(S), _tracker(4)
    extra = []
    try:
        pipe = DevicePipeline(a)
        plan = Plan(S, fail=[(2, 4)])
        for k in range(8):
            pipe.submit(_frames(torch, plan.batch(list(range(S)))), ids=list(range(S)))
        rec, ev = pipe.export_states([3, 5])
        assert tuple(rec.shape) == (2, a.record_bytes) and a.record_bytes % 16 == 0
        assert a.record_bytes == 64 + 640 + 16 * synth.WARPED_SIZE[1] + 16
        ev.synchronize()
        status = b.import_states([0, 1], rec)
        assert status.cpu().tolist() == [0, 0]
        assert np.array_equal(b.export_states([0, 1]).cpu().numpy(), rec.cpu().numpy())
        targets = [(b, "cuda", rec)]
        if torch.cuda.device_count() > 1:
            c = _tracker(4, device=1)
            extra.append(c)
            rec1 = rec.to("cuda:1")
            with torch.cuda.device(1):
                c.import_states([0, 1], rec1)
                assert np.array_equal(c.export_states([0, 1]).cpu().numpy(), rec.cpu().numpy())
            targets.append((c, "cuda:1", rec1))
        for s, slot in ((3, 0), (5, 1)):
            for t, _, _ in targets:
                assert _snapshot(a, s, False) == _snapshot(t, slot, False), (s, slot)
        for k in range(8):
            specs = plan.batch([3, 5])
            ra, oa = _run(torch, a, _frames(torch, specs), [3, 5])
            for t, dev, _ in targets:
                rt, ot = _run(torch, t, _frames(torch, specs, device=dev), [0, 1])
                assert ra.tobytes() == rt.tobytes(), (k, dev)
                assert np.array_equal(oa, ot), (k, dev)
        for s, slot in ((3, 0), (5, 1)):
            for t, _, _ in targets:
                assert _snapshot(a, s, False) == _snapshot(t, slot, False), (s, slot)
        assert ra["valid_lane_lines"].any()
    finally:
        for t in [a, b] + extra:
            t.close()


def test_import_refusals(torch_mod):
    """Records from a handle with another bv_h or n_average, and records whose ring_len or n_left_avg was corrupted:
    status nonzero, the slot keeps its bytes, import_states(check=True) raises naming the position."""
    from lane_tracker_b200 import _lib
    torch = torch_mod
    a = _tracker(4)
    try:
        plan = Plan(4)
        for k in range(3):
            _run(torch, a, _frames(torch, plan.batch([0, 1, 2, 3])), [0, 1, 2, 3])
        before = [_snapshot(a, s, False) for s in range(4)]
        good = a.export_states([0, 1, 2, 3])
        ring = 64 + _lib.lt_state.ring_len.offset
        nla = 64 + _lib.lt_state.n_left_avg.offset
        bad = good.clone()
        bad[1, ring:ring + 4] = torch.tensor([99, 0, 0, 0], dtype=torch.uint8)
        bad[3, nla:nla + 4] = torch.tensor([0xFF, 0xFF, 0xFF, 0x7F], dtype=torch.uint8)
        tgt = _tracker(4)
        try:
            for s in range(4):
                tgt.reset_async([s])
            tb = [_snapshot(tgt, s, False) for s in range(4)]
            st = tgt.import_states([3, 2, 1, 0], bad, check=False)
            assert st.cpu().tolist() == [0, _lib.LT_RECORD_BAD_STATE, 0, _lib.LT_RECORD_BAD_STATE]
            assert _snapshot(tgt, 2, False) == tb[2] and _snapshot(tgt, 0, False) == tb[0]
            assert _snapshot(tgt, 3, False) == before[0] and _snapshot(tgt, 1, False) == before[2]
            with pytest.raises(ValueError, match="position 1 .stream 2. refused: its state is inconsistent"):
                tgt.import_states([3, 2, 1, 0], bad)
            # a non-empty polygon row reaching past the bird's-eye view, and a non-empty box reaching past it
            W, H = synth.WARPED_SIZE
            rows = 64 + (C.sizeof(_lib.lt_state) + 15) // 16 * 16 + 8 * H
            box = (rows + 8 * H + 15) // 16 * 16
            geo = good.clone()
            geo[0, rows + 8 * 5:rows + 8 * 6] = torch.tensor(np.array([W - 10, W + 5], np.int32).view(np.uint8),
                                                             device="cuda")
            geo[2, box:box + 16] = torch.tensor(np.array([0, W, 0, 10], np.int32).view(np.uint8), device="cuda")
            tb = [_snapshot(tgt, s, False) for s in range(4)]
            st = tgt.import_states([2, 0], geo[[0, 2]].contiguous(), check=False)
            assert st.cpu().tolist() == [_lib.LT_RECORD_BAD_STATE] * 2
            for s in range(4):
                assert _snapshot(tgt, s, False) == tb[s], s
            st = tgt.import_states([2, 0], geo[[1, 3]].contiguous(), check=False)     # the untouched records pass
            assert st.cpu().tolist() == [0, 0]
        finally:
            tgt.close()
        small = _tracker(4, cal=synth.shipped_calibration(0.5))
        avg3 = _tracker(4, n_average=3)
        try:
            for t in (avg3, small):
                tb = [_snapshot(t, s, False) for s in range(4)]
                if t is small:
                    rec = torch.zeros((4, t.record_bytes), dtype=torch.uint8, device="cuda")
                    rec[:, :t.record_bytes] = good[:, :t.record_bytes]
                else:
                    rec = good
                st = t.import_states([0, 1, 2, 3], rec, check=False)
                assert st.cpu().tolist() == [_lib.LT_RECORD_BAD_HEADER] * 4
                for s in range(4):
                    assert _snapshot(t, s, False) == tb[s], s
                with pytest.raises(ValueError, match="position 0 .stream 0. refused: its header"):
                    t.import_states([0, 1, 2, 3], rec)
        finally:
            small.close()
            avg3.close()
        for s in range(4):
            assert _snapshot(a, s, False) == before[s]
    finally:
        a.close()


def test_refusals_before_anything_is_enqueued(torch_mod):
    """Bad ids, lengths, buffers and starts are refused before anything is enqueued: the launch count and every
    stream's state are unchanged."""
    from lane_tracker_b200 import DevicePipeline, HostPipeline, _lib
    torch = torch_mod
    lib = _lib.load()
    S = 6
    bt = _tracker(S)
    try:
        d = _frames(torch, [_spec(3000 + s, 0) for s in range(4)])
        out = torch.empty_like(d)
        bt.process(d, out, ids=[3, 1, 0, 2])
        before = [_snapshot(bt, s, False) for s in range(S)]
        rec = bt.export_states([0, 1])
        torch.cuda.synchronize()
        host = d.cpu().pin_memory()
        n0 = lib.lt_launch_count()
        cases = [(dict(starts=[True, False]), "2 starts for 4 frames"),
                 (dict(starts=[1, 0, 0, 0]), "starts must be bools"),
                 (dict(ids=[3, 3, 1, 3], sequence=True, starts=[False, True, False, False]), "split the batch there"),
                 (dict(ids=[3, 1, 0, 9], starts=[True] * 4), "stream id 9 outside")]
        for kw, msg in cases:
            with pytest.raises(ValueError, match=msg):
                bt.process(d, out, **kw)
            with pytest.raises(ValueError, match=msg):
                bt.process_back_async(d, out, 0, **kw)
            with pytest.raises(ValueError, match=msg):
                DevicePipeline(bt).submit(d, out, **kw)
            with pytest.raises(ValueError, match=msg):
                HostPipeline(bt, depth=1).submit(host, **kw)
        with pytest.raises(ValueError, match="appears more than once"):
            bt.reset_async([1, 1])
        with pytest.raises(ValueError, match="outside"):
            bt.export_states([0, 6])
        with pytest.raises(ValueError, match="must be a contiguous uint8 tensor"):
            bt.import_states([0, 1, 2], rec)
        with pytest.raises(ValueError, match="16-byte aligned"):
            flat = torch.empty(2 * bt.record_bytes + 16, dtype=torch.uint8, device="cuda")
            bt.import_states([0, 1], flat[8:8 + 2 * bt.record_bytes].view(2, bt.record_bytes))
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        P = C.c_void_p
        for ids, n, msg in [([3, 9], 2, "stream id 9 at batch position 1"), ([4, 2, 4], 3, "appears twice"),
                            ([0] * (S + 1), S + 1, "n_streams 7 outside"), ([0], 0, "n_streams 0 outside")]:
            arr = (C.c_int32 * len(ids))(*ids)
            assert lib.lt_reset_async(bt._h, arr, n, st) < 0 and msg in lib.lt_last_error().decode(), msg
            assert lib.lt_export_states(bt._h, arr, n, P(rec.data_ptr()), st) < 0 and msg in lib.lt_last_error().decode()
            assert lib.lt_import_states(bt._h, arr, n, P(rec.data_ptr()), None, st) < 0
            assert msg in lib.lt_last_error().decode(), msg
        arr = (C.c_int32 * 2)(0, 1)
        assert lib.lt_export_states(bt._h, arr, 2, P(rec.data_ptr() + 4), st) < 0
        assert "16-byte aligned" in lib.lt_last_error().decode()
        assert lib.lt_import_states(bt._h, arr, 2, None, None, st) < 0
        assert lib.lt_export_states(bt._h, None, 2, P(rec.data_ptr()), st) < 0
        torch.cuda.synchronize()
        assert lib.lt_launch_count() == n0
        for s in range(S):
            assert _snapshot(bt, s, False) == before[s], s
    finally:
        bt.close()


# ---- GraphedProcess -----------------------------------------------------------------------------------------------------

def test_graphed_process_keeps_the_state(torch_mod):
    """A GraphedProcess built mid-video (its warm-up run between an export and an import of the state records) leaves
    every stream's state records, polylines and cached polygon unchanged, and its replays continue the videos."""
    from lane_tracker_b200 import GraphedProcess
    torch = torch_mod
    S = 6
    a, b = _tracker(S), _tracker(S)
    try:
        plan = Plan(S, fail=[(3, 4)])
        for k in range(5):
            d = _frames(torch, plan.batch(list(range(S))))
            _run(torch, a, d, list(range(S)))
            _run(torch, b, d, list(range(S)))
        rec = a.export_states(range(S)).cpu().numpy()
        snaps = [_snapshot(a, s, False) for s in range(S)]
        g = GraphedProcess(a, S)
        torch.cuda.synchronize()
        assert np.array_equal(a.export_states(range(S)).cpu().numpy(), rec)
        for s in range(S):
            assert _snapshot(a, s, False) == snaps[s], s
        for k in range(2):
            d = _frames(torch, plan.batch(list(range(S))))
            g.frames.copy_(d)
            g.replay()
            got = g.fetch_results()
            want, wout = _run(torch, b, d, list(range(S)))
            assert got.tobytes() == want.tobytes() and np.array_equal(g.out.cpu().numpy(), wout), k
    finally:
        a.close()
        b.close()
