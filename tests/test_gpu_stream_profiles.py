"""Parameter profiles: every frame of a batch with its own lt_params and check_validity windows (``set_profile`` and
``profiles=`` of ``BatchedLaneTracker.process`` and the pipelines; C ABI: lt_set_profile, lt_process_profiles,
lt_process_front_profiles, lt_process_back_profiles).

Two references.  The GPU reference is a second handle that runs, per profile, ``process(..., ids=...)`` with that
profile's params and windows over exactly the frames that used it (per-stream results do not depend on batch
composition: tests/test_gpu_stream_ids.py).  The CPU anchor is the oracle (tests/_oracle_pool_profiles.py) run per
stream over the frames it received, each with the settings of its profile.  Compared as in the stream-id tests: result
records, final masks per position, annotated frames, state, averaged polylines and cached lane rows per stream id and
captured pixel lists bit for bit; against the oracle, fit coefficients within 1e-6 relative.  Every stream carries
distinct content: road videos of distinct seeds, photographs (which take the second attempt), noise and blank frames.
"""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

import _fixtures as fx
import _oracle_pool_profiles
from _oracle_pool import frame_from_spec
from lane_tracker_b200 import presets, synth
from lane_tracker_b200.tracker import RESULT_DTYPE

pytestmark = pytest.mark.gpu

FIT_RTOL = 1e-6
PHOTOS = fx.frame_names()

# (process() keywords, validity windows or None for the shipped ones)
DEFAULTS = ({}, None)
DEMO_1 = (presets.DEMO_1["process"], presets.DEMO_1["validity"])
DEMO_2 = (presets.DEMO_2["process"], presets.DEMO_2["validity"])
DEMO_3 = (presets.DEMO_3["process"], presets.DEMO_3["validity"])


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)


def _tracker(S, **kw):
    from lane_tracker_b200 import BatchedLaneTracker
    return BatchedLaneTracker(S, **synth.shipped_calibration(), **kw)


def _batch(torch, specs):
    return torch.as_tensor(np.stack([frame_from_spec(sp) for sp in specs])).cuda()


def _install(bt, profiles):
    for k, (kw, val) in profiles.items():
        bt.set_profile(k, validity=val, **kw)


def _failing(s, r):
    kind = ("image", "blank", "noise")[(s + r) % 3]
    if kind == "image":
        return ["image", PHOTOS[(s + 3 * r) % len(PHOTOS)]]
    if kind == "noise":
        return ["noise", 9000 + 100 * r + s]
    return ["blank", 20 + (11 * s + r) % 200]


def _specs(ids, r, seen, seed0, fail):
    """Frame specs of one round: stream s gets frame seen[s] of its own road video unless it is in `fail`.  Photos
    repeat across streams of a round here; distinct positions still differ in their stream's history."""
    out = []
    for s in ids:
        out.append(_failing(s, r) if s in fail else ["synth", seed0 + s, seen[s]])
        seen[s] += 1
    return out


def _state(bt, s):
    st, lx, rx = bt.get_state(s)
    return [bytes(st), lx.tobytes(), rx.tobytes(), bt.debug_read("lane_rows", s).tobytes()]


def _captures(bt, s):
    out = []
    for attempt in (0, 1):
        sides, cents = bt.read_capture(s, attempt)
        out.append(([(y.tobytes(), x.tobytes()) for y, x in sides], cents))
    return out


class Reference:
    """The GPU reference: per profile, process(ids=...) with its params and windows over the frames that used it."""

    def __init__(self, S, profiles, capture=False, **kw):
        self.bt = _tracker(S, **kw)
        self.profiles = profiles
        self.capture = capture
        if capture:
            self.bt.set_capture(True)

    def step(self, torch, d, ids, prof, overlay=True):
        """-> (records, out frames or None, masks per position, captures per stream id) in batch order."""
        n = len(ids)
        recs = np.zeros(n, dtype=RESULT_DTYPE)
        out = torch.empty_like(d) if overlay else None
        masks, caps = [None] * n, {}
        prof = np.asarray(prof)
        for k in sorted(set(int(v) for v in prof)):
            pos = np.flatnonzero(prof == k)
            kw, val = self.profiles[k]
            if val is None:
                self.bt.set_validity()
            else:
                self.bt.set_validity(**val)
            sub = d[torch.as_tensor(pos).cuda()].contiguous()
            so = torch.empty_like(sub) if overlay else None
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                recs[pos] = self.bt.process(sub, so, ids=[int(ids[p]) for p in pos], **kw)
            if overlay:
                out[torch.as_tensor(pos).cuda()] = so
            for j, p in enumerate(pos):
                masks[p] = self.bt.debug_read("mask", j)
                if self.capture:
                    caps[int(ids[p])] = _captures(self.bt, int(ids[p]))
        return recs, out, masks, caps

    def close(self):
        self.bt.close()


def _compare(bt, ref_step, res, out, ids, tag, masks=True):
    recs, rout, rmasks, rcaps = ref_step
    assert res.tobytes() == recs.tobytes(), tag
    if out is not None:
        assert np.array_equal(out.cpu().numpy(), rout.cpu().numpy()), tag
    for i, s in enumerate(int(v) for v in ids):
        if masks:
            assert np.array_equal(bt.debug_read("mask", i), rmasks[i]), (tag, i, s)
        if rcaps:
            assert _captures(bt, s) == rcaps[s], (tag, i, s)


def _compare_states(bt, ref, S, tag):
    for s in range(S):
        assert _state(bt, s) == _state(ref.bt, s), (tag, s)


def _check_oracle_record(res, want, tag):
    assert int(res["counter"]) == want["counter"], tag
    assert int(res["success"]) == want["success"], tag
    assert int(res["attempts"]) == want["attempts"], tag
    assert int(res["search_mode"]) == (1 if want["mode"] == "bs" else 0), tag
    assert bool(res["detected_pixels"]) == want["detected"], tag
    assert bool(res["valid_lane_lines"]) == want["valid"], tag
    assert int(res["last_detection"]) == want["last_detection"], tag
    assert bool(res["first_valid"]) == want["first_valid"], tag
    if want["detected"]:
        assert int(res["n_left"]) == want["n_left"] and int(res["n_right"]) == want["n_right"], tag
        np.testing.assert_allclose(res["left_fit"], want["left_fit"], rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_fit"], want["right_fit"], rtol=FIT_RTOL, err_msg=str(tag))
    if want["valid"]:
        assert int(res["average_curve_radius"]) == want["radius"], tag
        np.testing.assert_allclose(res["left_avg"], want["left_avg"], rtol=FIT_RTOL, err_msg=str(tag))
        np.testing.assert_allclose(res["right_avg"], want["right_avg"], rtol=FIT_RTOL, err_msg=str(tag))


def _oracle_entry(spec, profile):
    kw, val = profile
    return list(spec) + [dict(params=dict(kw), validity=dict(val or presets.SHIPPED_VALIDITY))]


def _oracle(plans):
    """plans: {stream: [(spec, profile), ...]} -> {stream: [oracle record per frame]}."""
    keys = sorted(plans)
    res = _oracle_pool_profiles.run_jobs([dict(kind="plan", plan=[_oracle_entry(sp, pr) for sp, pr in plans[s]])
                                          for s in keys])
    return dict(zip(keys, res))


# ---- 1. one profile equals plain process -----------------------------------------------------------------------------

@pytest.mark.parametrize("S,profile", [(64, "defaults"), (17, "demo1")])
def test_one_profile_equals_plain_process(torch_mod, S, profile):
    """Two handles, scattered ids, four rounds: one with process(ids=..., **params) (+ set_validity), the other with
    one profile holding the same settings.  Records, out frames, masks, state of every stream and captures are the
    same bytes: the single-group path is lt_process."""
    torch = torch_mod
    kw, val = DEFAULTS if profile == "defaults" else DEMO_1
    a, b = _tracker(S), _tracker(S)
    a.set_capture(True)
    b.set_capture(True)
    if val is not None:
        a.set_validity(**val)
    b.set_profile(5, validity=val, **kw)
    rng = np.random.default_rng(S)
    seen = [0] * S
    try:
        for r, m in enumerate((S, S // 2 + 1, S, 3)):
            ids = [int(v) for v in rng.permutation(S)[:m]]
            d = _batch(torch, _specs(ids, r, seen, 2000, {s for s in ids if s % 4 == r % 4}))
            oa, ob = torch.empty_like(d), torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ra = a.process(d, oa, ids=ids, **kw)
                ma = [a.debug_read("mask", i) for i in range(m)]
                rb = b.process(d, ob, ids=ids, profiles=[5] * m)
            assert ra.tobytes() == rb.tobytes(), r
            assert torch.equal(oa, ob), r
            for i in range(m):
                assert np.array_equal(ma[i], b.debug_read("mask", i)), (r, i)
            for s in range(S):
                assert _state(a, s) == _state(b, s), (r, s)
            for s in ids:
                assert _captures(a, s) == _captures(b, s), (r, s)
    finally:
        a.close()
        b.close()


# ---- 2. the documented presets interleaved, through DevicePipeline ---------------------------------------------------

def test_presets_interleaved_device_pipeline(torch_mod):
    """64 streams, 6 frames through DevicePipeline, profiles 0..3 = defaults, DEMO_1, DEMO_2, DEMO_3 interleaved by
    position with unequal group sizes (DEMO_1 and DEMO_3 share a filter configuration, so three filter groups).  Against
    the GPU reference every round, and the CPU oracle for two streams per profile."""
    from lane_tracker_b200 import DevicePipeline
    torch = torch_mod
    S, T = 64, 6
    profiles = {0: DEFAULTS, 1: DEMO_1, 2: DEMO_2, 3: DEMO_3}
    rng = np.random.default_rng(5)
    profile_of = rng.choice(4, size=S, p=[0.4, 0.1, 0.2, 0.3])
    sizes = np.bincount(profile_of, minlength=4)
    assert sizes.min() >= 2 and len(set(sizes.tolist())) == 4, sizes
    anchors = {int(s) for k in range(4) for s in np.flatnonzero(profile_of == k)[:2]}
    bt = _tracker(S)
    _install(bt, profiles)
    ref = Reference(S, profiles)
    pipe = DevicePipeline(bt)
    seen, plans = [0] * S, {s: [] for s in anchors}
    outs = []
    try:
        for r in range(T):
            ids = [int(v) for v in rng.permutation(S)]
            specs = _specs(ids, r, seen, 3000, {s for s in ids if (s + r) % 5 == 0})
            prof = [int(profile_of[s]) for s in ids]
            d = _batch(torch, specs)
            out = torch.empty_like(d)
            pipe.submit(d, out, ids=ids, profiles=prof)
            res = pipe.fetch_results(len(ids))
            step = ref.step(torch, d, ids, prof)
            _compare(bt, step, res, out, ids, r)
            _compare_states(bt, ref, S, r)
            outs.append((ids, res, out.cpu().numpy()))
            for i, s in enumerate(ids):
                if s in anchors:
                    plans[s].append((specs[i], profiles[prof[i]]))
        want = _oracle(plans)
        retries = 0
        for r, (ids, res, out) in enumerate(outs):
            for i, s in enumerate(ids):
                retries += int(res[i]["attempts"] == 2)
                if s in anchors:
                    _check_oracle_record(res[i], want[s][r], (r, i, s))
                    assert fx.sha(out[i]) == want[s][r]["out"], (r, i, s)
        assert retries > 0
    finally:
        ref.close()
        bt.close()


# ---- 3. filter-only differences at 33 streams ------------------------------------------------------------------------

FILTER_CASES = {
    # the vertical threshold takes the TMA kernel up to k = 40 and the cp.async ring above
    "tma_limit": [dict(ksize_b=40), dict(ksize_b=41), dict(ksize_r=40, ksize_b=41)],
    # k > 127: the threshold sums no longer fit packed u16 lanes
    "unpacked": [dict(ksize_r=131), {}, dict(ksize_b=201)],
    # neighbourhood groups get no morphology; the bilateral ones take it over a position list
    "bilateral_neighbourhood": [dict(filter_type="neighborhood"), {}, dict(filter_type="neighborhood", ksize_r=21)],
    # the group key includes the noise fields
    "noise_thresh": [dict(mask_noise=True, noise_thresh=100), dict(mask_noise=True), {}],
}


@pytest.mark.parametrize("case", sorted(FILTER_CASES))
def test_filter_groups(torch_mod, case):
    """33 streams, profiles that differ in filter settings only, group sizes 1, 15 and 17 scattered over the batch
    (scattered ids, three rounds), capture on.  Against the GPU reference; the bilateral / neighbourhood case also
    against the CPU oracle for one stream per profile."""
    torch = torch_mod
    S = 33
    profiles = {k: (kw, None) for k, kw in enumerate(FILTER_CASES[case])}
    rng = np.random.default_rng(len(case))
    bt = _tracker(S)
    bt.set_capture(True)
    _install(bt, profiles)
    ref = Reference(S, profiles, capture=True)
    seen = [0] * S
    plans, outs = {}, []
    try:
        for r in range(3):
            ids = [int(v) for v in rng.permutation(S)]
            prof = rng.permutation([0] + [1] * 15 + [2] * 17).tolist()
            specs = _specs(ids, r, seen, 4000, {s for s in ids if (s + r) % 6 == 0})
            d = _batch(torch, specs)
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, ids=ids, profiles=prof)
            _compare(bt, ref.step(torch, d, ids, prof), res, out, ids, (case, r))
            _compare_states(bt, ref, S, (case, r))
            outs.append((ids, res, out.cpu().numpy()))
            if case == "bilateral_neighbourhood":
                for i, s in enumerate(ids):
                    if s < 6:
                        plans.setdefault(s, []).append((specs[i], profiles[prof[i]]))
        if plans:
            want = _oracle(plans)
            done = {s: 0 for s in plans}
            for r, (ids, res, out) in enumerate(outs):
                for i, s in enumerate(ids):
                    if s in plans:
                        w = want[s][done[s]]
                        _check_oracle_record(res[i], w, (r, i, s))
                        assert fx.sha(out[i]) == w["out"], (r, i, s)
                        done[s] += 1
    finally:
        ref.close()
        bt.close()


# ---- 4. profiles follow batch positions, not stream ids --------------------------------------------------------------

def test_profile_follows_position_not_stream(torch_mod):
    """24 streams, four rounds of scattered ids, profile = position % 3 where the three profiles differ in search
    settings, validity windows and n_tries only (one filter group).  The position of every frame takes a stream id with
    id % 3 != position % 3, so a kernel that looked the profile up by stream id would use another profile everywhere."""
    torch = torch_mod
    S = 24
    profiles = {0: ({}, None),
                1: (dict(window_width=40, partial=0.5, n_tries=1), presets.DEMO_3["validity"]),
                2: (dict(search_range=10, bandwidth=20, mu=0.2), presets.DEMO_1["validity"])}
    rng = np.random.default_rng(44)
    bt = _tracker(S)
    bt.set_capture(True)
    _install(bt, profiles)
    ref = Reference(S, profiles, capture=True)
    seen = [0] * S
    try:
        for r in range(4):
            # positions i with i % 3 == c take the streams s with s % 3 == (c + 1 + r % 2) % 3, shuffled
            pools = {c: list(rng.permutation(np.arange((c + 1 + r % 2) % 3, S, 3))) for c in range(3)}
            ids = [int(pools[i % 3].pop()) for i in range(S)]
            prof = [i % 3 for i in range(S)]
            assert sorted(ids) == list(range(S)) and all(prof[i] != ids[i] % 3 for i in range(S))
            d = _batch(torch, _specs(ids, r, seen, 5000, {s for s in ids if (s + r) % 4 == 0}))
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, ids=ids, profiles=prof)
            _compare(bt, ref.step(torch, d, ids, prof), res, out, ids, r)
            _compare_states(bt, ref, S, r)
            assert not (res["attempts"][1::3] == 2).any()          # profile 1: n_tries = 1
    finally:
        ref.close()
        bt.close()


# ---- 5. attempt 2 under the profile's windows, n_tries per position ---------------------------------------------------

def test_second_attempt_uses_profile_windows(torch_mod):
    """12 streams, photographs (which fail attempt 1) and road frames under three profiles: DEMO_3 windows with
    n_tries = 2, DEMO_3 windows with n_tries = 1, the shipped windows with n_tries = 2.  Against the GPU reference and
    the CPU oracle for every stream."""
    torch = torch_mod
    S = 12
    profiles = {0: ({}, presets.DEMO_3["validity"]), 1: (dict(n_tries=1), presets.DEMO_3["validity"]), 2: ({}, None)}
    bt = _tracker(S)
    _install(bt, profiles)
    ref = Reference(S, profiles)
    plans = {s: [] for s in range(S)}
    outs = []
    try:
        for r in range(3):
            ids = list(range(S))
            # photograph offset 2: every oracle fit of this plan rests on >= 235 lane pixels.  With offset 0, a band
            # search on a photograph after a tracked frame finds 24 pixels on a few rows, whose fit the moment-based
            # solver rounds differently from np.polyfit by more than FIT_RTOL (the GPU reference agrees bit for bit).
            specs = [["image", PHOTOS[(s + r + 2) % len(PHOTOS)]] if (s + r) % 3 else ["synth", 6000 + s, r] for s in ids]
            prof = [(s + r) % 3 for s in ids]
            d = _batch(torch, specs)
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, ids=ids, profiles=prof)
            _compare(bt, ref.step(torch, d, ids, prof), res, out, ids, r)
            _compare_states(bt, ref, S, r)
            outs.append((res, out.cpu().numpy(), prof))
            for s in ids:
                plans[s].append((specs[s], profiles[prof[s]]))
        want = _oracle(plans)
        att2 = {0: 0, 1: 0, 2: 0}
        for r, (res, out, prof) in enumerate(outs):
            for s in range(S):
                _check_oracle_record(res[s], want[s][r], (r, s))
                assert fx.sha(out[s]) == want[s][r]["out"], (r, s)
                att2[prof[s]] += int(res[s]["attempts"] == 2)
        assert att2[0] > 0 and att2[2] > 0 and att2[1] == 0, att2
    finally:
        ref.close()
        bt.close()


# ---- 6. a stream that switches profile every frame -------------------------------------------------------------------

def test_stream_switches_profile_every_frame(torch_mod):
    """8 streams, 5 frames, stream s uses profile (s + t) % 4 at frame t (defaults, DEMO_1, DEMO_2, DEMO_3): its
    tracking state carries over between profiles as in the reference called with changing keyword options.  Against
    the CPU oracle for every stream."""
    torch = torch_mod
    S, T = 8, 5
    profiles = {0: DEFAULTS, 1: DEMO_1, 2: DEMO_2, 3: DEMO_3}
    bt = _tracker(S)
    _install(bt, profiles)
    plans = {s: [] for s in range(S)}
    outs = []
    try:
        for t in range(T):
            ids = [int(v) for v in np.random.default_rng(t).permutation(S)]
            specs = [_failing(s, t) if t == 2 and s % 2 else ["synth", 7000 + s, t] for s in ids]
            prof = [(s + t) % 4 for s in ids]
            d = _batch(torch, specs)
            out = torch.empty_like(d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = bt.process(d, out, ids=ids, profiles=prof)
            outs.append((ids, res, out.cpu().numpy(), [bt.debug_read("mask", i) for i in range(S)]))
            for i, s in enumerate(ids):
                plans[s].append((specs[i], profiles[prof[i]]))
        want = _oracle(plans)
        for t, (ids, res, out, masks) in enumerate(outs):
            for i, s in enumerate(ids):
                _check_oracle_record(res[i], want[s][t], (t, i, s))
                assert fx.sha(out[i]) == want[s][t]["out"], (t, i, s)
                assert fx.sha(masks[i]) == want[s][t]["mask"], (t, i, s)
    finally:
        bt.close()


# ---- 7. the front half's snapshot ------------------------------------------------------------------------------------

def test_back_half_uses_front_snapshot(torch_mod):
    """set_profile between front and back of a batch: that batch runs on the old table, the next on the new one."""
    torch = torch_mod
    S = 16
    old, new = DEFAULTS, DEMO_2          # different filter, bandwidth, n_tries and windows
    bt = _tracker(S)
    bt.set_capture(True)
    _install(bt, {0: old})
    ref = _tracker(S)
    ref.set_capture(True)
    seen = [0] * S
    try:
        ids = list(range(S))
        d1 = _batch(torch, _specs(ids, 0, seen, 8000, {1, 5, 9}))
        d2 = _batch(torch, _specs(ids, 1, seen, 8000, {2, 6}))
        o1, o2 = torch.empty_like(d1), torch.empty_like(d2)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            bt.process_front_async(d1, 0, profiles=[0] * S)
            _install(bt, {0: new})
            bt.process_back_async(d1, o1, 0, profiles=[0] * S)
            r1 = bt.fetch_results(S)
            m1 = [bt.debug_read("mask", i) for i in range(S)]
            r2 = bt.process(d2, o2, profiles=[0] * S)
            w1 = ref.process(d1, None, **old[0])
            wm = [ref.debug_read("mask", i) for i in range(S)]
            ref.set_validity(**new[1])
            w2 = ref.process(d2, None, **new[0])
        assert r1.tobytes() == w1.tobytes() and r2.tobytes() == w2.tobytes()
        assert all(np.array_equal(a, b) for a, b in zip(m1, wm))
        for s in range(S):
            assert _state(bt, s) == _state(ref, s) and _captures(bt, s) == _captures(ref, s), s
        assert (r1["attempts"] == 2).any() and not (r2["attempts"] == 2).any()
    finally:
        bt.close()
        ref.close()


# ---- 8. wiring: HostPipeline in place, GraphedProcess, NV12 ----------------------------------------------------------

def test_wiring_host_pipeline_graph_nv12(torch_mod):
    """The same 3 rounds of 20 frames (profiles DEMO_1 / DEMO_2 / defaults by position) through HostPipeline(inplace),
    GraphedProcess and, as NV12 frames, process: each equals process(profiles=...) of the same RGB frames."""
    from lane_tracker_b200 import GraphedProcess, HostPipeline
    torch = torch_mod
    S, T = 20, 3
    profiles = {0: DEMO_1, 1: DEMO_2, 2: DEFAULTS}
    prof = [i % 3 for i in range(S)]
    seen = [0] * S
    rounds = [_batch(torch, _specs(list(range(S)), r, seen, 8500, {s for s in range(S) if (s + r) % 5 == 0}))
              for r in range(T)]
    handles = [_tracker(S) for _ in range(4)]
    for h in handles:
        _install(h, profiles)
    ref, hp_t, g_t, nv_t = handles
    try:
        want = []
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for d in rounds:
                o = torch.empty_like(d)
                want.append((ref.process(d, o, profiles=prof), o.cpu().numpy()))
            hp = HostPipeline(hp_t, depth=2, inplace=True)
            got = []
            for d in rounds:
                hp.submit(d.cpu().pin_memory(), profiles=prof)
                got += [(res.copy(), out.numpy().copy()) for out, res in hp.ready()]
            got += [(res.copy(), out.numpy().copy()) for out, res in hp.drain()]
            g = GraphedProcess(g_t, S, profiles=prof)
            _install(g_t, {0: DEMO_2})                 # captured table: the graph keeps DEMO_1 for profile 0
            gg = []
            for d in rounds:
                g.frames.copy_(d)
                g.replay()
                gg.append((g.fetch_results(), g.out.cpu().numpy()))
            nv = []
            for d in rounds:
                o = torch.empty_like(d)
                f = torch.as_tensor(synth.rgb_to_nv12(d.cpu().numpy())).cuda()
                nv.append((nv_t.process(f, o, profiles=prof), o))
        for r in range(T):
            assert got[r][0].tobytes() == want[r][0].tobytes() and np.array_equal(got[r][1], want[r][1]), r
            assert gg[r][0].tobytes() == want[r][0].tobytes() and np.array_equal(gg[r][1], want[r][1]), r
        # NV12: against the same handle configuration fed nv12_to_rgb of the frames
        chk = _tracker(S)
        _install(chk, profiles)
        try:
            for r, d in enumerate(rounds):
                f = torch.as_tensor(synth.rgb_to_nv12(d.cpu().numpy())).cuda()
                o = torch.empty_like(d)
                w = chk.process(chk.nv12_to_rgb(f), o, profiles=prof)
                assert nv[r][0].tobytes() == w.tobytes() and torch.equal(nv[r][1], o), r
        finally:
            chk.close()
    finally:
        for h in handles:
            h.close()


# ---- 9. refusals -----------------------------------------------------------------------------------------------------

def test_refusals(torch_mod):
    """Every refusal returns an error naming the position (C ABI) or raises (Python), and launches nothing."""
    from lane_tracker_b200 import DevicePipeline, _lib, make_params
    from lane_tracker_b200._lib import LaneTrackerError
    torch = torch_mod
    S = 8
    bt = _tracker(S)
    lib = bt.lib
    try:
        d = _batch(torch, [["synth", 9000 + s, 0] for s in range(4)])
        out = torch.empty_like(d)
        res = torch.zeros(S * 512, dtype=torch.uint8, device="cuda")
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        fp, op, rp = C.c_void_p(d.data_ptr()), C.c_void_p(out.data_ptr()), C.c_void_p(res.data_ptr())
        arr = lambda v: (C.c_int32 * len(v))(*v)
        p = make_params()
        # lt_set_profile
        assert lib.lt_set_profile(bt._h, -1, C.byref(p), None) < 0 and b"profile -1" in lib.lt_last_error()
        assert lib.lt_set_profile(bt._h, _lib.LT_MAX_PROFILES, C.byref(p), None) < 0
        assert lib.lt_set_profile(bt._h, 0, None, None) < 0
        bad = make_params(window_width=0)
        assert lib.lt_set_profile(bt._h, 0, C.byref(bad), None) < 0
        assert b"window_width must lie in [1, 64]" in lib.lt_last_error()
        with pytest.raises(LaneTrackerError, match="Unexpected filter mode|window_height"):
            bt.set_profile(0, window_height=10 ** 6)
        bt.set_profile(0)
        bt.set_profile(3, **presets.DEMO_2["process"])
        n0 = lib.lt_launch_count()
        cases = [
            (lambda: lib.lt_process_profiles(bt._h, fp, op, None, None, 4, rp, st), b"null profile list"),
            (lambda: lib.lt_process_profiles(bt._h, fp, op, None, arr([0, 0, 16, 0]), 4, rp, st), b"position 2"),
            (lambda: lib.lt_process_profiles(bt._h, fp, op, None, arr([0, -3, 0, 0]), 4, rp, st), b"position 1"),
            (lambda: lib.lt_process_profiles(bt._h, fp, op, None, arr([0, 0, 0, 1]), 4, rp, st), b"position 3 is unset"),
            (lambda: lib.lt_process_profiles(bt._h, fp, op, arr([0, 1, 1, 2]), arr([0] * 4), 4, rp, st), b"twice"),
            (lambda: lib.lt_process_front_profiles(bt._h, fp, arr([0, 5, 0, 0]), 4, 0, st), b"position 1 is unset"),
            (lambda: lib.lt_process_front_profiles(bt._h, fp, arr([0] * 4), 4, 2, st), b"buffer set"),
        ]
        for fn, msg in cases:
            assert fn() < 0
            assert msg in lib.lt_last_error(), (msg, lib.lt_last_error())
        assert lib.lt_launch_count() == n0
        # back half against the front half of its set
        assert lib.lt_process_front(bt._h, fp, 4, C.byref(p), 0, st) == 0
        n0 = lib.lt_launch_count()
        assert lib.lt_process_back_profiles(bt._h, fp, op, None, arr([0] * 4), 4, 0, rp, st) < 0
        assert b"without profiles" in lib.lt_last_error()
        assert lib.lt_launch_count() == n0
        assert lib.lt_process_front_profiles(bt._h, fp, arr([0, 3, 0, 3]), 4, 0, st) == 0
        n0 = lib.lt_launch_count()
        assert lib.lt_process_back_profiles(bt._h, fp, op, None, arr([0, 3, 0]), 3, 0, rp, st) < 0
        assert b"of 4 frames, not 3" in lib.lt_last_error()
        assert lib.lt_process_back_profiles(bt._h, fp, op, None, arr([0, 3, 3, 3]), 4, 0, rp, st) < 0
        assert b"position 2" in lib.lt_last_error()
        assert lib.lt_launch_count() == n0
        assert lib.lt_process_back_profiles(bt._h, fp, op, None, arr([0, 3, 0, 3]), 4, 0, rp, st) == 0
        # capture on: the widest bandwidth of the profiles used decides
        bt.set_capture(True)                  # default capacity: enough for bandwidth <= 32, not for 100
        bt.set_profile(4, bandwidth=100)
        n0 = lib.lt_launch_count()
        assert lib.lt_process_profiles(bt._h, fp, op, None, arr([0, 0, 4, 0]), 4, rp, st) < 0
        assert b"bandwidth 100" in lib.lt_last_error()
        assert lib.lt_launch_count() == n0
        bt.set_capture(False)
        # Python
        n0 = lib.lt_launch_count()
        with pytest.raises(ValueError, match="without params"):
            bt.process(d, out, params=p, profiles=[0] * 4)
        with pytest.raises(ValueError, match="without params"):
            bt.process(d, out, profiles=[0] * 4, ksize_r=11)
        with pytest.raises(ValueError, match="4 frames"):
            bt.process(d, out, profiles=[0] * 3)
        with pytest.raises(ValueError, match="position 1"):
            bt.process(d, out, profiles=[0, 16, 0, 0])
        with pytest.raises(ValueError, match="CUDA tensor"):
            bt.process(d, out, profiles=torch.zeros(4, dtype=torch.int32, device="cuda"))
        with pytest.raises(LaneTrackerError, match="position 3 is unset"):
            bt.process(d, out, profiles=np.array([0, 0, 0, 9]))
        with pytest.raises(ValueError, match="4 frames"):
            DevicePipeline(bt).submit(d, out, profiles=[0])
        assert lib.lt_launch_count() == n0
    finally:
        bt.close()
