"""Cameras: every frame of a batch from its own calibration (``set_camera`` and ``cameras=`` of
``BatchedLaneTracker.process`` and the pipelines; C ABI: lt_set_camera, lt_process_cameras, lt_process_front_cameras,
lt_process_back_cameras).

The GPU reference is one handle per camera, created by lt_create with that camera's calibration and driven, per
camera, with the frames of that camera and the same stream ids.  A stream that changes camera has its state moved to
the reference handle of its new camera first (get_state / set_state).  Compared bit for bit: result records, final
masks per position, annotated frames, state, averaged polylines and cached lane rows per stream id.  Two streams of
non-shipped cameras are also anchored to the CPU oracle (tests/_oracle_pool_cameras.py).

Test cameras, all 1280x720 / 1080x1100, each with its own metres per pixel, and synthetic road video rendered
through each camera's own M:
  B  M composed with a bird's-eye shift and a small rotation (another mounting)
  C  a homography that looks further ahead: its ROI is taller than camera 0's
  D  another cam_matrix and k1 (fx x 0.95, cx + 10, k1 = -0.2)
  E  k1 = +0.2: taps fall outside the frame
"""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

import _oracle_pool_cameras
from lane_tracker_b200 import presets, synth
from lane_tracker_b200.tracker import RESULT_DTYPE

pytestmark = pytest.mark.gpu

FIT_RTOL = 1e-6


def _shift_rot(dx, dy, deg):
    """Bird's-eye transform: rotation by `deg` about the bird's-eye centre, then a shift."""
    bw, bh = synth.WARPED_SIZE
    a = np.deg2rad(deg)
    c, s = np.cos(a), np.sin(a)
    T0 = np.array([[1, 0, -bw / 2], [0, 1, -bh / 2], [0, 0, 1.0]])
    R = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])
    T1 = np.array([[1, 0, bw / 2 + dx], [0, 1, bh / 2 + dy], [0, 0, 1.0]])
    return T1 @ R @ T0


def _mounted(T, mpp=(1.0, 1.0), K=None, k1=None):
    cal = synth.shipped_calibration()
    M = T @ cal["warp_matrices"][0]
    cal["warp_matrices"] = (M, np.linalg.inv(M))
    cal["mpp_conversion"] = (synth.MPPV * mpp[0], synth.MPPH * mpp[1])
    if K is not None:
        cal["cam_matrix"] = K
    if k1 is not None:
        cal["dist_coeffs"] = cal["dist_coeffs"].copy()
        cal["dist_coeffs"][0, 0] = k1
    return cal


def _far():
    """Bird's-eye rows scaled by 0.8 about the bottom row: the view reaches further ahead."""
    bh = synth.WARPED_SIZE[1]
    return np.array([[1, 0, 0], [0, 0.8, 0.2 * (bh - 1)], [0, 0, 1.0]])


def _lens_d():
    K = synth.CAM_MATRIX.copy()
    K[0, 0] *= 0.95
    K[0, 2] += 10.0
    return K


CAMERAS = {
    1: _mounted(_shift_rot(12.0, -20.0, 1.5), mpp=(1.1, 0.95)),                 # B
    2: _mounted(_far(), mpp=(1.25, 1.0)),                                      # C
    3: _mounted(np.eye(3), mpp=(0.9, 1.05), K=_lens_d(), k1=-0.2),            # D
    4: _mounted(np.eye(3), mpp=(1.0, 0.9), k1=0.2),                            # E
}


def _cal(k):
    return synth.shipped_calibration() if k == 0 else CAMERAS[k]


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module", autouse=True)
def _no_pinned_bands():
    os.environ.pop("LT_MORPH_BANDS", None)


_VIDEOS = {}


def _frame(cam, seed, t):
    """Frame t of the road video of `seed` through camera `cam`; every seventh frame of a stream is noise."""
    if (seed + t) % 7 == 6:
        return np.random.default_rng(5000 + 37 * seed + t).integers(0, 256, (720, 1280, 3), dtype=np.uint8)
    key = (cam, seed)
    if key not in _VIDEOS:
        _VIDEOS[key] = synth.RoadVideo(seed, calibration=_cal(cam) if cam else None)
    return _VIDEOS[key].frame(t)


def _tracker(S, cameras=CAMERAS, **kw):
    from lane_tracker_b200 import BatchedLaneTracker
    bt = BatchedLaneTracker(S, **synth.shipped_calibration(), **kw)
    for k, cal in cameras.items():
        bt.set_camera(k, cal["cam_matrix"], cal["dist_coeffs"], cal["warp_matrices"], cal["mpp_conversion"])
    return bt


def _state(bt, s):
    st, lx, rx = bt.get_state(s)
    return [bytes(st), lx.tobytes(), rx.tobytes(), bt.debug_read("lane_rows", s).tobytes()]


class Reference:
    """One handle per camera; per camera (and profile), process(ids=...) over the frames of that camera."""

    def __init__(self, S, cams, **kw):
        from lane_tracker_b200 import BatchedLaneTracker
        self.bt = {k: BatchedLaneTracker(S, **_cal(k), **kw) for k in cams}
        self.owner = {}

    def step(self, torch, d, ids, cams, profiles=None, overlay=True):
        """-> (records, out frames or None, masks per position) in batch order.  profiles: per position a (process()
        keywords, validity or None) pair, or None for the defaults."""
        n = len(ids)
        recs = np.zeros(n, dtype=RESULT_DTYPE)
        out = torch.empty((n, 720, 1280, 3), dtype=torch.uint8, device=d.device) if overlay else None
        masks = [None] * n
        keys = [(int(cams[i]), 0 if profiles is None else repr(profiles[i])) for i in range(n)]
        for key in sorted(set(keys)):
            pos = [i for i in range(n) if keys[i] == key]
            bt = self.bt[key[0]]
            for p in pos:
                s = int(ids[p])
                src = self.owner.get(s, key[0])
                if src != key[0]:                          # the stream's state carries over to its new camera
                    st, lx, rx = self.bt[src].get_state(s)
                    bt.set_state(s, st, lx, rx)
                self.owner[s] = key[0]
            kw, val = ({}, None) if profiles is None else profiles[pos[0]]
            if val is None:
                bt.set_validity()
            else:
                bt.set_validity(**val)
            idx = torch.as_tensor(pos).cuda()
            sub = d[idx].contiguous()
            so = torch.empty((len(pos), 720, 1280, 3), dtype=torch.uint8, device=d.device) if overlay else None
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                recs[pos] = bt.process(sub, so, ids=[int(ids[p]) for p in pos], **kw)
            if overlay:
                out[idx] = so
            for j, p in enumerate(pos):
                masks[p] = bt.debug_read("mask", j)
        return recs, out, masks

    def state(self, s):
        return _state(self.bt[self.owner.get(s, 0)], s)

    def close(self):
        for bt in self.bt.values():
            bt.close()


def _batch(torch, ids, cams, seen, nv12=False):
    fr = []
    for s, k in zip(ids, cams):
        fr.append(_frame(int(k), int(s), seen[int(s)]))
        seen[int(s)] += 1
    a = np.stack(fr)
    return torch.as_tensor(synth.rgb_to_nv12(a) if nv12 else a).cuda()


def _compare(bt, ref, step, res, out, ids, tag):
    recs, rout, rmasks = step
    assert res.tobytes() == recs.tobytes(), tag
    if out is not None:
        assert np.array_equal(out.cpu().numpy(), rout.cpu().numpy()), tag
    for i in range(len(ids)):
        assert np.array_equal(bt.debug_read("mask", i), rmasks[i]), (tag, i)


def _compare_states(bt, ref, ids, tag):
    for s in ids:
        assert _state(bt, int(s)) == ref.state(int(s)), (tag, int(s))


def _run_rounds(torch, S, plan, nv12=False, profiles=None, cameras=CAMERAS):
    """plan: [(ids, cams)] per round through process(cameras=...) against the reference."""
    bt = _tracker(S, cameras)
    ref = Reference(S, sorted(set(int(k) for _, cs in plan for k in cs) | {0}))
    seen = [0] * S
    try:
        for r, (ids, cams) in enumerate(plan):
            d = _batch(torch, ids, cams, seen, nv12)
            out = torch.empty((len(ids), 720, 1280, 3), dtype=torch.uint8, device=d.device)
            prof = None if profiles is None else profiles(r, len(ids))
            if prof is None:
                res = bt.process(d, out, ids=ids, cameras=cams)
            else:
                table = {repr(p): i for i, p in enumerate(dict((repr(p), p) for p in prof).values())}
                for p in prof:
                    bt.set_profile(table[repr(p)], validity=p[1], **p[0])
                res = bt.process(d, out, ids=ids, cameras=cams, profiles=[table[repr(p)] for p in prof])
            step = ref.step(torch, d, ids, cams, prof)
            _compare(bt, ref, step, res, out, ids, r)
            _compare_states(bt, ref, ids, r)
    finally:
        bt.close()
        ref.close()


# ---- camera 0 only: the launches of lt_process ----------------------------------------------------------------------

def test_camera0_equals_process(torch_mod):
    """All positions on camera 0 through the camera call equal process() bit for bit, with the same launch count."""
    torch = torch_mod
    S = 16
    a, b = _tracker(S, {}), _tracker(S)
    seen = [0] * S
    try:
        for r in range(3):
            d = _batch(torch, list(range(S)), [0] * S, seen)
            oa, ob = torch.empty_like(d), torch.empty_like(d)
            c0 = a.lib.lt_launch_count()
            ra = a.process(d, oa)
            c1 = a.lib.lt_launch_count()
            rb = b.process(d, ob, cameras=[0] * S)
            assert b.lib.lt_launch_count() - c1 == c1 - c0, r
            assert ra.tobytes() == rb.tobytes(), r
            assert np.array_equal(oa.cpu().numpy(), ob.cpu().numpy()), r
            for i in range(S):
                assert np.array_equal(a.debug_read("mask", i), b.debug_read("mask", i)), (r, i)
                assert _state(a, i) == _state(b, i), (r, i)
    finally:
        a.close()
        b.close()


# ---- mixed batches ----------------------------------------------------------------------------------------------------

def test_interleaved_17_streams_3_cameras(torch_mod):
    """17 streams over cameras 0, B and C, interleaved, with runs that are not multiples of 4, in scattered order."""
    rng = np.random.default_rng(3)
    plan = []
    for r in range(4):
        ids = [int(v) for v in rng.permutation(17)]
        cams = [(0, 1, 2, 1, 2)[(s + r) % 5] for s in ids]
        plan.append((ids, cams))
    _run_rounds(torch_mod, 17, plan)


def test_interleaved_nv12(torch_mod):
    """NV12 frames from cameras 0, B, D and E."""
    plan = [(list(range(11)), [(0, 1, 3, 4)[s % 4] for s in range(11)]) for _ in range(3)]
    _run_rounds(torch_mod, 11, plan, nv12=True)


def test_taller_roi_then_shorter_on_same_slots(torch_mod):
    """A batch of camera C (taller ROI) leaves its rows in the camera buffer; a camera-B batch on the same slots must
    read zeros below its own ROI."""
    ids = list(range(8))
    plan = [(ids, [2] * 8), (ids, [1] * 8), (ids, [2] * 4 + [1] * 4), (ids, [1] * 8)]
    _run_rounds(torch_mod, 8, plan)


def test_33_streams_33_cameras(torch_mod):
    """33 streams on 33 distinct cameras: one stream per run, three pad slots per camera."""
    cams = {k: _mounted(_shift_rot(1.5 * k - 24.0, 0.7 * k, 0.05 * k - 0.8), mpp=(1.0 + 0.01 * k, 1.0 - 0.005 * k))
            for k in range(1, 33)}
    saved = dict(CAMERAS)
    CAMERAS.update(cams)
    try:
        plan = [(list(range(33)), list(range(33))) for _ in range(3)]
        _run_rounds(torch_mod, 33, plan, cameras=cams)
    finally:
        CAMERAS.clear()
        CAMERAS.update(saved)


def test_cameras_with_profiles_and_scattered_ids(torch_mod):
    """Profiles that change the filter group (DEMO_1 / DEMO_2), scattered ids and four cameras: the camera slot order
    against the filter position lists."""
    d1 = (presets.DEMO_1["process"], presets.DEMO_1["validity"])
    d2 = (presets.DEMO_2["process"], presets.DEMO_2["validity"])
    rng = np.random.default_rng(11)
    plan = []
    for r in range(3):
        ids = [int(v) for v in rng.permutation(20)[:14]]
        plan.append((ids, [(0, 1, 2, 3)[(s * 3 + r) % 4] for s in ids]))
    _run_rounds(torch_mod, 20, plan, profiles=lambda r, n: [(d1, d2)[(i + r) % 2] for i in range(n)])


def test_stream_changes_camera_every_frame(torch_mod):
    """Stream 0 changes camera every frame; its tracking state carries over."""
    plan = [([0, 1, 2], [(0, 1, 2, 3, 4)[r % 5], 1, 2]) for r in range(6)]
    _run_rounds(torch_mod, 3, plan)


def test_radii_follow_the_camera_mpp(torch_mod):
    """Two cameras that differ from camera 0 only in mppv / mpph: same masks and fits, radii and eccentricity of
    their own (k_update_state reads the position's camera)."""
    base = synth.shipped_calibration()
    cams = {1: dict(base, mpp_conversion=(synth.MPPV * 1.3, synth.MPPH)),
            2: dict(base, mpp_conversion=(synth.MPPV, synth.MPPH * 0.7))}
    saved = dict(CAMERAS)
    CAMERAS.update(cams)
    try:
        plan = [([0, 1, 2], [0, 1, 2])] * 4
        _run_rounds(torch_mod, 3, plan, cameras=cams)
    finally:
        CAMERAS.clear()
        CAMERAS.update(saved)


# ---- pipelines --------------------------------------------------------------------------------------------------------

def test_device_pipeline(torch_mod):
    """DevicePipeline with cameras over six batches equals the reference; results and states."""
    torch = torch_mod
    from lane_tracker_b200 import DevicePipeline
    S = 12
    bt = _tracker(S)
    ref = Reference(S, [0, 1, 2, 3, 4])
    seen, seen_ref = [0] * S, [0] * S
    try:
        pipe = DevicePipeline(bt)
        outs, batches, results = [], [], []
        for r in range(6):
            ids = [int(v) for v in np.random.default_rng(r).permutation(S)[:10]]
            cams = [(s + r) % 5 for s in ids]
            d = _batch(torch, ids, cams, seen)
            out = torch.empty((10, 720, 1280, 3), dtype=torch.uint8, device=d.device)
            pipe.submit(d, out, ids=ids, cameras=cams)
            results.append(pipe.fetch_results(10))
            outs.append(out)
            batches.append((d, ids, cams))
        for r, (d, ids, cams) in enumerate(batches):
            step = ref.step(torch, d, ids, cams)
            assert results[r].tobytes() == step[0].tobytes(), r
            assert np.array_equal(outs[r].cpu().numpy(), step[1].cpu().numpy()), r
        _compare_states(bt, ref, range(S), "end")
    finally:
        bt.close()
        ref.close()


@pytest.mark.parametrize("inplace", [False, True])
def test_host_pipeline_camera_c(torch_mod, inplace):
    """HostPipeline fits-only (NV12: only the rows the tracker reads go up) and inplace=True (RGB) with camera C,
    whose source rows reach beyond camera 0's: the row transfers cover the union of the cameras set."""
    torch = torch_mod
    from lane_tracker_b200 import HostPipeline
    S = 6
    bt = _tracker(S, {2: CAMERAS[2]})
    ref = Reference(S, [0, 2])
    src0, src2 = bt.camera_rows[0]["source_rows"], bt.camera_rows[2]["source_rows"]
    assert src2[0] < src0[0], (src0, src2)
    seen = [0] * S
    try:
        pipe = HostPipeline(bt, depth=2, overlay=inplace, inplace=inplace, frame_format="rgb" if inplace else "nv12")
        assert pipe.rows_in[0] <= src2[0]
        got, sent = [], []
        for r in range(4):
            ids = list(range(S))
            cams = [2 if (s + r) % 3 else 0 for s in ids]
            host = _batch(torch, ids, cams, seen, nv12=not inplace).cpu().pin_memory()
            sent.append((host.clone(), ids, cams))
            pipe.submit(host, ids=ids, cameras=cams)
            for o, res in pipe.ready():
                got.append((None if o is None else o.clone(), res.copy()))
        for o, res in pipe.drain():
            got.append((None if o is None else o.clone(), res.copy()))
        for r, ((host, ids, cams), (o, res)) in enumerate(zip(sent, got)):
            step = ref.step(torch, host.cuda(), ids, cams, overlay=inplace)
            assert res.tobytes() == step[0].tobytes(), r
            if inplace:
                assert np.array_equal(o.numpy(), step[1].cpu().numpy()), r
    finally:
        bt.close()
        ref.close()


def test_graphed_process_and_stale_graph(torch_mod):
    """GraphedProcess with cameras replays like process(cameras=...); after a set_camera it refuses to replay."""
    torch = torch_mod
    from lane_tracker_b200 import GraphedProcess
    S = 5
    bt = _tracker(S, {1: CAMERAS[1], 3: CAMERAS[3]})
    ref = Reference(S, [0, 1, 3])
    seen = [0] * S
    cams = [1, 0, 3, 1, 3]
    try:
        g = GraphedProcess(bt, S, cameras=cams)
        for r in range(3):
            d = _batch(torch, list(range(S)), cams, seen)
            g.frames.copy_(d)
            g.replay()
            res = g.fetch_results()
            step = ref.step(torch, d, list(range(S)), cams)
            assert res.tobytes() == step[0].tobytes(), r
            assert np.array_equal(g.out.cpu().numpy(), step[1].cpu().numpy()), r
        c = CAMERAS[2]                                    # a taller ROI: the camera buffer is reallocated
        bt.set_camera(2, c["cam_matrix"], c["dist_coeffs"], c["warp_matrices"], c["mpp_conversion"])
        with pytest.raises(RuntimeError, match="set_camera ran after this graph was captured"):
            g.replay()
    finally:
        bt.close()
        ref.close()


# ---- the CPU oracle ---------------------------------------------------------------------------------------------------

def _json_cal(c):
    return dict(img_size=list(c["img_size"]), warped_size=list(c["warped_size"]),
                cam_matrix=np.asarray(c["cam_matrix"]).tolist(), dist_coeffs=np.asarray(c["dist_coeffs"]).tolist(),
                warp_matrices=[np.asarray(m).tolist() for m in c["warp_matrices"]],
                mpp_conversion=list(c["mpp_conversion"]))


def test_oracle_anchor_cameras_b_and_d(torch_mod):
    """Two streams of cameras B and D against the oracle run with their calibrations."""
    torch = torch_mod
    S, T = 2, 5
    bt = _tracker(S, {1: CAMERAS[1], 3: CAMERAS[3]})
    cams = [1, 3]
    vids = [synth.RoadVideo(20 + s, calibration=CAMERAS[k]) for s, k in enumerate(cams)]
    got = []
    try:
        for t in range(T):
            d = torch.as_tensor(np.stack([v.frame(t) for v in vids])).cuda()
            got.append(bt.process(d, cameras=cams))
    finally:
        bt.close()
    want = _oracle_pool_cameras.run_jobs([dict(kind="synth", seed=20 + s, frames=T, calibration=_json_cal(CAMERAS[k]))
                                          for s, k in enumerate(cams)])
    for s in range(S):
        for t in range(T):
            res, w = got[t][s], want[s][t]
            tag = (s, t)
            assert int(res["counter"]) == w["counter"] and int(res["success"]) == w["success"], tag
            assert bool(res["detected_pixels"]) == w["detected"] and bool(res["valid_lane_lines"]) == w["valid"], tag
            assert int(res["last_detection"]) == w["last_detection"], tag
            if w["detected"]:
                assert int(res["n_left"]) == w["n_left"] and int(res["n_right"]) == w["n_right"], tag
                np.testing.assert_allclose(res["left_fit"], w["left_fit"], rtol=FIT_RTOL, err_msg=str(tag))
                np.testing.assert_allclose(res["right_fit"], w["right_fit"], rtol=FIT_RTOL, err_msg=str(tag))
            if w["valid"]:
                assert int(res["average_curve_radius"]) == w["radius"], tag
                assert float(res["eccentricity"]) == pytest.approx(w["ecc"], rel=1e-9, abs=1e-12), tag
    assert any(w["valid"] for job in want for w in job), "no valid frame: the anchor would test nothing"


# ---- refusals ---------------------------------------------------------------------------------------------------------

def _c_error(bt):
    return bt.lib.lt_last_error().decode()


def test_refusals(torch_mod):
    torch = torch_mod
    from lane_tracker_b200._lib import LaneTrackerError, lt_camera
    S = 4
    bt = _tracker(S, {1: CAMERAS[1]})
    c = CAMERAS[2]
    args = (c["cam_matrix"], c["dist_coeffs"], c["warp_matrices"], c["mpp_conversion"])
    try:
        with pytest.raises(LaneTrackerError, match="camera 0 is the calibration given to lt_create"):
            bt.set_camera(0, *args)
        with pytest.raises(LaneTrackerError, match=r"camera 64 outside \[1, 64\)"):
            bt.set_camera(64, *args)
        assert bt.lib.lt_set_camera(bt._h, 5, None) < 0 and "null camera" in _c_error(bt)
        with pytest.raises(ValueError, match="extra|5-coefficient"):
            bt.set_camera(5, c["cam_matrix"], np.array([0.1, 0, 0, 0, 0, 0.3]), c["warp_matrices"], c["mpp_conversion"])
        d = _batch(torch, [0, 1], [0, 1], [0] * S)
        with pytest.raises(ValueError, match="camera 5 at batch position 1 is unset"):
            bt.process(d, cameras=[0, 5])
        # the C checks name the position as well
        cams = (C.c_int32 * 2)(0, 7)
        from lane_tracker_b200.tracker import make_params, _ptr
        p = make_params()
        res = torch.zeros(2 * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=d.device)
        rc = bt.lib.lt_process_cameras(bt._h, _ptr(d), None, None, cams, 2, C.byref(p), None, _ptr(res), None)
        assert rc < 0 and "camera 7 at batch position 1 is unset" in _c_error(bt)
        cams = (C.c_int32 * 2)(0, 64)
        rc = bt.lib.lt_process_cameras(bt._h, _ptr(d), None, None, cams, 2, C.byref(p), None, _ptr(res), None)
        assert rc < 0 and "camera 64 at batch position 1 outside [0, 64)" in _c_error(bt)
        rc = bt.lib.lt_process_cameras(bt._h, _ptr(d), None, None, None, 2, C.byref(p), None, _ptr(res), None)
        assert rc < 0 and "null camera list" in _c_error(bt)
        # remap mode 1
        bt.set_remap_mode("fused")
        with pytest.raises(LaneTrackerError, match="remap mode 1"):
            bt.process(d, cameras=[0, 1])
        bt.set_remap_mode("exact")
        # a back half that does not match its front half
        bt.process_front_async(d, 0, cameras=[0, 1])
        with pytest.raises(LaneTrackerError, match="camera 0 at batch position 1 differs from the front half's camera 1"):
            bt.process_back_async(d, None, 0, cameras=[0, 0])
        # set_camera while that front half waits for its back half
        with pytest.raises(LaneTrackerError, match="buffer set 0 holds the front half of a camera batch"):
            bt.set_camera(2, *args)
        bt.process_back_async(d, None, 0, cameras=[0, 1])
        bt.set_camera(2, *args)
        bt.process_front_async(d, 1)
        with pytest.raises(LaneTrackerError, match="buffer set 1 was last filled by a front half without cameras"):
            bt.process_back_async(d, None, 1, cameras=[0, 1])
        torch.cuda.synchronize()
        assert isinstance(lt_camera(), C.Structure)
    finally:
        bt.close()
