"""What tests/test_oracle_live.py compares between the oracle and the original project, as JSON-able records.

Each function runs one comparison's inputs through a tracker (the original's ``LaneTracker`` or the oracle: same
attributes, same methods) and returns what the comparison looks at.  tests/golden/make_live_golden.py stores the
original's records in tests/golden/live_reference.json; the tests compute the oracle's and require equality.
Integer arrays are kept as digests of their int64 values, floats exactly.
"""
import numpy as np

import _fixtures as fx
import _masks
from lane_tracker_b200 import synth

SEQUENCE_ARRAYS = ("left_x", "left_y", "right_x", "right_y", "left_avg_x", "right_avg_x")
SWS_PARAMS = ((8, 1.0, 0.1), (50, 1.0, 0.1), (8, 0.5, 0.35))        # (no_success_limit, partial, mu)
DEBUG_VIEW_MODES = ("visualize_search", "split_view")


def _int_digest(v):
    if v is None:
        return None
    a = np.asarray(v)
    b = a.astype(np.int64)
    assert np.array_equal(a, b), "non-integer values"
    return fx.sha(b)


def sequence_frames():
    """Synthetic stream 3 with a two-frame outage on a bundled photograph (sliding window, tracking, failure, recovery)."""
    vid = synth.RoadVideo(3)
    return [vid.frame(t) for t in range(4)] + [fx.load_frame("test4.jpg")] * 2 + [vid.frame(6)]


def sequence(trk):
    """process() frame by frame on one tracker: overlay (text box blanked), state and the lane pixel sets."""
    out = []
    for f in sequence_frames():
        frame = fx.sha(f)
        img = trk.process(f.copy())
        rec = dict(frame=frame, out=fx.out_digest(img), last_detection=int(trk.last_detection),
                   valid=bool(trk.valid_lane_lines),
                   radius=None if trk.average_curve_radius is None else int(trk.average_curve_radius),
                   ecc=None if trk.eccentricity is None else float(trk.eccentricity))
        rec.update((nm, _int_digest(getattr(trk, nm))) for nm in SEQUENCE_ARRAYS)
        out.append(rec)
    return out


def sliding_window(trk):
    """sliding_window_search on masks built to hit its quirks: windows leaving the frame (NumPy slice wrap-around),
    one-sided masks, coupling fallback, no-success limits 8 and 50."""
    out = []
    for m in _masks.random_masks(36, seed=5):
        for nsl, partial, mu in SWS_PARAMS:
            trk.detected_pixels = False
            trk.sliding_window_search(m, 30, 40, 20, mu, nsl, 0.25, 360, 30, partial)
            rec = dict(detected=bool(trk.detected_pixels))
            if trk.detected_pixels:
                rec.update(pix=fx.pix_digest(trk.left_y, trk.left_x, trk.right_y, trk.right_x),
                           left_centroids=[int(v) for v in trk.left_window_centroids],
                           right_centroids=[int(v) for v in trk.right_window_centroids])
            out.append(rec)
    return out


def debug_view_frames():
    """Sliding-window frame, band-search frames, a frame that fails both attempts (still pixels: the sliding-window
    view of attempt 2) and a recovery."""
    vid = synth.RoadVideo(5)
    return [vid.frame(t) for t in range(3)] + [fx.load_frame("test4.jpg")] + [vid.frame(4)]


def debug_views(make_tracker):
    """process(visualize_search=True) and process(split_view=True), each on a fresh tracker."""
    out = {}
    for mode in DEBUG_VIEW_MODES:
        trk = make_tracker()
        recs = []
        for f in debug_view_frames():
            r = trk.process(f.copy(), **{mode: True})
            if mode == "visualize_search":
                recs.append(dict(out=fx.sha(r[0]), vis=fx.sha(r[1]), vis_shape=list(r[1].shape)))
            else:
                recs.append(dict(canvas=fx.sha(r), shape=list(r.shape)))
        out[mode] = recs
    return out
