"""Oracle vs the original project's outputs, recorded in tests/golden/live_reference.json by
tests/golden/make_live_golden.py (the records compared are defined in tests/_live_records.py)."""
import warnings

import pytest

import _fixtures as fx
import _live_records as records
from lane_tracker_b200 import synth
from oracle.tracker import OracleLaneTracker

LIVE = fx.golden("live_reference.json")
CAL = synth.shipped_calibration()


def _same_records(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, i


def test_process_matches_live_reference_on_a_sequence():
    warnings.simplefilter("ignore")
    _same_records(records.sequence(OracleLaneTracker(**CAL, backend="cv2")), LIVE["sequence"])


def test_sliding_window_restatement_on_adversarial_masks():
    """The integer restatement of sliding_window_search equals the original on masks built to hit the quirks:
    windows leaving the frame (NumPy slice wrap-around), one-sided masks, coupling fallback, limits 8 and 50."""
    want = LIVE["sliding_window"]
    assert sum(w["detected"] for w in want) > 20
    _same_records(records.sliding_window(OracleLaneTracker(**CAL)), want)


@pytest.mark.parametrize("backend", ["cv2", "numpy"])
def test_debug_views_match_live_reference(backend):
    """visualize_search / split_view (lane_tracker.py:689-793, 1130-1209, utils.py:57-103): sliding-window frame,
    band-search frames, a frame that fails both attempts (still pixels -> SWS view of attempt 2) and a recovery."""
    warnings.simplefilter("ignore")
    got = records.debug_views(lambda: OracleLaneTracker(**CAL, backend=backend))
    assert all(w["shape"] == [720 + 652, 1280, 3] for w in LIVE["debug_views"]["split_view"])
    for mode in records.DEBUG_VIEW_MODES:
        _same_records(got[mode], LIVE["debug_views"][mode])
