#!/usr/bin/env python3
"""Generate tests/golden/live_reference.json: the original project's outputs that tests/test_oracle_live.py compares
the oracle with (the records are defined in tests/_live_records.py).

Run:  python tests/golden/make_live_golden.py --reference DIR    # DIR: checkout of pierluigiferrari/lane_tracker
      python tests/golden/make_live_golden.py                    # the oracle (cv2 operators) stands in for it

With --reference the original is imported as tests/_liveref.py does it (SURVEY.md Appendix C patches).  The original
is not part of this repository, and the committed file was made without it: from the oracle, which these same
comparisons, run against the original itself, had held equal to it on exactly these inputs.  ``meta.source`` says
which of the two produced the file.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _live_records as records  # noqa: E402
from lane_tracker_b200 import synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", help="directory holding the original's lane_tracker.py, utils.py and pickles")
    args = ap.parse_args()
    warnings.simplefilter("ignore")
    import cv2
    if args.reference:
        import _liveref
        _liveref.REFERENCE_DIR = args.reference
        make_tracker, source = _liveref.make_tracker, "original (pierluigiferrari/lane_tracker)"
    else:
        from oracle.tracker import OracleLaneTracker
        make_tracker = lambda: OracleLaneTracker(**synth.shipped_calibration(), backend="cv2")  # noqa: E731
        source = "oracle (cv2 operators) standing in for the original"
    with contextlib.redirect_stdout(io.StringIO()):         # the original prints from process()
        gold = dict(meta=dict(source=source, cv2=cv2.__version__, generator="tests/golden/make_live_golden.py"),
                    sequence=records.sequence(make_tracker()),
                    sliding_window=records.sliding_window(make_tracker()),
                    debug_views=records.debug_views(make_tracker))
    with open(os.path.join(HERE, "live_reference.json"), "w") as f:
        json.dump(gold, f, indent=1)
    print("wrote live_reference.json from the", source)


if __name__ == "__main__":
    main()
