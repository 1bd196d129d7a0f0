"""tests/_oracle_pool.py with the tracker's frame counter drawn: every job runs an OracleLaneTracker created with
print_frame_count=True, so the "Frame: n" text shows in the oracle's output frames.  Same job format, same records.
Test infrastructure only.

    python tests/_oracle_pool_counted.py jobs.json out.json
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)


def run_jobs(jobs, params=None, workers=None):
    """Called from a test: spawns this file as a script and returns its result (see _oracle_pool.run_jobs)."""
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        jp, op = os.path.join(tmp, "jobs.json"), os.path.join(tmp, "out.json")
        with open(jp, "w") as f:
            json.dump({"jobs": jobs, "params": params or {}, "workers": workers}, f)
        subprocess.run([sys.executable, os.path.abspath(__file__), jp, op], check=True)
        with open(op) as f:
            return json.load(f)


def main():
    import _oracle_pool
    import oracle.tracker as ot

    class CountedOracleLaneTracker(ot.OracleLaneTracker):
        def __init__(self, *args, **kw):
            kw["print_frame_count"] = True
            super().__init__(*args, **kw)

    # _oracle_pool's workers look the class up in oracle.tracker when they build a tracker (forked after this point)
    ot.OracleLaneTracker = CountedOracleLaneTracker
    _oracle_pool.main()


if __name__ == "__main__":
    main()
