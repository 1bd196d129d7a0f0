"""tests/_oracle_pool.py with settings per frame: a plan entry may end with a dict {"params": {process() keyword
overrides}, "validity": {lt_validity names: min_dist_y1 ... tangent_thresh}} that applies to that frame only (the
job's "params" and the shipped windows otherwise), as parameter profiles give each frame of a batch its own settings.
Same job format otherwise, same records.  Test infrastructure only.

    python tests/_oracle_pool_profiles.py jobs.json out.json
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

# lt_validity field -> the oracle's key (oracle/tracker.py VALIDITY)
VALIDITY_KEYS = dict(min_dist_y1="min_d1", max_dist_y1="max_d1", min_dist_y2="min_d2", max_dist_y2="max_d2",
                     min_dist_y3="min_d3", max_dist_y3="max_d3", tangent_thresh="tan")


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

    pending = [{}]
    frame_from_spec = _oracle_pool.frame_from_spec

    def frame_with_settings(spec, scale=1.0):
        pending[0] = spec[-1] if isinstance(spec[-1], dict) else {}
        return frame_from_spec(spec, scale)

    class ProfiledOracleLaneTracker(ot.OracleLaneTracker):
        def process(self, img, **kw):
            extra = pending[0]
            self.validity = dict(ot.VALIDITY)
            for k, v in extra.get("validity", {}).items():
                self.validity[VALIDITY_KEYS[k]] = v
            return super().process(img, **dict(kw, **extra.get("params", {})))

    # _oracle_pool's workers look both up by name when they run a job (forked after this point)
    _oracle_pool.frame_from_spec = frame_with_settings
    ot.OracleLaneTracker = ProfiledOracleLaneTracker
    _oracle_pool.main()


if __name__ == "__main__":
    main()
