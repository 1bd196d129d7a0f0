"""tests/_oracle_pool.py with a calibration per job: a job may carry "calibration" (the constructor arguments of
``LaneTracker`` as lists: img_size, warped_size, cam_matrix, dist_coeffs, warp_matrices, mpp_conversion) that both the
oracle tracker and the synthetic video of the job use, as a stream of another camera would.  Same job format
otherwise, same records.  Test infrastructure only.

    python tests/_oracle_pool_cameras.py jobs.json out.json
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)


def run_jobs(jobs, params=None, workers=None):
    """Called from a test: spawns this file as a script and returns its result (see _oracle_pool.run_jobs)."""
    import json
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        jp, op = os.path.join(tmp, "jobs.json"), os.path.join(tmp, "out.json")
        with open(jp, "w") as f:
            json.dump({"jobs": jobs, "params": params or {}, "workers": workers}, f)
        subprocess.run([sys.executable, os.path.abspath(__file__), jp, op], check=True)
        with open(op) as f:
            return json.load(f)


def calibration_from_json(c):
    import numpy as np
    return dict(img_size=tuple(c["img_size"]), warped_size=tuple(c["warped_size"]),
                cam_matrix=np.array(c["cam_matrix"], dtype=np.float64),
                dist_coeffs=np.array(c["dist_coeffs"], dtype=np.float64),
                warp_matrices=tuple(np.array(m, dtype=np.float64) for m in c["warp_matrices"]),
                mpp_conversion=tuple(c["mpp_conversion"]))


def _run_with_calibration(job):
    import _oracle_pool
    from lane_tracker_b200 import synth
    spec, _ = job
    if "calibration" in spec:
        cal = calibration_from_json(spec["calibration"])
        # the job's tracker and its RoadVideo both take the calibration from here (one job per call: a worker that
        # runs several jobs starts each from an empty video cache)
        synth.shipped_calibration = lambda scale=1.0: cal
    _oracle_pool._VIDEOS.clear()
    return _oracle_pool._run_orig(job)


def main():
    import _oracle_pool
    _oracle_pool._run_orig = _oracle_pool._run
    _oracle_pool._run = _run_with_calibration     # looked up by name when main() maps the jobs
    _oracle_pool.main()


if __name__ == "__main__":
    main()
