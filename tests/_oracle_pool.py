"""Run the CPU oracle over many streams in parallel, in a separate process tree (the calling test process has CUDA
initialised, so it must not fork).  Test infrastructure only.

    python tests/_oracle_pool.py jobs.json out.json

jobs.json: {"jobs": [{"kind": "synth", "seed": 3, "frames": 6} | {"kind": "image", "name": "test1.jpg", "frames": 6}
                     | {"kind": "plan", "plan": [<frame spec>, ...]}, ...],
            "params": {process() keyword overrides}}
           A job may also carry "scale" (calibration and synthetic video scale, default 1.0).  A plan lists one
           frame spec per frame (see frame_from_spec), so a stream can mix synthetic video, photographs, noise and
           blank frames.
out.json : per job, per frame: the fields a parity test compares (state, digests of the mask, the pixel sets and the
           output frame).
"""
import json
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)


_VIDEOS = {}


def frame_from_spec(spec, scale=1.0):
    """One RGB frame from a plan entry: ["synth", seed, t] (synth.RoadVideo), ["image", name] (bundled photograph,
    shipped scale only), ["noise", seed] (uniform random bytes), ["blank", value] (one grey level)."""
    import numpy as np
    import _fixtures as fx
    from lane_tracker_b200 import synth
    w, h = synth.shipped_calibration(scale)["img_size"]
    kind = spec[0]
    if kind == "synth":
        key = (int(spec[1]), float(scale))
        if key not in _VIDEOS:
            _VIDEOS[key] = synth.RoadVideo(key[0], scale=scale)
        return _VIDEOS[key].frame(int(spec[2]))
    if kind == "image":
        return fx.load_frame(spec[1])
    if kind == "noise":
        return np.random.default_rng(int(spec[1])).integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "blank":
        return np.full((h, w, 3), int(spec[1]), np.uint8)
    raise ValueError("unknown frame spec %r" % (spec,))


def _run(job):
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    warnings.simplefilter("ignore")
    import numpy as np
    import _fixtures as fx
    from lane_tracker_b200 import synth
    from oracle.tracker import OracleLaneTracker
    backend = "numpy"
    try:
        import cv2
        cv2.setNumThreads(1)
        backend = "cv2"
    except Exception:
        pass
    spec, params = job
    scale = float(spec.get("scale", 1.0))
    trk = OracleLaneTracker(**synth.shipped_calibration(scale), backend=backend)
    if spec["kind"] == "synth":
        plan = [["synth", spec["seed"], t] for t in range(spec["frames"])]
    elif spec["kind"] == "image":
        plan = [["image", spec["name"]]] * spec["frames"]
    else:
        plan = spec["plan"]
    out = []
    for item in plan:
        frame = frame_from_spec(item, scale).copy()
        o = trk.process(frame, **params)
        att = trk.trace["attempts"]
        last = att[-1]
        rec = dict(counter=trk.counter, success=trk.success, attempts=len(att), mode=last["mode"],
                   detected=bool(trk.detected_pixels), valid=bool(trk.valid_lane_lines),
                   last_detection=int(trk.last_detection), mask=fx.sha(last["mask"]), out=fx.sha(o),
                   first_detected=bool(att[0]["detected"]), first_valid=bool(att[0]["valid"]))
        if last["detected"]:
            rec.update(left_fit=[float(v) for v in last["left_fit"]], right_fit=[float(v) for v in last["right_fit"]],
                       n_left=int(len(last["left_x"])), n_right=int(len(last["right_x"])),
                       pix=fx.pix_digest(last["left_y"], last["left_x"], last["right_y"], last["right_x"]))
        if trk.valid_lane_lines:
            rec.update(radius=int(trk.average_curve_radius), ecc=float(trk.eccentricity),
                       left_avg=[float(v) for v in trk.left_avg_coeffs], right_avg=[float(v) for v in trk.right_avg_coeffs])
        out.append(rec)
    return out


def run_jobs(jobs, params=None, workers=None):
    """Called from a test: spawns this file as a script and returns its result."""
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
    import multiprocessing as mp
    with open(sys.argv[1]) as f:
        spec = json.load(f)
    jobs = [(j, spec["params"]) for j in spec["jobs"]]
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    workers = spec.get("workers") or cores
    with mp.get_context("fork").Pool(max(1, min(workers, len(jobs)))) as pool:
        res = pool.map(_run, jobs, chunksize=1)
    with open(sys.argv[2], "w") as f:
        json.dump(res, f)


if __name__ == "__main__":
    main()
