"""DevicePipeline frames/s of batches whose frames come from different cameras, at the bench's default geometry.

    python tools/cameras_bench.py [--batches 48] [--warmup 8] [--repeats 3] [--stage-calls 16] [--out FILE]

64 streams of 1280x720 road video (four pre-rendered frames per stream, device-resident; one batch is 177 MB of
input, more than the 126 MB L2), timed with CUDA events around `--batches` submissions through DevicePipeline:
  plain        submit(frames, out)
  camera0      submit(frames, out, cameras=[0] * 64): the launches of plain
  one_camera   all 64 frames on camera 1: the camera undistort buffer and its slot indirection
  runs4        cameras 1..4 in runs of 16 positions
  interleaved4 cameras 1..4, position i -> 1 + i % 4 (sorted into runs inside the library: should match runs4)
  cameras64    64 cameras, one stream each: three pad slots per camera, and the four threads of a warp column gather
               from four cameras
Cameras 1..63 carry the shipped calibration with their own metres per pixel, so that every variant does the same
tracking work on the same frames and the differences are what the camera path costs.  The variants alternate within
each repeat (rotated order) and the tracker is reset before each one; the output reports the median and spread (min,
max) over repeats.  Per-stage times come from lt_profile_* over `--stage-calls` sequential process() calls per
variant, in a separate pass (event recording adds host work).  The card's name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

S, P = 64, 4


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


VARIANTS = {
    "plain": None,
    "camera0": [0] * S,
    "one_camera": [1] * S,
    "runs4": [1 + i // 16 for i in range(S)],
    "interleaved4": [1 + i % 4 for i in range(S)],
    "cameras64": list(range(S)),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--stage-calls", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("cameras_bench needs a CUDA device")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, synth
    pool = torch.from_numpy(np.ascontiguousarray(synth.render_streams(S, P).transpose(1, 0, 2, 3, 4))).cuda()  # [P, S, ...]
    outs = [torch.empty_like(pool[0]) for _ in range(2)]
    cal = synth.shipped_calibration()
    trk = BatchedLaneTracker(S, **cal)
    mem0 = torch.cuda.mem_get_info()[0]
    for k in range(1, S):
        trk.set_camera(k, cal["cam_matrix"], cal["dist_coeffs"], cal["warp_matrices"],
                       (synth.MPPV * (1.0 + 0.01 * k), synth.MPPH * (1.0 - 0.005 * k)))
    DevicePipeline(trk).submit(pool[0], outs[0], cameras=VARIANTS["cameras64"])    # both buffer sets allocated
    torch.cuda.synchronize()
    camera_mem_mb = (mem0 - torch.cuda.mem_get_info()[0]) / 1e6
    names = list(VARIANTS)
    times = {n: [] for n in names}
    valid = {}
    stream = torch.cuda.current_stream()
    for r in range(args.repeats):
        for name in names[r % len(names):] + names[:r % len(names)]:
            cams = VARIANTS[name]
            trk.reset()
            pipe = DevicePipeline(trk)
            for k in range(args.warmup):
                pipe.submit(pool[k % P], outs[k & 1], cameras=cams)
            pipe.join()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.warmup, args.warmup + args.batches):
                pipe.submit(pool[k % P], outs[k & 1], cameras=cams)
            pipe.join()
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.batches)
            valid[name] = float(pipe.fetch_results(S)["valid_lane_lines"].mean())
    stages = {}
    for name in names:
        cams = VARIANTS[name]
        trk.reset()
        for k in range(2):                                            # warm-up outside the recorded calls
            trk.process_async(pool[k % P], outs[k & 1], cameras=cams)
        trk.profile_begin(args.stage_calls)
        for k in range(args.stage_calls):
            trk.process_async(pool[k % P], outs[k & 1], cameras=cams)
        ms, calls = trk.profile_read()
        stages[name] = {st: round(v / max(calls, 1), 4) for st, v in ms.items() if v > 0}
    trk.close()
    out = dict(metric="DevicePipeline frames/s, 64 streams, frames from several cameras", streams=S,
               img_size=[1280, 720], batches=args.batches, warmup=args.warmup, repeats=args.repeats, card=card(),
               camera_buffers_mb_64_cameras_two_sets=round(camera_mem_mb, 1),
               variants={n: dict(fps_median=round(S * 1000.0 / float(np.median(v)), 1),
                                 ms_median=round(float(np.median(v)), 4), ms_min=round(float(min(v)), 4),
                                 ms_max=round(float(max(v)), 4), all_ms=[round(x, 4) for x in v],
                                 valid_rate_last_batch=valid[n], stage_ms_per_call=stages[n])
                         for n, v in times.items()})
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
