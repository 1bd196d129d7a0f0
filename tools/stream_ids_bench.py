"""DevicePipeline ms per batch with and without stream ids, at the bench's default geometry.

    python tools/stream_ids_bench.py [--batches 48] [--warmup 8] [--repeats 5] [--out FILE]

64 streams of 1280x720 road video (four pre-rendered frames per stream, device-resident; one batch is 177 MB of
input, more than the 126 MB L2), timed with CUDA events around `--batches` submissions through DevicePipeline:
  prefix      submit(frames, out)                      -- lt_process_front + lt_process_back
  identity    submit(frames, out, ids=range(64))       -- + the id upload, state addressed through the id map
  permuted    submit(frames, out, ids=<fixed permutation of 64>)
  subset32    submit(frames32, out32, ids=<random 32 of 64, changing per batch>)
The variants alternate within each repeat (rotated order), the tracker is reset before each one, and the output
reports the median and the spread (min, max) over repeats with the card's name and power limit."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stream_ids_bench needs a CUDA device")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, synth
    pool = torch.from_numpy(np.ascontiguousarray(synth.render_streams(S, P).transpose(1, 0, 2, 3, 4))).cuda()  # [P, S, ...]
    rng = np.random.default_rng(64)
    perm = rng.permutation(S)
    subsets = [np.sort(rng.choice(S, 32, replace=False)) for _ in range(2 * P)]
    # frames of a subset batch: stream s always sees its own road (seed s), gathered once outside the timed region
    sub_frames = [pool[j % P][torch.as_tensor(ids, device=pool.device)].contiguous() for j, ids in enumerate(subsets)]
    outs = [torch.empty_like(pool[0]) for _ in range(2)]
    outs32 = [torch.empty_like(sub_frames[0]) for _ in range(2)]
    trk = BatchedLaneTracker(S, **synth.shipped_calibration())

    def batch(name, k):
        if name == "prefix":
            return pool[k % P], outs[k & 1], None
        if name == "identity":
            return pool[k % P], outs[k & 1], range(S)
        if name == "permuted":      # frame i (road of seed i) belongs to stream perm[i], every batch
            return pool[k % P], outs[k & 1], perm
        j = k % len(subsets)
        return sub_frames[j], outs32[k & 1], subsets[j]

    names = ["prefix", "identity", "permuted", "subset32"]
    times = {n: [] for n in names}
    stream = torch.cuda.current_stream()
    for r in range(args.repeats):
        for name in names[r % 4:] + names[:r % 4]:
            trk.reset()
            pipe = DevicePipeline(trk)
            for k in range(args.warmup):
                f, o, ids = batch(name, k)
                pipe.submit(f, o, ids=ids)
            pipe.join()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.warmup, args.warmup + args.batches):
                f, o, ids = batch(name, k)
                pipe.submit(f, o, ids=ids)
            pipe.join()
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.batches)
            res = pipe.fetch_results(len(ids) if ids is not None else S)
            assert res["valid_lane_lines"].mean() > 0.5, (name, res["valid_lane_lines"].mean())
    trk.close()
    out = dict(metric="DevicePipeline ms per batch", streams=S, img_size=[1280, 720], batches=args.batches,
               warmup=args.warmup, repeats=args.repeats, card=card(),
               variants={n: dict(median_ms=float(np.median(v)), min_ms=float(min(v)), max_ms=float(max(v)),
                                 all_ms=[round(x, 4) for x in v]) for n, v in times.items()})
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
