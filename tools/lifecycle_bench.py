"""Cost of stream starts inside DevicePipeline, and of moving streams with state records.

    python tools/lifecycle_bench.py [--batches 60] [--warmup 8] [--repeats 3] [--out profiles/r03_lifecycle_bench.json]

64 streams of 1280x720 road video (four pre-rendered frames per stream, device-resident; one batch is 177 MB of
input, more than the 126 MB L2) through DevicePipeline, frames/s over `--batches` submissions timed with CUDA events:
  none            submit(frames, out)
  starts8         8 streams start a new video in every batch (starts=, a different 8 each batch)
  all64_every10   all 64 streams start a new video every 10th batch (starts=)
  join_reset_every10   what a caller without starts does every 10th batch: join, synchronise, reset(range(64)),
                  then submit
The variants alternate within each repeat (rotated order); the output reports the median and the spread (min, max)
over repeats.  Then export_states + import_states of 64 streams between two handles on one GPU (CUDA events, mean
over 50 moves), and, when a second GPU is present, export on cuda:0, a tensor copy to cuda:1 and import there (CUDA
events on each device around its part, mean over 50 moves; the copy runs on cuda:0's stream).  The card's name and
power limit are read in the same run."""
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
    ap.add_argument("--batches", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lifecycle_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("lifecycle_bench needs a CUDA device")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, synth
    pool = torch.from_numpy(np.ascontiguousarray(synth.render_streams(S, P).transpose(1, 0, 2, 3, 4))).cuda()  # [P, S, ...]
    outs = [torch.empty_like(pool[0]) for _ in range(2)]
    trk = BatchedLaneTracker(S, **synth.shipped_calibration())
    none = [False] * S

    def starts(name, k):
        if name == "starts8":
            return [(s - 8 * k) % S < 8 for s in range(S)]
        if name == "all64_every10" and k % 10 == 0:
            return [True] * S
        return None

    names = ["none", "starts8", "all64_every10", "join_reset_every10"]
    fps = {n: [] for n in names}
    stream = torch.cuda.current_stream()
    for r in range(args.repeats):
        for name in names[r % 4:] + names[:r % 4]:
            trk.reset()
            pipe = DevicePipeline(trk)
            for k in range(args.warmup):
                pipe.submit(pool[k % P], outs[k & 1], starts=starts(name, k) or none)
            pipe.join()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.warmup, args.warmup + args.batches):
                if name == "join_reset_every10" and k % 10 == 0:
                    pipe.join()
                    torch.cuda.synchronize()
                    trk.reset(range(S))
                pipe.submit(pool[k % P], outs[k & 1], starts=starts(name, k))
            pipe.join()
            e1.record(stream)
            e1.synchronize()
            fps[name].append(S * args.batches * 1000.0 / e0.elapsed_time(e1))
            res = pipe.fetch_results(S)
            assert res["valid_lane_lines"].mean() > 0.5, (name, res["valid_lane_lines"].mean())

    # state records: 64 streams between two handles on one GPU
    other = BatchedLaneTracker(S, **synth.shipped_calibration())
    ids = list(range(S))
    rec = trk.export_states(ids)
    st = other.import_states(ids, rec)
    n_moves = 50
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    ev[0].record(stream)
    for _ in range(n_moves):
        trk.export_states(ids, out=rec)
    ev[1].record(stream)
    for _ in range(n_moves):
        other.import_states(ids, rec, check=False)
    ev[2].record(stream)
    ev[2].synchronize()
    assert (st.cpu().numpy() == 0).all()
    assert torch.equal(other.export_states(ids), trk.export_states(ids))
    records = dict(streams=S, record_bytes=trk.record_bytes, total_bytes=S * trk.record_bytes,
                   export_ms=ev[0].elapsed_time(ev[1]) / n_moves, import_ms=ev[1].elapsed_time(ev[2]) / n_moves)
    cross = None
    if torch.cuda.device_count() > 1:
        far = BatchedLaneTracker(S, **synth.shipped_calibration(), device=1)
        rec1 = torch.empty(rec.shape, dtype=torch.uint8, device="cuda:1")
        s1 = torch.cuda.current_stream(1)
        t = dict(export_ms=0.0, copy_ms=0.0, import_ms=0.0)

        def move(timed):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            f = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record(stream)
            trk.export_states(ids, out=rec)
            e[1].record(stream)
            rec1.copy_(rec, non_blocking=True)          # on cuda:0's current stream
            e[2].record(stream)
            with torch.cuda.device(1):
                s1.wait_event(e[2])
                f[0].record(s1)
                far.import_states(ids, rec1, check=False)
                f[1].record(s1)
            f[1].synchronize()
            if timed:
                t["export_ms"] += e[0].elapsed_time(e[1]) / n_moves
                t["copy_ms"] += e[1].elapsed_time(e[2]) / n_moves
                t["import_ms"] += f[0].elapsed_time(f[1]) / n_moves

        move(False)
        for _ in range(n_moves):
            move(True)
        cross = dict(t, clock="CUDA events: export and copy on cuda:0, import on cuda:1")
        with torch.cuda.device(1):
            assert torch.equal(far.export_states(ids).cpu(), trk.export_states(ids).cpu())
        far.close()
    other.close()
    trk.close()
    out = dict(metric="DevicePipeline frames/s with stream starts; state record moves", streams=S,
               img_size=[1280, 720], batches=args.batches, warmup=args.warmup, repeats=args.repeats, card=card(),
               variants={n: dict(median_fps=float(np.median(v)), min_fps=float(min(v)), max_fps=float(max(v)),
                                 all_fps=[round(x, 1) for x in v]) for n, v in fps.items()},
               records_one_gpu=records, records_cuda0_to_cuda1=cross)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
