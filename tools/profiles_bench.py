"""DevicePipeline frames/s of batches whose frames use different parameter profiles, at the bench's default geometry.

    python tools/profiles_bench.py [--batches 48] [--warmup 8] [--repeats 5] [--stage-calls 16] [--out FILE]

64 streams of 1280x720 road video (four pre-rendered frames per stream, device-resident; one batch is 177 MB of
input, more than the 126 MB L2), timed with CUDA events around `--batches` submissions through DevicePipeline:
  plain        submit(frames, out) with params = DEMO_2 (and its windows through set_validity)
  one_profile  the same settings as profile 0 for every frame: submit(frames, out, profiles=[0] * 64)
  two_filters  DEMO_1 / DEMO_2 alternating by position (32 + 32): two filter groups
  presets4     DEMO_1, DEMO_2, DEMO_3 and the defaults, position i -> i % 4: three filter groups (DEMO_1 and DEMO_3
               share a filter configuration), four sets of search settings and windows
  search4      four profiles with DEMO_2's filter that differ in search settings and windows only: one filter group
The variants alternate within each repeat (rotated order) and the tracker is reset before each one; the output reports
the median and spread (min, max) over repeats.  Per-stage times come from lt_profile_* over `--stage-calls` sequential
process() calls per variant, in a separate pass (event recording adds host work).  The card's name and power limit
are read in the same run."""
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


def variants():
    """name -> (profile table {k: (process keywords, validity)}, profile of each position or None for plain)."""
    from lane_tracker_b200 import presets
    d1, d2, d3 = (presets.DEMO_1, presets.DEMO_2, presets.DEMO_3)
    p2, v2 = d2["process"], d2["validity"]
    return {
        "plain": ({}, None),
        "one_profile": ({0: (p2, v2)}, [0] * S),
        "two_filters": ({1: (d1["process"], d1["validity"]), 2: (p2, v2)}, [1 + (i & 1) for i in range(S)]),
        "presets4": ({0: ({}, None), 1: (d1["process"], d1["validity"]), 2: (p2, v2), 3: (d3["process"], d3["validity"])},
                     [i % 4 for i in range(S)]),
        "search4": ({0: (p2, v2), 1: (dict(p2, window_width=40), d1["validity"]),
                     2: (dict(p2, search_range=30, mu=0.2), d3["validity"]), 3: (dict(p2, partial=0.8), v2)},
                    [i % 4 for i in range(S)]),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--stage-calls", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("profiles_bench needs a CUDA device")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, make_params, presets, synth
    pool = torch.from_numpy(np.ascontiguousarray(synth.render_streams(S, P).transpose(1, 0, 2, 3, 4))).cuda()  # [P, S, ...]
    outs = [torch.empty_like(pool[0]) for _ in range(2)]
    trk = BatchedLaneTracker(S, **synth.shipped_calibration())
    plain_params = make_params(**presets.DEMO_2["process"])
    table = variants()

    def install(name):
        profs, prof = table[name]
        trk.reset()
        if prof is None:
            trk.set_validity(**presets.DEMO_2["validity"])
        else:
            trk.set_validity()
            for k, (kw, val) in profs.items():
                trk.set_profile(k, validity=val, **kw)
        return prof

    names = list(table)
    times = {n: [] for n in names}
    valid = {}
    stream = torch.cuda.current_stream()
    for r in range(args.repeats):
        for name in names[r % len(names):] + names[:r % len(names)]:
            prof = install(name)
            pipe = DevicePipeline(trk, params=plain_params)
            for k in range(args.warmup):
                pipe.submit(pool[k % P], outs[k & 1], profiles=prof)
            pipe.join()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(args.warmup, args.warmup + args.batches):
                pipe.submit(pool[k % P], outs[k & 1], profiles=prof)
            pipe.join()
            e1.record(stream)
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.batches)
            res = pipe.fetch_results(S)
            valid[name] = float(res["valid_lane_lines"].mean())
    stages = {}
    for name in names:
        prof = install(name)
        kw = {} if prof is not None else dict(params=plain_params)
        for k in range(2):                                            # warm-up outside the recorded calls
            trk.process_async(pool[k % P], outs[k & 1], profiles=prof, **kw)
        trk.profile_begin(args.stage_calls)
        for k in range(args.stage_calls):
            trk.process_async(pool[k % P], outs[k & 1], profiles=prof, **kw)
        ms, calls = trk.profile_read()
        stages[name] = {st: round(v / max(calls, 1), 4) for st, v in ms.items() if v > 0}
    trk.close()
    out = dict(metric="DevicePipeline frames/s, 64 streams, per-frame parameter profiles", streams=S,
               img_size=[1280, 720], batches=args.batches, warmup=args.warmup, repeats=args.repeats, card=card(),
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
