"""Frame sequences (sequence=True) against one frame per stream per batch, at the bench's 1280x720 geometry.

    python tools/sequence_bench.py [--frames 1000] [--repeats 3] [--out FILE]

Cases (the variants of a case alternate in rotated order over `--repeats` timed runs; the tracker is reset before
every run, and each variant is warmed up by an untimed parity pass first):
  single      one stream of `--frames` frames (BASELINE configs[1]: 200 distinct frames of one road video, cycled)
              graph       GraphedProcess, one frame per replay, records read every frame (the configs[1] line of
                          bench.py --config single)
              seq_B       process(B frames, ids=[0] * B, sequence=True), records read every call
              pipe_B      DevicePipeline.submit(B frames, ids=[0] * B, sequence=True), records read at the end
              for B in 16, 32, 64
  multi_KxM   K streams x M frames per batch of 64 (4x16, 8x8, 16x4; round-major), 1024 frames, DevicePipeline
              seq         submit(64 frames, ids=..., sequence=True)
              per_frame   submit(K frames, ids=range(K)): one frame per stream per batch
  distinct64  64 streams, 16 batches of one frame per stream, ids a fixed permutation, DevicePipeline
              seq         submit(..., ids=perm, sequence=True)
              ids         submit(..., ids=perm)
Reported per variant: frames/s (median, min, max over the runs), host enqueue ms per call (median), and stage ms per
frame from a separate profiled pass through process().  Parity, in the same run: each variant's untimed first pass
(the pipelines read the records after every batch there) gives every frame's record and the sha256 of the annotated
frames of its first 128 frames, keyed by (stream, frame); they must equal the first variant's (the per-frame path)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def summary(v):
    return dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sequence_bench needs a CUDA device")
    import warnings
    warnings.simplefilter("ignore")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, GraphedProcess, synth
    # render first: the renderer forks worker processes, which should not inherit a CUDA context
    vid = synth.RoadVideo(0)
    pool_np = np.stack([vid.frame(t) for t in range(200)])
    T = 16
    vids_np = synth.render_streams(16, T, workers=16)                                # [16 streams, T, H, W, 3]
    v64_np = synth.render_streams(64, 4, first_seed=100, workers=16)                 # [64, 4, H, W, 3]
    cal = synth.shipped_calibration()
    big = BatchedLaneTracker(64, **cal)
    one = BatchedLaneTracker(1, **cal)
    graph = GraphedProcess(one, 1)
    outs = [torch.empty((64, 720, 1280, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]

    def sha(t):
        return hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()[:16]

    # A variant is a list of batches (frames, ids, sequence, keys): keys[i] = (stream, frame index) of position i.
    def run(batches, mode, profile=False, check=False):
        """mode 'graph' (one-frame batches of stream 0), 'process' or 'pipe' -> (seconds, enqueue ms per call,
        {key: record bytes}, {key: out sha} of the first 128 frames, stage ms)."""
        trk = one if mode == "graph" else big
        trk.reset()
        pipe = DevicePipeline(big) if mode == "pipe" else None
        recs, hashes, enq = {}, {}, []
        if profile:
            trk.profile_begin(len(batches))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k, (f, ids, seq, keys) in enumerate(batches):
            e0 = time.perf_counter()
            if mode == "graph":
                graph.frames.copy_(f, non_blocking=True)
                graph.replay()
                enq.append(1e3 * (time.perf_counter() - e0))
                res, out = graph.fetch_results(), graph.out
            elif mode == "process":
                out = outs[k & 1][:len(f)]
                trk.process_async(f, out, ids=ids, sequence=seq)
                enq.append(1e3 * (time.perf_counter() - e0))
                res = trk.fetch_results(len(f))
            else:
                out = outs[k & 1][:len(f)]
                pipe.submit(f, out, ids=ids, sequence=seq)
                enq.append(1e3 * (time.perf_counter() - e0))
                res = pipe.fetch_results(len(f)) if (check or k == len(batches) - 1) else None
            if check:
                for i, key in enumerate(keys):
                    recs[key] = res[i].tobytes()
                    if len(hashes) < 128:
                        hashes[key] = sha(out[i])
        if pipe is not None:
            pipe.join()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        stages = trk.profile_read()[0] if profile else None
        return dt, float(np.median(enq)) if enq else None, recs, hashes, stages

    result = dict(metric="frames/s", img_size=[1280, 720], repeats=args.repeats, card=card(), cases={})

    def case(name, variants, workload):
        """variants: {name: (batches, mode)}; the first is the reference of the parity check."""
        names = list(variants)
        nf = {v: sum(len(b[0]) for b in variants[v][0]) for v in names}
        ref, parity, stages = None, True, {}
        for v in names:                                    # untimed parity pass (and warm-up)
            batches, mode = variants[v]
            _, _, recs, hashes, _ = run(batches, mode, check=True)
            if ref is None:
                ref = (recs, hashes)
            else:
                parity &= recs == ref[0] and all(ref[1].get(k) == h for k, h in hashes.items())
            if mode != "graph":
                b = batches[:max(1, 256 // len(batches[0][0]))]
                st = run(b, "process", profile=True)[4]
                stages[v] = {k: x / sum(len(x_[0]) for x_ in b) for k, x in st.items() if x > 0}
        times = {v: [] for v in names}
        enqs = {v: [] for v in names}
        for r in range(args.repeats):
            for v in names[r % len(names):] + names[:r % len(names)]:
                batches, mode = variants[v]
                dt, enq, _, _, _ = run(batches, mode)
                times[v].append(nf[v] / dt)
                if enq is not None:
                    enqs[v].append(enq)
        result["cases"][name] = dict(workload=workload, parity=bool(parity),
                                     frames_per_s={v: summary(x) for v, x in times.items()},
                                     enqueue_ms_per_call={v: float(np.median(x)) for v, x in enqs.items() if x},
                                     stage_ms_per_frame=stages)
        print(name, json.dumps(result["cases"][name]["frames_per_s"]), "parity", parity, flush=True)

    # ---- single: one stream ----------------------------------------------------------------------------------------
    N = args.frames
    pool = torch.from_numpy(pool_np).cuda()

    def chunks(B):
        return [(pool[torch.arange(a, min(a + B, N), device="cuda") % len(pool)].contiguous(), [0] * (min(a + B, N) - a),
                 True, [(0, t) for t in range(a, min(a + B, N))]) for a in range(0, N, B)]

    single = {"graph": ([(pool[t % len(pool)][None], [0], False, [(0, t)]) for t in range(N)], "graph")}
    for mode, tag in (("process", "seq"), ("pipe", "pipe")):
        for B in (16, 32, 64):
            single["%s_%d" % (tag, B)] = (chunks(B), mode)
    case("single", single, "one stream, %d frames (200 distinct frames of one road video, cycled)" % N)
    del single

    # ---- several streams -------------------------------------------------------------------------------------------
    vids = torch.from_numpy(vids_np).cuda()
    for K, M in ((4, 16), (8, 8), (16, 4)):
        per = 1024 // K
        seq = []
        for t0 in range(0, per, M):
            ids = [s for _ in range(M) for s in range(K)]
            ts = [t0 + j for j in range(M) for _ in range(K)]
            f = vids[torch.as_tensor(ids, device="cuda"), torch.as_tensor(ts, device="cuda") % T].contiguous()
            seq.append((f, ids, True, list(zip(ids, ts))))
        flat = [(vids[:K, t % T].contiguous(), list(range(K)), False, [(s, t) for s in range(K)]) for t in range(per)]
        case("multi_%dx%d" % (K, M), {"per_frame": (flat, "pipe"), "seq": (seq, "pipe")},
             "%d streams x %d frames per batch of 64 (round-major), 1024 frames, DevicePipeline; per_frame: batches of "
             "%d, one frame per stream" % (K, M, K))
    del vids
    v64 = torch.from_numpy(v64_np).cuda()
    perm = [int(x) for x in np.random.default_rng(64).permutation(64)]
    d64 = [(v64[perm, t % 4].contiguous(), perm, None, [(s, t) for s in perm]) for t in range(16)]
    case("distinct64", {"ids": ([b[:2] + (False,) + b[3:] for b in d64], "pipe"),
                        "seq": ([b[:2] + (True,) + b[3:] for b in d64], "pipe")},
         "64 distinct streams, 16 batches of one frame per stream, ids a fixed permutation, DevicePipeline")
    big.close()
    one.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    bad = [n for n, c in result["cases"].items() if not c["parity"]]
    if bad:
        raise SystemExit("parity failed: %s" % bad)


if __name__ == "__main__":
    main()
