"""NV12 input frames against a separate NV12 -> RGB pass, and what NV12 saves across PCIe.

    python tools/nv12_bench.py [--batches 32] [--warmup 6] [--repeats 5] [--out FILE]

64 streams of 1280x720 road video (four pre-rendered frames per stream, converted to NV12 by synth.rgb_to_nv12; the
device pools are 354 MB NV12 and 708 MB RGB, more than the 126 MB L2).  Variants, ms per batch of 64 frames:
  (a) DevicePipeline, device-resident frames, with overlay and fits only (out=None):
        convert_*   nv12_to_rgb into one of two RGB buffers, then submit(rgb)   (before converting into a buffer the
                    current stream waits for the batch that last read it)
        native_*    submit(nv12)
  (b) HostPipeline(overlay=False), pinned host frames:
        host_fits_rgb    RGB, whole frames uploaded
        host_fits_nv12   NV12, only the rows the tracker reads and their chroma rows uploaded
  (c) HostPipeline with the annotated frames returned:
        host_inplace_rgb   RGB inplace=True (rows the tracker reads go up, overlay rows come back)
        host_overlay_nv12  NV12 overlay=True (whole NV12 frames up, whole RGB frames back)
The variants of a group alternate within each repeat (rotated order), the tracker is reset before each one, and the
output reports the median and the spread (min, max) over repeats, with the card's name and power limit and the bytes
each variant moves per frame."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

S, P = 64, 4
W, H = 1280, 720


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nv12_bench needs a CUDA device")
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, HostPipeline, synth
    nv_host = synth.rgb_to_nv12(synth.render_streams(S, P, workers=8).transpose(1, 0, 2, 3, 4))     # [P, S, H*3/2, W]
    trk = BatchedLaneTracker(S, **synth.shipped_calibration())
    nv_pool = torch.from_numpy(np.ascontiguousarray(nv_host)).cuda()
    rgb_pool = torch.stack([trk.nv12_to_rgb(nv_pool[k]) for k in range(P)])                       # [P, S, H, W, 3]
    nv_pinned = [torch.from_numpy(np.ascontiguousarray(nv_host[k])).pin_memory() for k in range(P)]
    rgb_pinned = [rgb_pool[k].cpu().pin_memory() for k in range(P)]
    del nv_host
    outs = [torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
    conv = [torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
    stream = torch.cuda.current_stream()
    src0, src1 = trk.geometry["source_rows"]
    rgb_frame, nv_frame = H * W * 3, H * W * 3 // 2

    def run_device(name, k0, k1, pipe, done):
        for k in range(k0, k1):
            out = outs[k & 1] if name.endswith("overlay") else None
            if name.startswith("convert"):
                if k >= 2:
                    stream.wait_event(done[k - 2])
                f = trk.nv12_to_rgb(nv_pool[k % P], out=conv[k & 1])
            else:
                f = nv_pool[k % P]
            done[k] = pipe.submit(f, out)

    def time_device(name):
        trk.reset()
        pipe, done = DevicePipeline(trk), {}
        run_device(name, 0, args.warmup, pipe, done)
        pipe.join()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_device(name, args.warmup, args.warmup + args.batches, pipe, done)
        pipe.join()
        e1.record(stream)
        e1.synchronize()
        res = pipe.fetch_results(S)
        assert res["valid_lane_lines"].mean() > 0.5, (name, res["valid_lane_lines"].mean())
        return e0.elapsed_time(e1) / args.batches

    def time_host(name):
        trk.reset()
        if name == "host_fits_rgb":
            pipe, pool = HostPipeline(trk, overlay=False), rgb_pinned
        elif name == "host_fits_nv12":
            pipe, pool = HostPipeline(trk, overlay=False, frame_format="nv12"), nv_pinned
        elif name == "host_inplace_rgb":
            pipe, pool = HostPipeline(trk, inplace=True), [f.clone().pin_memory() for f in rgb_pinned]
        else:
            pipe, pool = HostPipeline(trk, frame_format="nv12"), nv_pinned
        valid = []

        def feed(k0, k1):
            for k in range(k0, k1):
                if pipe.inflight == pipe.depth:
                    for _, r in pipe.ready():
                        valid.append(r["valid_lane_lines"].mean())
                pipe.submit(pool[k % P])
            for _, r in pipe.drain():
                valid.append(r["valid_lane_lines"].mean())

        feed(0, args.warmup)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        feed(args.warmup, args.warmup + args.batches)
        dt = (time.perf_counter() - t0) * 1e3 / args.batches
        assert np.mean(valid[-args.batches:]) > 0.5, (name, np.mean(valid))
        if name == "host_inplace_rgb":
            for f, g in zip(pool, rgb_pinned):
                f.copy_(g)
        return dt

    groups = {
        "a_overlay": (["convert_overlay", "native_overlay"], time_device),
        "a_fits": (["convert_fits", "native_fits"], time_device),
        "b_host_fits": (["host_fits_rgb", "host_fits_nv12"], time_host),
        "c_host_overlay": (["host_inplace_rgb", "host_overlay_nv12"], time_host),
    }
    times = {n: [] for names, _ in groups.values() for n in names}
    for r in range(args.repeats):
        for names, fn in groups.values():
            for name in (names if r % 2 == 0 else names[::-1]):
                times[name].append(fn(name))
    trk.close()
    g = trk.geometry
    ov0, ov1 = g["overlay_rows"]
    in_rows = (max(0, min(src0, ov0) - 2), min(H, max(src1, ov1) + 2))
    h2d = dict(convert_overlay=0, native_overlay=0, convert_fits=0, native_fits=0, host_fits_rgb=rgb_frame,
               host_fits_nv12=(src1 - src0) * W + ((src1 + 1) // 2 - src0 // 2) * W,
               host_inplace_rgb=(in_rows[1] - in_rows[0]) * W * 3, host_overlay_nv12=nv_frame)
    d2h = dict(host_inplace_rgb=(ov1 - ov0) * W * 3, host_overlay_nv12=rgb_frame)
    out = dict(metric="ms per batch of 64 frames", streams=S, img_size=[W, H], batches=args.batches,
               warmup=args.warmup, repeats=args.repeats, card=card(), source_rows=[src0, src1],
               overlay_rows=[ov0, ov1],
               variants={n: dict(median_ms=float(np.median(v)), min_ms=float(min(v)), max_ms=float(max(v)),
                                 frames_per_s=float(S * 1e3 / np.median(v)), all_ms=[round(x, 4) for x in v],
                                 h2d_bytes_per_frame=h2d.get(n, 0), d2h_frame_bytes_per_frame=d2h.get(n, 0))
                         for n, v in times.items()})
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
