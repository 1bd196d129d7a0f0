#!/usr/bin/env python3
"""Stage times of the filter front half at S=64 for a list of morphology band splits.
The morphology kernels do not branch on pixel values, so random frames are as good as rendered ones."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def one():
    import torch
    sys.path.insert(0, ROOT)
    from lane_tracker_b200 import BatchedLaneTracker, synth
    S = int(os.environ.get("LT_BENCH_STREAMS", "64"))
    dev = torch.device("cuda", 0)
    if os.environ.get("LT_BENCH_SYNTH"):
        pool = torch.from_numpy(synth.render_streams(S, 2, first_seed=0, workers=16)).to(dev).permute(1, 0, 2, 3, 4).contiguous()
    else:
        g = torch.Generator(device="cuda").manual_seed(1)
        pool = torch.randint(0, 256, (2, S, 720, 1280, 3), dtype=torch.uint8, device=dev, generator=g)
    out = torch.empty_like(pool[0])
    trk = BatchedLaneTracker(S, **synth.shipped_calibration(), device=0)
    for i in range(3):
        trk.process_async(pool[i % 2], out, n_tries=1)
    torch.cuda.synchronize()
    n = 30
    trk.profile_begin(n)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        trk.process_async(pool[i % 2], out, n_tries=1)
    e1.record()
    torch.cuda.synchronize()
    st, calls = trk.profile_read()
    print(json.dumps({"bands": os.environ.get("LT_MORPH_BANDS", "auto"), "chosen": trk.morph_bands(), "ms_per_step": e0.elapsed_time(e1) / n,
                      "stages": {k: round(v / calls, 4) for k, v in st.items() if v > 0}}), flush=True)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--one":
        return one()
    for bands in sys.argv[1:] or ["auto", "2,5", "2,4", "3,5", "3,6", "2,6", "4,8"]:
        env = dict(os.environ)
        env.pop("LT_MORPH_BANDS", None)
        if bands != "auto":
            env["LT_MORPH_BANDS"] = bands
        subprocess.run([sys.executable, os.path.abspath(__file__), "--one"], env=env, check=False)


if __name__ == "__main__":
    main()
