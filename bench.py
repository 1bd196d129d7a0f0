#!/usr/bin/env python3
"""Benchmark of the lane-tracking hot path (BASELINE.json metric: frames/sec at 1280x720, batched streams).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, BASELINE configs[2] (x N = configs[3] weak)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores
    python bench.py --config single|512|1080p|2160p|mixed    # the other BASELINE configs (see DESIGN.md section 7)
    python bench.py --steps K --dump-outputs DIR             # also write what the last timed step computed (OutputDump)

Default workload (BASELINE.json configs[2] per GPU): 64 independent synthetic 1280x720 road videos per GPU, one frame per
stream per batch, full process() semantics (sliding-window search on the first frame, band-search tracking afterwards,
overlay rendered).  A driver "step" is BATCHES_PER_STEP consecutive batches, so that the timed region is long enough to
be clocked.  Streams are sharded across ranks with no collective on the data path; torch.distributed is used only for
the timing barrier (and, in --config 512, a host-side gloo gather of the result records).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "frames/sec at 1280x720 (batched streams)"
STREAMS_PER_GPU = 64
FRAME_POOL = 4                       # pre-rendered frames per stream, cycled
BATCHES_PER_STEP = 16                # a driver step = 16 batches of STREAMS_PER_GPU frames (>= 0.3 s timed at the default 20 steps)
FRAME_BYTES = 1280 * 720 * 3
ALGO_BYTES_PER_FRAME = 2 * FRAME_BYTES + 128          # SURVEY.md 8(d): frame in + annotated frame out + results
PLANE_PIXELS = 1080 * 1100
MORPH_ALGO_BYTES_PER_FRAME = 4 * PLANE_PIXELS         # per morphology stage: two u8 planes (R, Lab-b) read + two written
PARITY_FRAMES = 6                    # frames per stream compared with the oracle by the in-bench parity check
PARITY_RTOL = 1e-6                   # polynomial coefficients vs np.polyfit (BASELINE.json north_star)
DUMP_FRAME_SAMPLES = 12288           # --dump-outputs: bytes of each annotated frame kept (16 x 64 x 12288 float32 = 50 MB)


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:32]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [v.strip() for v in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port with the reference's own cv2 calls)
# ----------------------------------------------------------------------------------------------

def _cpu_worker(args):
    """One stream on one core: (frames processed, seconds, success count, operator backend, parity records).
    The parity records are what the GPU arm's in-bench check compares: result fields plus digests of the final mask and
    of the output frame for the first `n_records` frames of the stream."""
    seed, n_frames, warm, n_records = args
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    import warnings
    warnings.simplefilter("ignore")
    from lane_tracker_b200 import synth
    from oracle.tracker import OracleLaneTracker
    backend = "numpy"
    try:
        import cv2
        cv2.setNumThreads(1)
        backend = "cv2"
    except Exception:
        pass
    vid = synth.RoadVideo(seed)
    total = warm + n_frames
    frames = [vid.frame(t) for t in range(min(FRAME_POOL, max(total, n_records)))]
    trk = OracleLaneTracker(**synth.shipped_calibration(), backend=backend)
    records = []

    def one(t):
        out = trk.process(frames[t % len(frames)].copy())
        if t < n_records:
            last = trk.trace["attempts"][-1]
            rec = dict(counter=trk.counter, attempts=len(trk.trace["attempts"]), mode=last["mode"],
                       detected=bool(trk.detected_pixels), valid=bool(trk.valid_lane_lines),
                       last_detection=int(trk.last_detection), mask=sha(last["mask"]), out=sha(out))
            if last["detected"]:
                rec.update(left_fit=[float(v) for v in last["left_fit"]], right_fit=[float(v) for v in last["right_fit"]],
                           n_left=int(len(last["left_x"])), n_right=int(len(last["right_x"])))
            if trk.valid_lane_lines:
                rec.update(radius=int(trk.average_curve_radius), ecc=float(trk.eccentricity))
            records.append(rec)

    for t in range(warm):
        one(t)
    t0 = time.perf_counter()
    for t in range(warm, total):
        one(t)
    dt = time.perf_counter() - t0
    for t in range(total, n_records):          # (only when the timed sample was shorter than the parity window)
        one(t)
    return n_frames, dt, trk.success, backend, records


def cpu_baseline(budget_s=20.0, n_records=PARITY_FRAMES):
    """Bounded sample of the same workload on all host cores: one stream per core.  Also returns the oracle's records of
    the first frames of those streams for the GPU arm's parity check."""
    import multiprocessing as mp
    cores = host_cores()
    per_frame = 0.35            # s/frame/core with cv2 single-threaded (SURVEY.md section 6)
    n_frames = max(n_records, int(budget_s / per_frame))
    jobs = [(s, n_frames, 1, n_records) for s in range(cores)]
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    frames = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    line = {"value": frames / slowest, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": "%d streams x %d frames (1 warm-up frame each), one process per core, %s operators, "
                      "single-threaded; %.1f s wall" % (cores, n_frames, res[0][3], wall),
            "success_ratio": sum(r[2] for r in res) / float(sum(r[0] + 1 for r in res))}
    return line, [r[4] for r in res]


def run_reference_arm(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    import multiprocessing as mp
    cores = host_cores()
    n_frames = args.steps                      # per stream; a step = one frame on each of `cores` parallel streams
    jobs = [(s, n_frames, args.warmup, 0) for s in range(cores)]
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    slowest = max(r[1] for r in res)
    value = sum(r[0] for r in res) / slowest
    sample = ("%d of the %d streams (one per host core) x %d frames after %d warm-up frames; %s operators, "
              "1 thread per process" % (cores, STREAMS_PER_GPU * args.gpus, n_frames, args.warmup, res[0][3]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * slowest / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(n_gpus):
    return {"workload": "64 independent synthetic 1280x720 streams batched per B200 (BASELINE.json configs[2]; "
                        "x N GPUs = configs[3] sharding, no collective)",
            "streams_per_gpu": STREAMS_PER_GPU, "frame_pool_per_stream": FRAME_POOL, "mode": "process() with overlay",
            "step": "%d consecutive batches of %d frames per GPU" % (BATCHES_PER_STEP, STREAMS_PER_GPU),
            "bird_view": "1080x1100", "parallelism": "streams sharded over %d GPU(s), no data-path collective" % n_gpus,
            "pipelining": "DevicePipeline: two batches in flight per GPU on two CUDA streams (front half of batch k+1 "
                          "under the back half of batch k); results identical to sequential process() calls",
            "l2": "inputs larger than L2: %.0f MB of distinct frames read per batch" % (STREAMS_PER_GPU * FRAME_BYTES / 1e6)}


# ----------------------------------------------------------------------------------------------
# GPU arm, shared pieces
# ----------------------------------------------------------------------------------------------

class Ctx:
    """Device, process group and timing helpers of one rank."""

    def __init__(self, need_host_group=False):
        import torch
        self.torch = torch
        self.rank, self.world, self.local = dist_env()
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.distributed = self.world > 1
        self.host_group = None
        if self.distributed:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=self.dev)      # timing barrier only; the data path has no collective
            if need_host_group:
                self.host_group = dist.new_group(backend="gloo")     # host-side gather of the result records
        self.pin_to_cores()

    def pin_to_cores(self):
        """Each rank keeps to its own slice of the host cores (its submit loop and pinned-memory traffic do not migrate)."""
        try:
            cores = sorted(os.sched_getaffinity(0))
            if self.world > 1 and len(cores) >= self.world:
                per = len(cores) // self.world
                os.sched_setaffinity(0, set(cores[self.local * per:(self.local + 1) * per]))
        except Exception:
            pass

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, values):
        if not self.distributed:
            return list(values)
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def close(self):
        if self.distributed:
            self.dist.destroy_process_group()


def timed(ctx, stream, fn):
    """fn() enqueues work; returns the CUDA-event time [ms] between barriers, on `stream`."""
    torch = ctx.torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record(stream)
    fn()
    e1.record(stream)
    ctx.barrier()
    return e0.elapsed_time(e1)


def parity_check(ctx, trk, pool_dev, want, S):
    """Untimed: the first PARITY_FRAMES batches through DevicePipeline from a reset tracker, compared with the oracle's
    records of the same streams (computed on the host cores in the cpu_baseline leg): state machine, pixel counts,
    coefficients (rtol 1e-6), radius, and digests of the final mask and of every output frame (bit-exact)."""
    from lane_tracker_b200 import DevicePipeline
    torch = ctx.torch
    n = min(len(want), S)
    if n == 0:
        return {"parity_checked": False, "reason": "no oracle records (cpu baseline skipped)"}
    trk.reset()
    pipe = DevicePipeline(trk)
    outs = [torch.empty_like(pool_dev[0]) for _ in range(2)]
    bad = []
    P = pool_dev.shape[0]
    frames = min(PARITY_FRAMES, min(len(w) for w in want[:n]))
    for t in range(frames):
        pipe.submit(pool_dev[t % P], outs[t & 1])
        res = pipe.fetch_results(S)
        out = outs[t & 1][:n].cpu().numpy()
        for s in range(n):
            w, r = want[s][t], res[s]
            ok = (int(r["counter"]) == w["counter"] and int(r["attempts"]) == w["attempts"] and
                  int(r["search_mode"]) == (1 if w["mode"] == "bs" else 0) and bool(r["detected_pixels"]) == w["detected"] and
                  bool(r["valid_lane_lines"]) == w["valid"] and int(r["last_detection"]) == w["last_detection"] and
                  sha(out[s]) == w["out"])
            if ok and w["detected"]:
                ok = (int(r["n_left"]) == w["n_left"] and int(r["n_right"]) == w["n_right"] and
                      np.allclose(r["left_fit"], w["left_fit"], rtol=PARITY_RTOL, atol=0) and
                      np.allclose(r["right_fit"], w["right_fit"], rtol=PARITY_RTOL, atol=0))
            if ok and w["valid"]:
                ok = int(r["average_curve_radius"]) == w["radius"] and abs(float(r["eccentricity"]) - w["ecc"]) <= 1e-12
            if ok and t == frames - 1:
                ok = sha(trk.debug_read("mask", s)) == w["mask"]
            if not ok:
                bad.append([s, t])
    trk.reset()
    return {"parity_checked": len(bad) == 0, "streams": n, "frames_per_stream": frames, "mismatches": bad[:8],
            "compared": "per frame: counter, attempts, search mode, detected, valid, last_detection, pixel counts, fit "
                        "coefficients (rtol 1e-6), curve radius, eccentricity, sha256 of the output frame; final mask sha256",
            "morph_bands": list(trk.morph_bands())}


class OutputDump:
    """--dump-outputs: what a DevicePipeline caller receives from the last timed step, kept for comparing two builds.
    Each batch of that step writes its annotated frames to a buffer of its own, and its lt_result records are copied
    out on a side stream; before the pipeline reuses a results buffer (two batches later) the launch stream waits for
    that copy.  The inputs depend only on the arguments (seeded synthetic streams), so runs are comparable file by file."""

    def __init__(self, torch, like, batches):
        from lane_tracker_b200.tracker import RESULT_DTYPE
        self.torch, self.dtype = torch, RESULT_DTYPE
        self.frames = [torch.empty_like(like) for _ in range(batches)]
        self.results = torch.empty((batches, like.shape[0] * RESULT_DTYPE.itemsize), dtype=torch.uint8, device=like.device)
        self.copied = [None] * batches
        self.stream = torch.cuda.Stream(like.device)

    def submit(self, pipe, frames, j):
        """Batch j of the last step through `pipe`."""
        torch = self.torch
        if j >= 2:
            torch.cuda.current_stream(frames.device).wait_event(self.copied[j - 2])
        done = pipe.submit(frames, self.frames[j])
        self.stream.wait_event(done)
        with torch.cuda.stream(self.stream):
            self.results[j].copy_(pipe.last_results_dev()[:self.results.shape[1]])
            self.copied[j] = torch.cuda.Event()
            self.copied[j].record(self.stream)

    def write(self, path):
        """DIR/frames_sample.npy: float32 [batch, stream, DUMP_FRAME_SAMPLES], the annotated frames' bytes at fixed
        positions (ascending, drawn with numpy.random.default_rng(0)); DIR/result_<field>.npy: float64 [batch, stream
        (, 3)], every lt_result field."""
        torch = self.torch
        self.stream.synchronize()
        os.makedirs(path, exist_ok=True)
        S, n = self.frames[0].shape[0], self.frames[0][0].numel()
        pos = np.sort(np.random.default_rng(0).choice(n, DUMP_FRAME_SAMPLES, replace=False))
        pos = torch.from_numpy(pos).to(self.results.device)
        sample = torch.stack([f.view(S, -1)[:, pos] for f in self.frames]).cpu().numpy()
        np.save(os.path.join(path, "frames_sample.npy"), sample.astype(np.float32))
        res = self.results.cpu().numpy().view(self.dtype)
        for name in self.dtype.names:
            if not name.startswith("reserved"):
                np.save(os.path.join(path, "result_%s.npy" % name), res[name].astype(np.float64))


def render_pool(ctx, S, P, first_seed, scale=1.0, photos=None):
    """[P, S, H, W, 3] device pool and its pinned host twin; `photos`: frames that replace the LAST len(photos) streams."""
    torch = ctx.torch
    from lane_tracker_b200 import synth
    t0 = time.perf_counter()
    n_syn = S - (len(photos) if photos is not None else 0)
    pool_np = synth.render_streams(n_syn, P, scale=scale, first_seed=first_seed,
                                   workers=max(1, min(host_cores(), 32)))      # (a rank's cores: see Ctx.pin_to_cores)
    if photos is not None:
        pool_np = np.concatenate([pool_np, np.repeat(np.asarray(photos)[:, None], P, axis=1)])
    t_render = time.perf_counter() - t0
    host_batches = torch.from_numpy(np.ascontiguousarray(pool_np.transpose(1, 0, 2, 3, 4))).pin_memory()   # [P, S, H, W, 3]
    return host_batches.to(ctx.dev), host_batches, t_render


def e2e_runs(ctx, trk, host_batches, steps, batches_per_step, warm=3):
    """Host-to-host throughput through the public HostPipeline API (pinned frames in, annotated frames + results out,
    every batch): the row-ROI in-place form (the documented default host path) and the full-frame form."""
    from lane_tracker_b200 import HostPipeline
    torch = ctx.torch
    P = host_batches.shape[0]
    nb = steps * batches_per_step
    out = {}
    for name, kw in (("inplace", dict(inplace=True)), ("full", dict(overlay=True))):
        trk.reset()
        pipe = HostPipeline(trk, depth=3, **kw)
        src = [host_batches[i].clone().pin_memory() for i in range(P)] if name == "inplace" else host_batches
        seen = []

        def consume(batch):
            seen.append(int(batch[1]["counter"][0]))          # the host really reads every batch's result records

        def run(n):
            for i in range(n):
                pipe.submit(src[i % P])
                for b in pipe.ready():
                    consume(b)
            for b in pipe.drain():
                consume(b)

        run(warm)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.s_in)
        run(nb)
        e1.record(pipe.s_out)
        ctx.barrier()
        assert seen[-1] == warm + nb, "e2e pipeline lost a batch"
        out[name] = dict(ms=e0.elapsed_time(e1), rows_in=pipe.rows_in, rows_out=pipe.rows_out, rows_text=pipe.rows_text)
    return out


# ----------------------------------------------------------------------------------------------
# default config: BASELINE configs[2] per GPU (weak scaling over N GPUs)
# ----------------------------------------------------------------------------------------------

def run_default(args, photos_in_batch=False):
    rank, world, local = dist_env()
    cpu_line, want = None, []
    if rank == 0 and not args.no_cpu_baseline and not photos_in_batch:
        cpu_line, want = cpu_baseline(args.cpu_budget)        # before CUDA is initialised: the workers are forked
    ctx = Ctx()
    torch = ctx.torch
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, _lib, synth
    S, P, B = STREAMS_PER_GPU, FRAME_POOL, BATCHES_PER_STEP
    photos = load_photos() if photos_in_batch else None
    pool_dev, host_batches, t_render = render_pool(ctx, S, P, first_seed=rank * S, photos=photos)
    out_ring = [torch.empty_like(pool_dev[0]) for _ in range(2)]       # two batches in flight: two output buffers
    trk = BatchedLaneTracker(S, **synth.shipped_calibration(), device=local)
    lib = _lib.load()
    stream = torch.cuda.current_stream(ctx.dev)

    parity = parity_check(ctx, trk, pool_dev, want, S) if rank == 0 else None

    # ---- device-resident throughput through DevicePipeline, the public throughput API.  The two morphology stages
    # are timed live in this region (three events per batch, on the stream they are launched on).
    dpipe = DevicePipeline(trk)
    k = 0
    for _ in range(max(args.warmup, 3) * B):
        dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
    dpipe.join()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    nb = args.steps * B
    dump = OutputDump(torch, pool_dev[0], B) if args.dump_outputs and rank == 0 else None
    trk.profile_select(["warp", "erode55", "tophat55"])
    trk.profile_begin(min(nb, 400))                            # the first 400 batches of the region
    launches0 = lib.lt_launch_count()

    def region():
        nonlocal k
        for _ in range(nb - (B if dump else 0)):
            dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
        for j in range(B if dump else 0):                      # the last step, kept for --dump-outputs
            dump.submit(dpipe, pool_dev[k % P], j); k += 1
        dpipe.join()                                            # the launch stream waits for the last back half
    ms = timed(ctx, stream, region)
    launches = lib.lt_launch_count() - launches0
    morph_ms, morph_calls = trk.profile_read()
    res = dpipe.fetch_results(S)
    if dump:
        dump.write(args.dump_outputs)
        dump = None
    tracking = {"valid_fraction_last_batch": float(res["valid_lane_lines"].mean()),
                "band_search_fraction_last_batch": float((res["search_mode"] == 1).mean()),
                "two_attempt_fraction_last_batch": float((res["attempts"] == 2).mean())}

    # ---- stage breakdown: a separate, sequential, fully instrumented pass (an event at every stage boundary)
    trk.profile_select(None)
    prof_batches = min(nb, 50)
    trk.profile_begin(prof_batches)

    def seq():
        nonlocal k
        for _ in range(prof_batches):
            trk.process_async(pool_dev[k % P], out_ring[0]); k += 1
    ms_seq = timed(ctx, stream, seq) / prof_batches
    stage_ms, prof_calls = trk.profile_read()

    # ---- separately reported variant: fused single-resample remap (not bit-exact; stated mask-IoU tolerance)
    trk.set_remap_mode("fused")
    trk.reset()
    fpipe = DevicePipeline(trk)
    for i in range(3):
        fpipe.submit(pool_dev[i % P], out_ring[i & 1])
    fpipe.join()
    nbf = min(nb, 50)

    def fused():
        for i in range(nbf):
            fpipe.submit(pool_dev[i % P], out_ring[i & 1])
        fpipe.join()
    ms_fused = timed(ctx, stream, fused)
    fused_valid = float(fpipe.fetch_results(S)["valid_lane_lines"].mean())
    trk.set_remap_mode("exact")

    # ---- end to end (host buffers, copies inside the timed region)
    e2e_steps = max(1, min(args.steps, 10))
    e2e = e2e_runs(ctx, trk, host_batches, e2e_steps, B)
    clocks = sampler.stop() if rank == 0 else None
    nb_e2e = e2e_steps * B

    ms, ms_inpl, ms_full, ms_fused = ctx.max_over_ranks([ms, e2e["inplace"]["ms"], e2e["full"]["ms"], ms_fused])
    frames_total = world * S * nb
    value = frames_total / (ms * 1e-3)
    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        morph = {k_: morph_ms[k_] for k_ in ("erode55", "tophat55")}      # measured inside the timed region
        dom = max(morph, key=morph.get)
        dom_ms = morph[dom] / max(morph_calls, 1)
        achieved = S * MORPH_ALGO_BYTES_PER_FRAME / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        kname = "k_morph<55|29, %s>" % ("max, top-hat" if dom == "tophat55" else "min")
        traffic = None
        try:    # dram__bytes_read.sum + dram__bytes_write.sum of the stage's two kernels from the committed ncu --set full capture
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            traffic = tj["dram_bytes_per_stage"].get(dom)
            if traffic is not None:
                traffic = traffic * S / tj["streams"]
        except Exception:
            traffic = None
        rows_in = e2e["inplace"]["rows_in"][1] - e2e["inplace"]["rows_in"][0]
        rows_out = e2e["inplace"]["rows_out"][1] - e2e["inplace"]["rows_out"][0]
        rt = e2e["inplace"]["rows_text"]
        rows_text = (rt[1] - rt[0]) if rt[1] > rt[0] else 0
        res_bytes = trk._results_dev.numel()
        path_gbs = value * ALGO_BYTES_PER_FRAME / 1e9 / world
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "ms_per_batch": ms / nb, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world) if not photos_in_batch else mixed_config(world),
            "roofline": {"bound": "hbm", "kernel": "%s: the two concurrent ellipse kernels of the %s stage" % (kname, "dilation + top-hat" if dom == "tophat55" else "erosion"),
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "ms_per_launch": dom_ms,
                         "algorithmic_bytes_per_launch": S * MORPH_ALGO_BYTES_PER_FRAME,
                         "share_of_batch": dom_ms / (ms / nb),
                         "note": "the 55x55 (Lab-b) and 29x29 (R) kernels of a stage run concurrently on two streams and are "
                                 "timed together; the ellipse morphology is bound by the VIMNMX pipe and shared memory, not by "
                                 "HBM (DESIGN.md section 4); whole-path figure in roofline_path"},
            "roofline_path": {"bound": "hbm", "achieved": path_gbs, "peak": peak, "unit": "GB/s",
                              "frac": path_gbs / peak, "algorithmic_bytes_per_frame": ALGO_BYTES_PER_FRAME, "per_gpu": True},
            "stage_ms_per_batch": {k_: v / max(prof_calls, 1) for k_, v in stage_ms.items() if v > 0},
            "stage_pass": {"ms_per_batch": ms_seq, "batches": prof_batches,
                           "note": "separate sequential pass (one stream, an event at every stage boundary) after the "
                                   "timed region; the timed region itself overlaps consecutive batches"},
            "e2e": {"value": world * S * nb_e2e / (ms_inpl * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": S * (rows_in + rows_text) * 1280 * 3 * world * B,
                    "d2h_bytes_per_step": (S * (rows_out + rows_text) * 1280 * 3 + res_bytes) * world * B,
                    "ms_per_batch": ms_inpl / nb_e2e, "steps": e2e_steps,
                    "api": "HostPipeline(inplace=True): the caller's pinned frames are annotated in place; only the frame rows "
                           "the tracker reads go up and only the rows the overlay / text can change come back (the final host "
                           "image is identical to the full-frame form: tests/test_gpu_parity.py::test_inplace_annotation_and_roi_pipeline)"},
            "e2e_full": {"value": world * S * nb_e2e / (ms_full * 1e-3), "unit": "frames/s",
                         "h2d_bytes_per_step": S * FRAME_BYTES * world * B,
                         "d2h_bytes_per_step": (S * FRAME_BYTES + res_bytes) * world * B,
                         "ms_per_batch": ms_full / nb_e2e,
                         "api": "HostPipeline(overlay=True): every whole frame up, every whole annotated frame down"},
            "fused_remap_variant": {"value": world * S * nbf / (ms_fused * 1e-3), "unit": "frames/s",
                                    "ms_per_batch": ms_fused / nbf, "valid_fraction_last_batch": fused_valid,
                                    "tolerance": "not bit-exact: mask IoU vs the exact remap >= 0.6 per frame and >= 0.8 "
                                                 "mean on the 11 bundled frames (measured 0.886-0.946, mean 0.915; "
                                                 "tests/test_gpu_parity.py::test_fused_remap_variant)"},
            "gpu_launches": int(launches), "clocks": clocks, "tracking": tracking, "render_s": t_render,
        }
        line.update(parity if parity is not None else {"parity_checked": False})
        if cpu_line is not None:
            line["cpu_baseline"] = cpu_line
        print(json.dumps(line))
    trk.close()
    ctx.close()
    return 0


# ----------------------------------------------------------------------------------------------
# --config mixed: 11 of the 64 streams are the bundled photographs (two attempts + sliding-window search every frame)
# ----------------------------------------------------------------------------------------------

def load_photos():
    import cv2
    d = os.path.join(ROOT, "tests", "golden", "frames")
    return np.stack([cv2.cvtColor(cv2.imread(os.path.join(d, n)), cv2.COLOR_BGR2RGB) for n in sorted(os.listdir(d))
                     if n.endswith(".jpg")])


def mixed_config(n_gpus):
    c = workload_config(n_gpus)
    c["workload"] = ("64 streams per B200 of which 11 are the reference's bundled photographs (every frame invalid: both "
                     "attempts + sliding-window search) and 53 synthetic tracking streams")
    return c


# ----------------------------------------------------------------------------------------------
# --config single: BASELINE configs[1], one stream, 1000 sequential frames, per-frame state carry
# ----------------------------------------------------------------------------------------------

def _single_oracle(args):
    """Free-running oracle on the first n frames of the stream (forked before CUDA is initialised)."""
    n = args
    import warnings
    warnings.simplefilter("ignore")
    from lane_tracker_b200 import synth
    from oracle.tracker import OracleLaneTracker
    try:
        import cv2
        cv2.setNumThreads(max(1, host_cores()))
        backend = "cv2"
    except Exception:
        backend = "numpy"
    vid = synth.RoadVideo(0)
    trk = OracleLaneTracker(**synth.shipped_calibration(), backend=backend)
    recs = []
    for t in range(n):
        out = trk.process(vid.frame(t).copy())
        last = trk.trace["attempts"][-1]
        recs.append(dict(valid=bool(trk.valid_lane_lines), mode=last["mode"], out=sha(out),
                         left_fit=[float(v) for v in last.get("left_fit", [0, 0, 0])],
                         n_left=int(len(last["left_x"])) if last["detected"] else 0))
    return recs


def run_single(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    import multiprocessing as mp
    n_frames, n_check = args.frames, min(args.frames, args.check_frames)
    with mp.get_context("fork").Pool(1) as pool:
        want = pool.apply(_single_oracle, (n_check,)) if not args.no_cpu_baseline else []
    import torch
    from lane_tracker_b200 import BatchedLaneTracker, GraphedProcess, LaneTracker, synth
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cal = synth.shipped_calibration()
    vid = synth.RoadVideo(0)
    t0 = time.perf_counter()
    frames = np.stack([vid.frame(t) for t in range(min(n_frames, 200))])        # 200 distinct frames, cycled
    t_render = time.perf_counter() - t0

    # (a) the drop-in: LaneTracker.process(img) -> annotated frame, NumPy in / NumPy out, one call per frame
    lt = LaneTracker(**cal, device=local)
    first_div, checked = None, 0
    for t in range(n_check):                                    # free-running parity against the oracle
        out = lt.process(frames[t % len(frames)])
        w = want[t] if t < len(want) else None
        if w is None:
            break
        checked += 1
        ok = (lt.valid_lane_lines == w["valid"] and sha(out) == w["out"] and
              (not w["n_left"] or (len(lt.left_x) == w["n_left"] and np.allclose(lt.last_result["left_fit"], w["left_fit"], rtol=PARITY_RTOL, atol=0))))
        if not ok and first_div is None:
            first_div = t
    lt = LaneTracker(**cal, device=local)
    for t in range(5):
        lt.process(frames[t])
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for t in range(5, 5 + n_frames):
        lt.process(frames[t % len(frames)])
    torch.cuda.synchronize(dev)
    ms_dropin = 1e3 * (time.perf_counter() - t0) / n_frames
    valid_dropin = lt.get_success_ratio()[0]

    # (b) device-resident frames through the batched interface with one stream, results read by the host every frame;
    # (c) the same chain replayed as one CUDA graph per frame
    dframes = torch.from_numpy(frames).to(dev)
    out = torch.empty_like(dframes[:1])
    lat = {}
    for name in ("process", "graph"):
        bt = BatchedLaneTracker(1, **cal, device=local)
        g = GraphedProcess(bt, 1) if name == "graph" else None
        stream = torch.cuda.current_stream(dev)

        def one(t):
            if g is None:
                bt.process_async(dframes[t % len(frames)][None], out)
                return bt.fetch_results(1)
            g.frames.copy_(dframes[t % len(frames)][None], non_blocking=True)
            g.replay()
            return g.fetch_results()
        for t in range(5):
            one(t)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record(stream)
        ok = 0
        for t in range(5, 5 + n_frames):
            ok += int(one(t)["valid_lane_lines"][0])
        e1.record(stream)
        torch.cuda.synchronize(dev)
        lat[name] = dict(ms_per_frame=e0.elapsed_time(e1) / n_frames, valid_fraction=ok / n_frames)
        bt.close()
    best = min(v["ms_per_frame"] for v in lat.values())
    line = {
        "metric": "frames/sec, one 1280x720 stream, sequential frames with per-frame state carry", "value": 1e3 / best,
        "unit": "frames/s", "n_gpus": 1, "steps": n_frames, "warmup": 5, "ms_per_step": best, "higher_is_better": True,
        "scaling": "none", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "single-stream %d-frame synthetic 1280x720 video, band-search tracking with per-frame state "
                               "carry, 1 B200 (BASELINE.json configs[1])" % n_frames, "distinct_frames": int(len(frames))},
        "latency_ms_per_frame": {"dropin_LaneTracker.process_numpy_in_numpy_out": ms_dropin,
                                 "batched_process_device_frames_host_reads_result": lat["process"]["ms_per_frame"],
                                 "graphed_process_device_frames_host_reads_result": lat["graph"]["ms_per_frame"]},
        "valid_fraction": {"dropin": valid_dropin, "process": lat["process"]["valid_fraction"], "graph": lat["graph"]["valid_fraction"]},
        "parity_checked": bool(checked and first_div is None),
        "parity": {"free_running_frames_compared": checked, "first_divergence": first_div,
                   "compared": "validity, lane-pixel count, left fit (rtol 1e-6), sha256 of the annotated frame, every frame, "
                               "state never re-synchronised with the oracle"},
        "e2e": {"value": 1e3 / ms_dropin, "unit": "frames/s", "h2d_bytes_per_step": FRAME_BYTES, "d2h_bytes_per_step": FRAME_BYTES + 312},
        "render_s": t_render,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# --config 512: BASELINE configs[3], 512 streams in total sharded over the N GPUs (strong scaling), fits gathered to rank 0
# ----------------------------------------------------------------------------------------------

def run_512(args):
    ctx = Ctx(need_host_group=True)
    torch = ctx.torch
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, HostPipeline, sharding, synth
    from lane_tracker_b200.tracker import RESULT_DTYPE
    total = 512
    ids = sharding.stream_range(total, ctx.world, ctx.rank)
    S, P = len(ids), 2
    pool_dev, host_batches, t_render = render_pool(ctx, S, P, first_seed=ids[0])
    trk = BatchedLaneTracker(S, **synth.shipped_calibration(), device=ctx.local)
    stream = torch.cuda.current_stream(ctx.dev)
    out_ring = [torch.empty_like(pool_dev[0]) for _ in range(2)]
    rec = RESULT_DTYPE.itemsize
    gathered = torch.empty(total * rec, dtype=torch.uint8) if ctx.rank == 0 else None
    pinned = torch.empty(S * rec, dtype=torch.uint8).pin_memory()
    nb = args.steps
    seen = []
    copy_stream = torch.cuda.Stream(ctx.dev)

    def gather(res_dev):
        """Per batch: D2H of this rank's records, then ONE host-side gather on rank 0 (no device collective)."""
        with torch.cuda.stream(copy_stream):
            pinned.copy_(res_dev[:S * rec], non_blocking=True)
        copy_stream.synchronize()
        if ctx.distributed:
            allr = sharding.gather_records(pinned, total, group=ctx.host_group, out=gathered)
        else:
            allr = pinned
        if ctx.rank == 0:
            r = allr.numpy().view(RESULT_DTYPE)
            seen.append((int(r["counter"][0]), int(r["counter"][-1]), float(r["valid_lane_lines"].mean())))

    dpipe = DevicePipeline(trk)
    k = 0
    for _ in range(max(args.warmup, 3)):
        dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
    dpipe.join()

    def region():
        # batch j's records are gathered while batch j + 1 runs: its result buffer is not rewritten before batch j + 2
        nonlocal k
        prev = None
        for _ in range(nb):
            done = dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
            if prev is not None:
                prev[0].synchronize()
                gather(prev[1])
            prev = (done, dpipe.last_results_dev())
        prev[0].synchronize()
        gather(prev[1])
        dpipe.join()
    ms = timed(ctx, stream, region)
    # host-to-host: frames in pinned host memory, annotated in place, records gathered on rank 0 every batch
    trk.reset()
    hp = HostPipeline(trk, depth=3, inplace=True)
    src = [host_batches[i].clone().pin_memory() for i in range(P)]

    def consume(b):
        pinned.copy_(torch.from_numpy(b[1].view(np.uint8).reshape(-1)))
        if ctx.distributed:
            allr = sharding.gather_records(pinned, total, group=ctx.host_group, out=gathered)
        else:
            allr = pinned
        if ctx.rank == 0:
            seen.append((int(allr.numpy().view(RESULT_DTYPE)["counter"][0]), 0, 0.0))

    def run(n):
        for i in range(n):
            hp.submit(src[i % P])
            for b in hp.ready():
                consume(b)
        for b in hp.drain():
            consume(b)
    run(3)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(hp.s_in)
    run(nb)
    e1.record(hp.s_out)
    ctx.barrier()
    ms_e2e = e0.elapsed_time(e1)
    ms, ms_e2e = ctx.max_over_ranks([ms, ms_e2e])
    if ctx.rank == 0:
        rows_in = hp.rows_in[1] - hp.rows_in[0]
        rows_out = hp.rows_out[1] - hp.rows_out[0]
        line = {
            "metric": METRIC, "value": total * nb / (ms * 1e-3), "unit": "frames/s", "n_gpus": ctx.world, "steps": nb,
            "warmup": args.warmup, "ms_per_step": ms / nb, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "512 synthetic 1280x720 streams sharded across %d B200 (BASELINE.json configs[3]): %d streams "
                                   "per GPU, no data-path collective, the lt_result records of all 512 streams gathered to the "
                                   "host of rank 0 after every batch (gloo tensor gather of pinned records)" % (ctx.world, S),
                       "streams_total": total, "streams_per_gpu": S, "step": "one batch of all 512 streams"},
            "gather": {"records_per_batch": total, "bytes_per_batch": total * rec, "valid_fraction_last_batch": seen[nb - 1 + 0][2] if len(seen) >= nb else None},
            "e2e": {"value": total * nb / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e / nb,
                    "h2d_bytes_per_step": total * rows_in * 1280 * 3, "d2h_bytes_per_step": total * (rows_out * 1280 * 3 + rec),
                    "api": "HostPipeline(inplace=True) per rank + host gather of the records on rank 0"},
            "render_s": t_render,
        }
        print(json.dumps(line))
    trk.close()
    ctx.close()
    return 0


# ----------------------------------------------------------------------------------------------
# --config 1080p / 2160p: BASELINE configs[4], rescaled calibration, larger bird's-eye view (bandwidth stress)
# ----------------------------------------------------------------------------------------------

def run_scaled(args, scale, S):
    ctx = Ctx()
    torch = ctx.torch
    from lane_tracker_b200 import BatchedLaneTracker, DevicePipeline, synth
    cal = synth.shipped_calibration(scale)
    P = 2
    pool_dev, host_batches, t_render = render_pool(ctx, S, P, first_seed=ctx.rank * S, scale=scale)
    trk = BatchedLaneTracker(S, **cal, device=ctx.local)
    stream = torch.cuda.current_stream(ctx.dev)
    out_ring = [torch.empty_like(pool_dev[0]) for _ in range(2)]
    # the reference's pixel-valued constants do not scale (SURVEY 8d): every frame is invalid there; n_tries=1, as a
    # bandwidth stress of the per-frame kernels only
    from lane_tracker_b200.tracker import make_params
    params = make_params(n_tries=1)
    dpipe = DevicePipeline(trk, params=params)
    k = 0
    for _ in range(3):
        dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
    dpipe.join()
    nb = args.steps

    def region():
        nonlocal k
        for _ in range(nb):
            dpipe.submit(pool_dev[k % P], out_ring[k & 1]); k += 1
        dpipe.join()
    ms = timed(ctx, stream, region)
    trk.profile_select(None)
    trk.profile_begin(min(nb, 20))

    def seq():
        nonlocal k
        for _ in range(min(nb, 20)):
            trk.process_async(pool_dev[k % P], out_ring[0], params=params); k += 1
    timed(ctx, stream, seq)
    stage_ms, calls = trk.profile_read()
    (ms,) = ctx.max_over_ranks([ms])
    if ctx.rank == 0:
        w, h = cal["img_size"]
        bw, bh = cal["warped_size"]
        peak, peak_src = measured_peak_hbm()
        fps = ctx.world * S * nb / (ms * 1e-3)
        algo = 2 * w * h * 3 + 128
        line = {
            "metric": "frames/sec at %dx%d (batched streams)" % (w, h), "value": fps, "unit": "frames/s", "n_gpus": ctx.world,
            "steps": nb, "warmup": 3, "ms_per_step": ms / nb, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "%d synthetic %dx%d streams per B200 with rescaled warp/calibration matrices, bird's-eye view "
                                   "%dx%d (BASELINE.json configs[4]); n_tries=1 (the reference's pixel-valued constants do not "
                                   "scale, so every frame is invalid there: bandwidth stress only)" % (S, w, h, bw, bh),
                       "streams_per_gpu": S, "step": "one batch"},
            "roofline_path": {"bound": "hbm", "achieved": fps * algo / 1e9 / ctx.world, "peak": peak, "unit": "GB/s",
                              "frac": fps * algo / 1e9 / ctx.world / peak, "algorithmic_bytes_per_frame": algo, "peak_source": peak_src},
            "stage_ms_per_batch": {k_: v / max(calls, 1) for k_, v in stage_ms.items() if v > 0},
            "morph_bands": list(trk.morph_bands()), "render_s": t_render,
        }
        print(json.dumps(line))
    trk.close()
    ctx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="64", choices=["64", "single", "512", "1080p", "2160p", "mixed"])
    ap.add_argument("--frames", type=int, default=1000, help="--config single: frames in the sequence")
    ap.add_argument("--check-frames", type=int, default=64, help="--config single: frames compared free-running with the oracle")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--config 64|mixed: write the annotated frames (a fixed sample) and the result records of every "
                         "batch of the last timed step of rank 0 to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config not in ("64", "mixed")):
        ap.error("--dump-outputs applies to --impl ours with --config 64 or mixed")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.config == "single":
        return run_single(args)
    if args.config == "512":
        return run_512(args)
    if args.config == "1080p":
        return run_scaled(args, 1.5, 32)
    if args.config == "2160p":
        return run_scaled(args, 3.0, 8)
    return run_default(args, photos_in_batch=(args.config == "mixed"))


if __name__ == "__main__":
    sys.exit(main())
