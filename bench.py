#!/usr/bin/env python
"""bench.py - frames/s scored, ContentDetector @1080p (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps K --warmup W                  # this repo's CUDA path
    torchrun ... bench.py --gpus N ...                             # one rank per GPU, time shards + halo
    python bench.py --impl reference ...                           # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                         # + DIR/<name>.npy of the last timed step

A "step" is one pass of the hot path over the whole workload: `--frames` synthetic 1920x1080
BGR24 frames per GPU (default 10 000 = 62.2 GB, far larger than L2, so no flush is needed),
resident in HBM before the timed region.  One JSON line is printed by rank 0.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/sec scored (1080p, ContentDetector)"
UNIT = "frames/s"
DUMP_BYTES = 60 * 2**20  # --dump-outputs: larger outputs are written as a fixed, seeded sample of frames


def _positive_int(text: str) -> int:
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=10000, help="frames per GPU per step")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=None, help="steps for the host-buffer e2e leg")
    ap.add_argument("--host-ring", type=int, default=256, help="distinct pinned host frames for e2e")
    ap.add_argument("--cpu-sample", type=int, default=400, help="frames in the cpu_baseline sample")
    ap.add_argument("--edge-batch", type=int, default=2048,
                    help="frames per engine batch when the Canny/dilate edge component is on (its per-pixel "
                         "scratch - V plane, class map, union-find labels - is 6 B/px per frame of a batch)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--detector", default="content",
                    choices=["content", "content_edges", "adaptive", "threshold", "histogram", "hash"],
                    help="adaptive = BASELINE.json configs[2]: edge component + AdaptiveDetector(window_width=5)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --frames per GPU; strong: --frames in total, split into contiguous time shards")
    ap.add_argument("--parity-frames", type=int, default=None,
                    help="frames of the timed run re-scored with the oracle (default: the cpu sample, 48 with --no-cpu)")
    ap.add_argument("--ref-frames-per-proc", type=int, default=64, help="reference arm: frames per process per step")
    ap.add_argument("--resident-gb", type=float, default=150.0,
                    help="HBM budget for resident input per GPU; a larger shard cycles a resident ring of distinct frames")
    ap.add_argument("--sweep", action="store_true",
                    help="BASELINE.json configs[4]: one line per (size, total frames) cell, strong scaling over the ranks")
    ap.add_argument("--sweep-cells", default="640x360,1280x720,1920x1080,3840x2160:1000,10000,100000")
    ap.add_argument("--auto-downscale", action="store_true",
                    help="score at SceneManager's default auto-downscaled size (256 px wide) instead of full resolution")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the per-frame arrays the last timed step computed as DIR/<name>.npy (float32/float64; "
                         f"a seeded sample of frames above {DUMP_BYTES >> 20} MiB; _rank<r> suffix with several GPUs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.sweep or args.impl != "ours"):
        ap.error("--dump-outputs needs --impl ours and no --sweep")
    return args


def dump_outputs(path: str, arrays: dict, suffix: str = "") -> None:
    """Per-frame result arrays -> path/<name><suffix>.npy.  Above DUMP_BYTES, the same seeded sample of frames
    is kept from every array and its frame indices are written as frame_index<suffix>.npy."""
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(arrays.values())))
    per_frame = sum(a.nbytes // n for a in arrays.values())
    if per_frame * n > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (per_frame + 8), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["frame_index"] = keep.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}{suffix}.npy"), a)


# ------------------------------------------------------------------------------------------
# clocks / throttle sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines: list[tuple[float, str]] = []   # (arrival time, csv line)
        self.thread = None
        self.window: tuple[float, float] | None = None  # keep only samples that arrived inside it

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def collect(window):
            sm, smax, power, reasons = [], [], [], set()
            for stamp, line in self.lines:
                # nvidia-smi needs ~0.1 s to start, so the sampler is started before the warm-up steps
                # and the samples are cut to the timed region afterwards (25 ms period)
                if window is not None and not (window[0] <= stamp <= window[1]):
                    continue
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, smax, power, reasons

        sm, smax, power, reasons = collect(self.window)
        scope = "timed region"
        if not sm and self.window is not None:  # timed region shorter than one sample period
            sm, smax, power, reasons = collect(None)
            scope = "warm-up + timed region"
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)),
                "power_w_max": float(max(power)), "samples": len(sm), "scope": scope, "reasons": sorted(reasons)}


def measured_peak_gbs() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
# detector configuration per --detector
# ------------------------------------------------------------------------------------------
def detector_setup(kind: str):
    from pyscenedetect_b200.detectors import (AdaptiveDetector, ContentDetector, HashDetector, HistogramDetector,
                                              ThresholdDetector)
    from pyscenedetect_b200.engine import F_BGRSUM, F_EDGES, F_HASH, F_HSV, F_YHIST
    if kind == "hash":
        return F_HASH, (lambda: HashDetector()), "HashDetector() defaults: size 8, lowpass 2, threshold 0.35"
    if kind == "adaptive":
        return F_HSV | F_EDGES, (lambda: AdaptiveDetector(window_width=5, weights=ContentDetector.Components(1, 1, 1, 1))), \
            "AdaptiveDetector(window_width=5, weights=(1,1,1,1)) [edge component on]"
    if kind == "content":
        return F_HSV, (lambda: ContentDetector()), "ContentDetector() defaults: weights (1,1,1,0), threshold 27"
    if kind == "content_edges":
        return F_HSV | F_EDGES, (lambda: ContentDetector(weights=ContentDetector.Components(1, 1, 1, 1))), \
            "ContentDetector(weights=(1,1,1,1))"
    if kind == "threshold":
        return F_BGRSUM, (lambda: ThresholdDetector()), "ThresholdDetector()"
    return F_YHIST, (lambda: HistogramDetector(bins=256)), "HistogramDetector(bins=256)"


def ref_detector(kind: str):
    from oracle import ref_detectors as R
    if kind == "content":
        return R.RefContentDetector()
    if kind == "adaptive":
        return R.RefAdaptiveDetector(window_width=5, weights=(1.0, 1.0, 1.0, 1.0))
    if kind == "content_edges":
        return R.RefContentDetector(weights=(1.0, 1.0, 1.0, 1.0))
    if kind == "threshold":
        return R.RefThresholdDetector()
    if kind == "hash":
        return R.RefHashDetector()
    return R.RefHistogramDetector(bins=256)


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own cv2/numpy path (oracle port) on all host cores
# ------------------------------------------------------------------------------------------
def _ref_worker(idx, kind, first, count, w, h, seed, plan_frames, rounds, barrier, out_q):
    """One CPU worker = one contiguous time shard (+1 halo frame).  All workers of a round start
    together at `barrier`; the round ends when the slowest one is done."""
    import cv2
    cv2.setNumThreads(1)
    from pyscenedetect_b200.synth import ScenePlan, render_frames
    plan = ScenePlan(plan_frames, seed=seed)
    lo = max(0, first - 1)  # one-frame halo so the shard's first frame is scored like the serial run
    frames = render_frames(plan.params, w, h, first=lo, count=first + count - lo)
    times = []
    for _ in range(rounds):
        det = ref_detector(kind)
        barrier.wait()
        t0 = time.perf_counter()
        for i in range(frames.shape[0]):
            det.process_frame(lo + i, frames[i])
        times.append(time.perf_counter() - t0)
        barrier.wait()
    out_q.put((idx, times))


def _ref_run_pool(kind, n_proc, per_proc, w, h, seed, rounds):
    """-> list of per-round wall times (max over workers) for n_proc shards of per_proc frames."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(n_proc)
    q = ctx.SimpleQueue()
    procs = [ctx.Process(target=_ref_worker, args=(c, kind, c * per_proc, per_proc, w, h, seed,
                                                   n_proc * per_proc, rounds, barrier, q))
             for c in range(n_proc)]
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    return [max(t[r] for _i, t in res) for r in range(rounds)]


def run_reference(args):
    """Time shards over the host cores, one process per shard, cv2 single-threaded in each
    (BASELINE.md §3 variant ii).  A step is a bounded sample: `n_proc * per_proc` frames.
    The process count comes from a WARM probe (2 untimed + 1 timed round of 16 frames per process) over a few
    candidates; the timed steps then run >= 64 frames per process so that a step lasts seconds, not tenths."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_proc = max(8, int(args.ref_frames_per_proc))
    t0 = time.time()
    # The numpy temporaries of _mean_pixel_distance make this path memory/allocator bound, so
    # "all hardware threads" is not always the fastest process count: probe a few counts and keep the
    # best one for the timed steps (the CPU gets its best shot).
    candidates = sorted({max(1, cores // d) for d in (1, 2, 4)} | {min(cores, c) for c in (8, 12, 16, 24, 32, 48)}, reverse=True)
    probe = {}
    for p in candidates:
        rounds = _ref_run_pool(args.detector, p, 16, args.width, args.height, args.seed, 3)
        probe[p] = p * 16 / rounds[-1]
    n_proc = max(probe, key=probe.get)
    sample = n_proc * per_proc
    rounds = _ref_run_pool(args.detector, n_proc, per_proc, args.width, args.height, args.seed,
                           args.warmup + args.steps)
    step_times = rounds[args.warmup:]
    ms = 1000.0 * float(np.mean(step_times))
    value = sample / (ms / 1000.0)
    import cv2
    _feat, _mk, det_desc = None, None, {"content": "ContentDetector() defaults: weights (1,1,1,0), threshold 27",
                                        "content_edges": "ContentDetector(weights=(1,1,1,1))",
                                        "adaptive": "AdaptiveDetector(window_width=5, weights=(1,1,1,1)) [edge component on]",
                                        "threshold": "ThresholdDetector()",
                                        "histogram": "HistogramDetector(bins=256)"}[args.detector]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_text(det_desc, args.frames, args.width, args.height, args.seed,
                                             (args.width, args.height)),
                   "sample": f"bounded sample of {sample} frames per step ({per_proc} per process) of that sequence",
                   "parallelism": f"{n_proc} processes (best of {candidates} in a warm probe; host has {cores} hardware threads) "
                                  "x contiguous time shards with 1-frame halo, cv2.setNumThreads(1)",
                   "probe_frames_per_s": {str(k): round(v, 1) for k, v in probe.items()},
                   "step_frames_per_s": {"min": round(sample / max(step_times), 1),
                                         "median": round(sample / float(np.median(step_times)), 1),
                                         "max": round(sample / min(step_times), 1)}},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_proc, "kind": "port",
                         "sample": f"{sample} frames/step ({per_proc} per process) of the same synthetic sequence; "
                                   f"oracle.ref_detectors = the reference's cv2 {cv2.__version__}/numpy {np.__version__} calls"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


def workload_text(det_desc, frames_per_gpu, w, h, seed, scored) -> str:
    """Same wording in both arms (the driver compares the `config.workload` strings)."""
    return (f"{det_desc} on {frames_per_gpu} synthetic {w}x{h} BGR24 frames per GPU (BASELINE.json configs[1]), "
            f"seed {seed}, " + ("full resolution" if tuple(scored) == (w, h) else f"auto-downscaled on the device to {scored[0]}x{scored[1]}"))


def ncu_traffic_per_frame() -> tuple[float | None, str]:
    """dram bytes per 1080p frame of the fused HSV pass from the committed ncu summary (a citation, not a
    measurement of this run): newest profiles/r*_ncu_score_ws_kernel*.txt that holds the counters."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_score_ws_kernel*.txt")), reverse=True):
        try:
            text = open(path).read()
            rd = re.search(r"dram__bytes_read\.sum\s+(\w+)\s+([0-9.]+)", text)
            wr = re.search(r"dram__bytes_write\.sum\s+(\w+)\s+([0-9.]+)", text)
            fr = re.search(r"(\d+) frames 1920x1080", text)
            if not (rd and wr and fr):
                continue
            unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            total = float(rd.group(2)) * unit[rd.group(1)] + float(wr.group(2)) * unit[wr.group(1)]
            return total / int(fr.group(1)), os.path.relpath(path, ROOT)
        except (OSError, KeyError, ValueError):
            continue
    return None, "no ncu summary with dram counters under profiles/"


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from oracle import ref_detectors as R  # cpu_baseline leg only (the checker, never the product path)
    from pyscenedetect_b200 import _capi
    from pyscenedetect_b200.engine import Engine, PinnedBuffer, synth_frames_device
    from pyscenedetect_b200.scene_manager import SceneManager
    from pyscenedetect_b200.synth import ScenePlan
    from pyscenedetect_b200.video import ArrayVideoStream

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    dev = local
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    lib = _capi.load()

    W, H = args.width, args.height
    fbytes = W * H * 3
    features, make_det, det_desc = detector_setup(args.detector)
    if args.scaling == "strong":
        # fixed job: --frames in total, contiguous near-equal time shards (sharding.shard_bounds)
        from pyscenedetect_b200.sharding import shard_bounds
        total_frames = args.frames
        bounds = shard_bounds(total_frames, world)
        first, N = bounds[rank], bounds[rank + 1] - bounds[rank]
    else:
        N = args.frames
        total_frames = N * world
        first = rank * N
    plan = ScenePlan(total_frames, seed=args.seed)

    # ---- resident input: this rank's contiguous time range, generated on the device.  A shard larger than the
    #      HBM budget keeps a ring of its first R frames resident and walks it N / R times (the sequence is then
    #      periodic; bytes read from HBM per step are unchanged) ----
    R = N
    free_b, _tot_b = torch.cuda.mem_get_info(dev)
    budget = min(args.resident_gb * 1e9, 0.85 * free_b)
    if N * fbytes > budget:
        R = max(2, int(budget // fbytes))
    frames_t = torch.empty(R * fbytes, dtype=torch.uint8, device=f"cuda:{dev}")
    synth_frames_device(frames_t.data_ptr(), plan.params[first:first + R], W, H, device=dev)
    halo_t = torch.empty(fbytes, dtype=torch.uint8, device=f"cuda:{dev}") if world > 1 else None
    torch.cuda.synchronize()

    max_batch = 2048 if not (features & 8) else args.edge_batch
    sw, sh = W, H
    if args.auto_downscale:
        from pyscenedetect_b200.scene_manager import compute_downscale_factor
        f = compute_downscale_factor(max(W, H))
        sw, sh = (max(1, round(W / f)), max(1, round(H / f))) if f > 1.0 else (W, H)
        max_batch = min(max_batch, 1024)
    eng = Engine(W, H, features, width=sw, height=sh, device=dev, max_batch=max_batch,
                 **(make_det().engine_kwargs() if args.detector == "hash" else {}))
    weights = (1.0, 1.0, 1.0, 1.0 if args.detector in ("content_edges", "adaptive") else 0.0)
    sums_ptr = None
    n_scan = N
    d_val = torch.empty(N, dtype=torch.float64, device=f"cuda:{dev}")
    d_comp = torch.empty(N * 4, dtype=torch.float64, device=f"cuda:{dev}")
    d_flag = torch.empty(N, dtype=torch.uint8, device=f"cuda:{dev}")
    d_ratio = torch.empty(N, dtype=torch.float64, device=f"cuda:{dev}") if args.detector == "adaptive" else None
    wsum = float(sum(abs(x) for x in weights))
    import ctypes as C
    warr = (C.c_double * 4)(*weights)

    ext_stream = torch.cuda.ExternalStream(eng.compute_stream, device=f"cuda:{dev}")
    halo_ready = torch.cuda.Event()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        """Whole hot path for this rank's shard: halo exchange (N>1) -> fused score pass ->
        trailing device scan.  No host sync inside."""
        eng.reset()
        if world > 1:
            # ring shift of one frame over NCCL/NVLink: last frame -> rank+1, halo <- rank-1
            ops = []
            if rank + 1 < world:
                last = (N - 1) % R
                ops.append(dist.P2POp(dist.isend, frames_t[last * fbytes:(last + 1) * fbytes], rank + 1))
            if rank > 0:
                ops.append(dist.P2POp(dist.irecv, halo_t, rank - 1))
            if ops:
                for r in dist.batch_isend_irecv(ops):
                    r.wait()  # stream-level: torch's current stream waits for the NCCL transfer, the host does not
            if rank > 0:
                halo_ready.record(torch.cuda.current_stream())
                ext_stream.wait_event(halo_ready)  # the engine's compute stream picks the halo up when it has landed
                eng.set_halo_device(halo_t.data_ptr())
        done = 0
        while done < N:  # one submit unless the shard cycles a resident ring
            k = min(R - done % R, N - done)
            eng.submit_device(frames_t.data_ptr() + (done % R) * fbytes, k, fbytes)
            done += k
        sp, hp = eng.device_results()
        st = eng.compute_stream  # scans are ordered after the score kernel on the engine's stream
        if args.detector in ("content", "content_edges", "adaptive"):
            _capi.check(lib.psd_scan_content(sp, N, sw * sh, warr, wsum, d_comp.data_ptr(), d_val.data_ptr(), st))
            if args.detector == "adaptive":
                # the rolling adaptive window as a trailing device scan (adaptive_detector.py:100-143)
                _capi.check(lib.psd_scan_adaptive(d_val.data_ptr(), N, 5, 15.0, d_ratio.data_ptr(), st))
            else:
                _capi.check(lib.psd_scan_compare(d_val.data_ptr(), N, 27.0, 0, d_flag.data_ptr(), st))
        elif args.detector == "threshold":
            _capi.check(lib.psd_scan_average(sp, N, sw * sh * 3, d_val.data_ptr(), st))
        elif args.detector == "hash":
            # the halo frame's hash sits in the slot before stream frame 0, like the histograms
            hh = eng.device_hash()
            prev_hash = (hh - _capi.HASH_WORDS * 8) if (world > 1 and rank > 0) else None
            _capi.check(lib.psd_scan_hash_dist(hh, N, 8, prev_hash, d_val.data_ptr(), st))
        else:
            # the halo frame's histogram sits in the slot before stream frame 0 (psd_b200.h results layout)
            prev_hist = (hp - 256 * 4) if (world > 1 and rank > 0) else None
            _capi.check(lib.psd_scan_hist_correl(hp, N, 256, prev_hist, d_val.data_ptr(), st))

    def step_synced():
        one_step()
        eng.sync()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_synced()
    launches0 = lib.psd_launch_count()
    eng.timing_reset()
    barrier()
    t0 = time.perf_counter()
    ev_begin, ev_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_begin.record(ext_stream)  # CUDA events on the stream the kernels are launched on
    score_ms_total = 0.0
    score_launches = 0
    for _ in range(args.steps):
        eng.timing_reset()
        one_step()
        eng.sync()
        _tot, sc, nl = eng.timing_ms()
        score_ms_total += sc
        score_launches += nl
    ev_end.record(ext_stream)
    barrier()
    wall = time.perf_counter() - t0
    ev_ms_total = ev_begin.elapsed_time(ev_end)
    sampler.window = (t0, t0 + wall)
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.psd_launch_count() - launches0
    if args.dump_outputs:
        # what a caller of the timed path receives from its last step: the per-frame metric, and for the
        # content detectors the four components and the >= threshold flags (adaptive: the ratio instead)
        name = {"threshold": "average_rgb", "histogram": "hist_diff", "hash": "hash_dist"}.get(args.detector, "content_val")
        out = {name: d_val.cpu().numpy()}
        if args.detector in ("content", "content_edges", "adaptive"):
            out["components"] = d_comp.view(N, 4).cpu().numpy()
        if args.detector == "adaptive":
            out["adaptive_ratio"] = d_ratio.cpu().numpy()
        elif args.detector in ("content", "content_edges"):
            out["above_threshold"] = d_flag.cpu().numpy().astype(np.float32)
        dump_outputs(args.dump_outputs, out, f"_rank{rank}" if world > 1 else "")
    # device time per step (CUDA events on the engine's compute stream) and wall time; max over ranks
    t = torch.tensor([ev_ms_total / args.steps, 1000.0 * wall / args.steps], dtype=torch.float64, device=f"cuda:{dev}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ev_ms, wall_ms = float(t[0]), float(t[1])
    value = total_frames / (ev_ms / 1000.0)  # device-timed (CUDA events), max over ranks

    # correctness spot check of what was timed (rank 0): cuts == ground-truth cuts of the plan
    flags = d_flag.cpu().numpy() if args.detector.startswith("content") else None

    # ---- parity of what was timed: the device metric of this rank's first frames against the oracle, and at
    #      N > 1 the shard boundary (frame `first` scored against the neighbour's last frame = the halo) ----
    parity = None
    if args.parity_frames != 0:
        want_n = args.parity_frames if args.parity_frames else (48 if args.no_cpu else args.cpu_sample)
        n_par = max(2, min(want_n, N, R)) if rank == 0 else 1
        n_dl = n_par
        sample = np.empty((n_dl, H, W, 3), dtype=np.uint8)
        _capi.check(lib.psd_memcpy_d2h(dev, sample.ctypes.data, frames_t.data_ptr(), n_dl * fbytes))
        det = ref_detector(args.detector)
        if args.detector == "hash":
            det.with_stats = True   # hash_dist is only kept in the stats dict
        t_lo = first
        ds_factor = 1.0
        if (sw, sh) != (W, H):   # auto-downscale: the reference's SceneManager resizes before process_frame
            from pyscenedetect_b200.scene_manager import compute_downscale_factor
            ds_factor = compute_downscale_factor(max(W, H))
        from oracle import ref_detectors as RD   # (`R` is the resident-ring length in this function)
        scored = [RD.downscale_frame(sample[i], ds_factor) for i in range(n_dl)] if ds_factor > 1.0 else sample
        if rank > 0:
            halo_host = np.empty((H, W, 3), dtype=np.uint8)
            _capi.check(lib.psd_memcpy_d2h(dev, halo_host.ctypes.data, halo_t.data_ptr(), fbytes))
            halo_host = RD.downscale_frame(halo_host, ds_factor)
            det.process_frame(first - 1, halo_host)
        t_cpu0 = time.perf_counter()
        oracle_vals, oracle_cuts = [], []
        for i in range(n_dl):
            oracle_cuts += det.process_frame(t_lo + i, scored[i])
            if args.detector == "threshold":
                oracle_vals.append(float(np.mean(scored[i])))
            elif args.detector == "histogram":
                oracle_vals.append(None)
            elif args.detector == "hash":
                oracle_vals.append(float(det.metrics.get(t_lo + i, {}).get(det.metric_key, float("nan"))))
            else:
                oracle_vals.append(float(det._frame_score))
        cpu_dt = time.perf_counter() - t_cpu0
        dev_vals = d_val[:n_dl].cpu().numpy()
        if args.detector == "histogram":
            # cv2.compareHist on the oracle side; BASELINE tolerance 1e-4 (the device sums in a different order)
            h_det = ref_detector(args.detector)
            h_det.with_stats = True
            if rank > 0:
                h_det.process_frame(first - 1, halo_host)
            for i in range(n_dl):
                h_det.process_frame(t_lo + i, scored[i])
            pairs = [(h_det.metrics[t_lo + i][h_det.metric_key], dev_vals[i]) for i in range(n_dl) if (t_lo + i) in h_det.metrics]
            ok = all(abs(a - b) < 1e-4 for a, b in pairs)
            max_err = max([abs(a - b) for a, b in pairs], default=0.0)
        else:
            skip0 = 1 if (rank == 0 and args.detector != "threshold") else 0  # frame 0 has no predecessor: no score
            ok = all(float(dev_vals[i]) == oracle_vals[i] for i in range(skip0, n_dl))
            max_err = max([abs(float(dev_vals[i]) - oracle_vals[i]) for i in range(skip0, n_dl)], default=0.0)
        cuts_ok = None
        if rank == 0 and args.detector in ("content", "content_edges"):
            # FlashFilter over the device flags of the same frames == the oracle's cuts among them
            from oracle.ref_detectors import RefFlashFilter, _as_rate
            ff = RefFlashFilter(RefFlashFilter.MERGE, 15, _as_rate(30.0))
            dev_cuts = []
            for i in range(n_dl):
                dev_cuts += ff.filter(i, bool(flags[i]) and i > 0)
            cuts_ok = dev_cuts == oracle_cuts
        mine = torch.tensor([1.0 if ok else 0.0, max_err, 1.0 if cuts_ok in (None, True) else 0.0], dtype=torch.float64,
                            device=f"cuda:{dev}")
        allp = [torch.zeros_like(mine) for _ in range(world)] if world > 1 else [mine]
        if world > 1:
            dist.all_gather(allp, mine)
        if rank == 0:
            parity = {"frames": int(n_par), "bit_equal": bool(allp[0][0] > 0.5) if args.detector != "histogram" else None,
                      "within_1e-4": bool(allp[0][0] > 0.5), "max_abs_err": float(max(float(x[1]) for x in allp)),
                      "cuts_equal": (bool(allp[0][2] > 0.5) if cuts_ok is not None else None),
                      "metric": {"threshold": "average_rgb", "histogram": "hist_diff", "hash": "hash_dist"}.get(args.detector, "content_val"),
                      "oracle": "oracle.ref_detectors on the same frames (downloaded from HBM after the timed steps)"}
            if world > 1:
                parity["shard_boundaries_checked"] = world - 1
                parity["shard_boundaries_equal"] = all(bool(x[0] > 0.5) for x in allp[1:])
            parity["_cpu_fps"] = n_dl / cpu_dt if cpu_dt > 0 else None

    line = None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        sbytes = sw * sh * 3  # bytes of a frame as the fused pass sees it (smaller than fbytes when auto-downscaled)
        alg_bytes = sbytes * N * args.steps  # per-rank algorithmic bytes through the score kernel
        achieved = alg_bytes / (score_ms_total / 1000.0) / 1e9
        traffic_pf, traffic_src = ncu_traffic_per_frame()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ev_ms, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": workload_text(det_desc, args.frames if args.scaling == "weak" else f"{total_frames} (total, split over {world})",
                                          W, H, args.seed, (sw, sh)),
                "frames_per_gpu": N, "total_frames": total_frames,
                "parallelism": f"{world} contiguous time shards, 1-frame halo over NCCL p2p" if world > 1 else "single GPU",
                "l2": f"inputs are {N * fbytes / 1e9:.1f} GB per step per GPU, larger than L2 (126 MB): no flush needed"
                      + ("" if R == N else f"; {R} distinct frames ({R * fbytes / 1e9:.1f} GB) stay resident and are walked {N / R:.2f} times per step"),
                "timed_region": "halo exchange + fused score kernel + trailing device scan, inputs resident in HBM",
            },
            "wall_ms_per_step": wall_ms,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {
                "bound": "hbm", "kernel": ("psd_hash_rows_kernel + psd_hash_finish_kernel (gray, INTER_AREA, DCT, median)"
                                           if args.detector == "hash" else "psd_score_ws_kernel (fused TMA time-marching pass)"
                                           + ("" if (sw, sh) == (W, H) else f" on the {sw}x{sh} frames; the resize kernel that feeds it is outside this figure")),
                "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "algorithmic_bytes_per_frame": sbytes,
                "launches": int(score_launches), "avg_launch_ms": score_ms_total / max(1, score_launches),
                # dram__bytes_read+write of one `ncu --set full` capture of this kernel (a citation from the
                # committed summary, NOT measured in this run), scaled to the average launch of this run
                "traffic": (traffic_pf * (N * args.steps / max(1, score_launches)) / 1e9
                            if (traffic_pf and args.detector == "content" and (W, H) == (1920, 1080) and (sw, sh) == (W, H)) else None),
                "traffic_unit": f"GB per launch, cited from {traffic_src} (one ncu capture, scaled by frames per launch; not measured in this run)",
                "achieved_bytes_per_launch_gb": sbytes * N * args.steps / max(1, score_launches) / 1e9,
            },
        }
        if parity is not None:
            line["parity_check"] = {k: v for k, v in parity.items() if not k.startswith("_")}
        if flags is not None:
            line["config"]["frames_above_threshold"] = int(flags.sum())
        if world == 1 and args.detector == "content" and (sw, sh) == (W, H):
            # whole detection on the device (scores -> flags -> FlashFilter automaton) vs the plan's
            # ground-truth hard cuts; fades add extra cuts, so report both numbers
            from pyscenedetect_b200.device_cuts import DeviceCuts
            dev_cuts = DeviceCuts(eng).content(weights, 27.0, 15, 30.0)
            truth = set(plan.cut_frames)
            line["config"]["device_cut_list"] = {"cuts": len(dev_cuts), "ground_truth_hard_cuts": len(truth),
                                                 "hard_cuts_found": len(truth & set(dev_cuts))}

    # ---- e2e: same metric through the public API with HOST buffers (rank-local shard) ----
    if not args.no_e2e:
        from pyscenedetect_b200.engine import bind_host_to_gpu_numa_node
        orig_affinity = os.sched_getaffinity(0)
        numa = bind_host_to_gpu_numa_node(dev)  # page-locked frames on the GPU's own NUMA node
        ring = min(args.host_ring, N, R)
        pin = PinnedBuffer(ring * fbytes)
        _capi.check(lib.psd_memcpy_d2h(dev, pin.array.ctypes.data, frames_t.data_ptr(), ring * fbytes))
        host_frames = pin.array.reshape(ring, H, W, 3)
        e2e_steps = args.e2e_steps if args.e2e_steps is not None else args.steps
        repeat = (N + ring - 1) // ring

        def e2e_step_sharded():
            # N > 1: host frames -> halo over NCCL -> per-rank fused pass -> integer results gathered
            # on rank 0 -> device scans + cut state machines once (equals the serial run)
            from pyscenedetect_b200.sharding import TorchComm, detect_sharded
            comm = TorchComm(device=torch.device("cuda", dev))
            cuts, _sums = detect_sharded(host_frames, first, total_frames, make_det(), 30.0, comm,
                                         batch_size=64, n_local=N, pinned=True, device=dev, timings=e2e_phases)
            return N, (len(cuts) if cuts is not None else 0)

        def e2e_step_single():
            sm = SceneManager(device=dev, batch_size=64)
            sm.auto_downscale = False
            sm.downscale = 1
            sm.add_detector(make_det())
            n = sm.detect_scenes(ArrayVideoStream(host_frames, 30.0, pinned=True, repeat=repeat), duration=N)
            cuts = sm.get_cut_list()  # device->host read of the results happens inside detect_scenes
            return n, len(cuts)

        e2e_step = e2e_step_sharded if world > 1 else e2e_step_single
        e2e_phases: dict = {}

        for _ in range(min(args.warmup, 1)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            n_done, n_cuts = e2e_step()
        barrier()
        e2e_wall = (time.perf_counter() - t0) / e2e_steps
        t = torch.tensor([e2e_wall], dtype=torch.float64, device=f"cuda:{dev}")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            line["e2e"] = {
                "value": total_frames / float(t[0]), "unit": UNIT,
                "h2d_bytes_per_step": int(N * fbytes), "d2h_bytes_per_step": int(N * 5 * 8),
                "steps": e2e_steps, "ms_per_step": 1000.0 * float(t[0]),
                "api": ("SceneManager.detect_scenes(ArrayVideoStream(pinned host frames)) + get_cut_list()"
                        if world == 1 else "sharding.detect_sharded(pinned host frames, TorchComm(nccl))"),
                "host_frames": f"{ring} distinct page-locked frames cycled to {N} frames per step",
                "cuts_found": n_cuts,
                "host_numa": numa,
            }
            if e2e_phases:  # rank 0's last step: halo exchange, H2D + fused pass, result gather, scans + cut automata
                line["e2e"]["breakdown"] = {k.replace("_s", "_ms"): round(1000.0 * v, 2) for k, v in e2e_phases.items()}
        pin.close()
        os.sched_setaffinity(0, orig_affinity)

    # ---- cpu_baseline: oracle port (the reference's cv2/numpy calls) on the host cores, N=1 only ----
    if rank == 0 and world == 1 and not args.no_cpu:
        import cv2
        ns = min(args.cpu_sample, N, R)
        sample = np.empty((ns, H, W, 3), dtype=np.uint8)
        _capi.check(lib.psd_memcpy_d2h(dev, sample.ctypes.data, frames_t.data_ptr(), ns * fbytes))
        det = ref_detector(args.detector)
        for i in range(min(5, ns)):
            det.process_frame(i, sample[i])
        det = ref_detector(args.detector)
        t0 = time.perf_counter()
        for i in range(ns):
            det.process_frame(i, sample[i])
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {
            "value": ns / dt, "unit": UNIT, "cores": cv2.getNumThreads(), "kind": "port",
            "sample": f"first {ns} frames of the same workload, single process as shipped "
                      f"(cv2 {cv2.__version__} pool of {cv2.getNumThreads()} threads, numpy {np.__version__} single-threaded), "
                      f"host has {os.cpu_count()} logical cores",
            "ms_per_frame": 1000.0 * dt / ns,
        }
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    del frames_t, d_val, d_comp, d_flag
    torch.cuda.empty_cache()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.sweep:
        import copy
        sizes, totals = args.sweep_cells.split(":")
        for size in sizes.split(","):
            for total in totals.split(","):
                a = copy.copy(args)
                a.width, a.height = (int(v) for v in size.split("x"))
                a.frames, a.scaling = int(total), "strong"
                a.no_e2e = a.no_cpu = True
                a.steps, a.warmup = args.steps, args.warmup
                a.parity_frames = 8
                run_ours(a)
    else:
        run_ours(args)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
