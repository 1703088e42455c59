#!/usr/bin/env python
"""Continuous batching with per-stream calls (crispy_ns_process_streams_subset, crispy_ns_batch_reset_streams) against
padded batches, on one GPU.

1. Ragged queue: R recordings with lengths drawn log-uniform in [--min-minutes, --max-minutes] (seeded) go through
   --slots slots.
     A (padded, as crispy_ns_denoise_wav_files does): groups of --slots recordings in queue order, each group run to
       its longest recording in calls of --call-frames frames, the batch reset between groups.
     B (continuous): calls of --call-frames frames over every busy slot; a slot whose recording ends inside a call is
       padded to the call's end, reset (reset_streams) and refilled from the queue; when the queue is empty the
       remaining slots run as subset calls over the busy slots only.
   Useful stream-seconds (the recordings' own frames) per wall-second for both arms, their ratio, and the scheduled
   utilisation (useful frames / processed frames).  The input is one resident device block of synthetic audio
   (crispy_b200/synth.py) that every call reads from; its content does not change the work done.
2. Live ticks: --slots streams; each tick a seeded random --active fraction of them has one 10 ms frame, and one
   device-resident subset call with n_frames = 1 processes them.  Per-tick latency p50 / p99 from CUDA events (each
   tick starts on an idle GPU, as ticks 10 ms apart would), the host's wall time of the call, and the row-copy kernels'
   (gather + scatter) device time per tick from torch.profiler in a separate run.
3. Drain cost: the same --call-frames calls over all slots as full-batch calls and as subset calls listing every slot
   (the subset call adds the gather, the scatter and a drained pipeline at its end).

--dry-run computes the schedules only (no GPU): the processed / useful frame counts and the utilisation of both arms.
Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FRAMES_PER_S = 100  # 480-sample frames at 48 kHz


def recording_lengths(n: int, lo_min: float, hi_min: float, seed: int) -> np.ndarray:
    """frames per recording, log-uniform in [lo_min, hi_min] minutes"""
    rng = np.random.default_rng(seed)
    minutes = np.exp(rng.uniform(math.log(lo_min), math.log(hi_min), n))
    return np.maximum(1, np.rint(minutes * 60 * FRAMES_PER_S)).astype(np.int64)


def padded_schedule(lengths: np.ndarray, slots: int, call_frames: int):
    """arm A: [(n_streams, [n_frames of each call])] per group, processed and useful frames"""
    groups, processed = [], 0
    for g in range(0, len(lengths), slots):
        grp = lengths[g:g + slots]
        longest = int(grp.max())
        calls = [min(call_frames, longest - f) for f in range(0, longest, call_frames)]
        groups.append((len(grp), calls))
        processed += len(grp) * longest
    return groups, processed, int(lengths.sum())


def continuous_schedule(lengths: np.ndarray, slots: int, call_frames: int):
    """arm B: [(busy slot ids, or None when every slot is busy; slots to reset after the call)], processed and useful
    frames.  Every call runs call_frames frames; a recording ending inside a call is padded to the call's end."""
    queue = list(lengths[::-1])
    rem = np.zeros(slots, np.int64)
    for s in range(slots):
        if queue:
            rem[s] = queue.pop()
    calls, processed = [], 0
    while (rem > 0).any():
        busy = np.flatnonzero(rem > 0)
        processed += len(busy) * call_frames
        rem[busy] -= call_frames
        ended = busy[rem[busy] <= 0]
        refill = []
        for s in ended:
            rem[s] = 0
            if queue:
                rem[s] = queue.pop()
                refill.append(int(s))
        calls.append((None if len(busy) == slots else busy.tolist(), refill))
    return calls, processed, int(lengths.sum())


def gpu_info() -> dict:
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not measured"
    return info


def run_gpu(args, lengths) -> dict:
    import torch
    import crispy_b200 as cb
    from crispy_b200.synth import synth_chunk

    S, T = args.slots, args.call_frames
    block = synth_chunk(S, T * 480, device="cuda")  # resident input: every call reads these rows
    res = {}

    def timed(fn) -> float:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    # warm every shape both arms use
    den = cb.BatchDenoiser(S)
    den.process_streams(block)
    den.process_streams_subset(list(range(S // 2)), block[:S // 2])
    den.reset_streams([0])
    den.reset()

    # ---- 1. ragged queue
    groups, proc_a, useful = padded_schedule(lengths, S, T)

    def arm_a():
        for n, calls in groups:
            den.reset_async()
            for nf in calls:
                den.process_streams(block[:n, :nf * 480])
    t_a = timed(arm_a)

    calls, proc_b, _ = continuous_schedule(lengths, S, T)

    def arm_b():
        den.reset_async()
        for ids, refill in calls:
            if ids is None:
                den.process_streams(block)
            else:
                den.process_streams_subset(ids, block[:len(ids)])
            if refill:
                den.reset_streams(refill)
    t_b = timed(arm_b)
    useful_s = useful / FRAMES_PER_S
    res["ragged"] = {
        "recordings": len(lengths), "slots": S, "call_frames": T,
        "lengths": f"log-uniform {args.min_minutes}-{args.max_minutes} min, seed {args.seed}",
        "useful_stream_s": useful_s,
        "padded": {"wall_s": t_a, "stream_s_per_s": useful_s / t_a, "utilisation": useful / proc_a,
                   "calls": sum(len(c) for _, c in groups)},
        "continuous": {"wall_s": t_b, "stream_s_per_s": useful_s / t_b, "utilisation": useful / proc_b,
                       "calls": len(calls), "subset_calls": sum(ids is not None for ids, _ in calls)},
        "ratio_continuous_over_padded": t_a / t_b,
    }

    # ---- 2. live ticks
    rng = np.random.default_rng(args.seed + 1)
    m = int(round(args.active * S))
    ticks = [np.sort(rng.permutation(S)[:m]).tolist() for _ in range(args.ticks + args.warm)]
    frame = block[:m, :480].contiguous()
    live = cb.BatchDenoiser(S)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dev_ms, host_ms = [], []
    for i, ids in enumerate(ticks):
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        ev0.record()
        live.process_streams_subset(ids, frame)
        ev1.record()
        ev1.synchronize()
        h1 = time.perf_counter()
        if i >= args.warm:
            dev_ms.append(ev0.elapsed_time(ev1))
            host_ms.append((h1 - h0) * 1e3)
    from torch.profiler import ProfilerActivity, profile
    n_prof = min(200, args.ticks)
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for ids in ticks[:n_prof]:
            live.process_streams_subset(ids, frame)
        torch.cuda.synchronize()
    kernels = [e for e in prof.key_averages() if e.key.startswith("ns_")]
    rows_us = sum(e.device_time_total for e in kernels if e.key.startswith("ns_state_rows_kernel"))
    pipe_us = sum(e.device_time_total for e in kernels if not e.key.startswith("ns_state_rows_kernel"))
    row_bytes = 2784 * 4
    rows_us_tick = rows_us / n_prof
    res["live"] = {
        "streams": S, "active_per_tick": m, "ticks": args.ticks, "warmup_ticks": args.warm,
        "device_ms_p50": float(np.percentile(dev_ms, 50)), "device_ms_p99": float(np.percentile(dev_ms, 99)),
        "host_wall_ms_p50": float(np.percentile(host_ms, 50)), "host_wall_ms_p99": float(np.percentile(host_ms, 99)),
        "frame_period_ms": 10.0,
        "gather_scatter_us_per_tick": rows_us_tick,
        "pipeline_kernels_us_per_tick": pipe_us / n_prof,
        # gather + scatter each read and write m rows
        "gather_scatter_hbm_gb_s": (4 * m * row_bytes) / (rows_us_tick * 1e-6) / 1e9 if rows_us_tick else None,
    }

    # ---- 3. drain cost: the same calls over every slot, full-batch against a subset listing every slot
    every = list(range(S))
    n_calls = args.drain_calls
    full_s, sub_s = [], []
    for _ in range(3):  # alternating
        full_s.append(timed(lambda: [den.process_streams(block) for _ in range(n_calls)]))
        sub_s.append(timed(lambda: [den.process_streams_subset(every, block) for _ in range(n_calls)]))
    res["drain"] = {"calls": n_calls, "call_frames": T, "streams": S,
                    "full_ms_per_call": [t / n_calls * 1e3 for t in full_s],
                    "subset_all_ms_per_call": [t / n_calls * 1e3 for t in sub_s]}
    res.update(gpu_info())
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--recordings", type=int, default=4096)
    ap.add_argument("--slots", type=int, default=1024)
    ap.add_argument("--min-minutes", type=float, default=1.0)
    ap.add_argument("--max-minutes", type=float, default=20.0)
    ap.add_argument("--call-frames", type=int, default=1000, help="frames per call (1,000 = 10 s)")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--warm", type=int, default=200)
    ap.add_argument("--active", type=float, default=0.9)
    ap.add_argument("--drain-calls", type=int, default=10)
    ap.add_argument("--dry-run", action="store_true", help="schedules only, no GPU")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    lengths = recording_lengths(args.recordings, args.min_minutes, args.max_minutes, args.seed)
    if args.dry_run:
        _, proc_a, useful = padded_schedule(lengths, args.slots, args.call_frames)
        calls, proc_b, _ = continuous_schedule(lengths, args.slots, args.call_frames)
        res = {"dry_run": True, "recordings": args.recordings, "slots": args.slots, "call_frames": args.call_frames,
               "useful_frames": useful, "padded_processed_frames": proc_a, "continuous_processed_frames": proc_b,
               "padded_utilisation": useful / proc_a, "continuous_utilisation": useful / proc_b,
               "continuous_calls": len(calls), "continuous_subset_calls": sum(ids is not None for ids, _ in calls)}
    else:
        res = run_gpu(args, lengths)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
