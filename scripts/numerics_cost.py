#!/usr/bin/env python
"""What each numerics setting (crispy_ns_model_set_numerics) costs on the c2 workload: 1,024 streams x 60 s, f32 unit
scale, device-resident, one call per step.

For each of the six combinations of sum order (SEQUENTIAL, DOT4, DOT4_XCORR) and biquad form (f64 intermediates, F32)
one batch is created; the steps alternate between the batches (the order rotates every round), so that drift of the
card or of other work on the host spreads over all of them.  Whole-step times come from CUDA events around the call
with profiling off; per-kernel times from crispy_ns_batch_profile in a separate pass.  The card's name and power limit
are read in the same run.  Prints the record as one JSON line; --out / --md also write it as JSON and as a Markdown
table (profiles/r3_numerics.md is such a table).

    python scripts/numerics_cost.py --md OUT_DIR/r3_numerics.md
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = {0: "SEQUENTIAL", 1: "DOT4", 2: "DOT4_XCORR"}


def label(nm: int) -> str:
    return NAMES[nm & 3] + (" + BIQUAD_F32" if nm & 16 else "")


def card() -> dict:
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [s.strip() for s in q.split(",")]
    except (OSError, subprocess.SubprocessError, ValueError):
        info["power_limit"] = info["sm_max_clock"] = "not measured"
    return info


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--seconds", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the JSON record here")
    ap.add_argument("--md", default=None)
    args = ap.parse_args()

    import torch
    import crispy_b200 as cb
    from crispy_b200 import _lib
    from crispy_b200.synth import synth_chunk
    if not torch.cuda.is_available():
        raise SystemExit("numerics_cost.py measures on a CUDA device; none is present")

    combos = [s | b for b, s in itertools.product((0, _lib.BIQUAD_F32), (0, _lib.SUM_DOT4, _lib.SUM_DOT4_XCORR))]
    n, nf = args.streams, args.seconds * 100
    x = torch.cat([synth_chunk(n, min(100, nf - f) * 480, start_sample=f * 480, device="cuda") for f in range(0, nf, 100)], 1)
    out = torch.empty_like(x)
    vad = torch.empty((n, nf), dtype=torch.float32, device="cuda")
    dens = {}
    for nm in combos:
        m = cb.Model.synthetic(0)
        m.numerics = nm
        dens[nm] = cb.BatchDenoiser(n, m)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step(nm: int) -> float:
        den = dens[nm]
        den.reset()
        torch.cuda.synchronize()
        ev0.record()
        den.process_streams(x, unit_scale=True, out=out, vad=vad)
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    for nm in combos:  # warm-up: module load, first-touch of every workspace
        step(nm)
    times = {nm: [] for nm in combos}
    for r in range(args.rounds):
        for nm in combos[r % len(combos):] + combos[:r % len(combos)]:
            times[nm].append(step(nm))
    kernels = {}
    for nm in combos:  # per-kernel device time, in a pass of its own (events around every launch)
        den = dens[nm]
        den.profile(True)
        step(nm)
        kernels[nm] = {k: ms for k, (ms, _) in den.profile_read().items()}
        den.profile(False)

    stream_seconds = n * args.seconds
    base = statistics.median(times[0])
    rows = []
    for nm in combos:
        med = statistics.median(times[nm])
        rows.append({"numerics": nm, "label": label(nm), "step_ms_median": med, "step_ms_all": times[nm],
                     "stream_seconds_per_s": stream_seconds / (med / 1e3), "step_vs_default": med / base,
                     "kernel_ms": kernels[nm]})
    res = {"workload": f"{n} streams x {args.seconds} s, f32 unit scale, device-resident, one call per step",
           "rounds": args.rounds, **card(), "results": rows}
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)
    print(json.dumps(res))
    if args.md:
        ks = list(rows[0]["kernel_ms"])
        lines = [f"# Cost of the numerics settings on the c2 workload",
                 "",
                 f"Measured by `scripts/numerics_cost.py` on {res['gpu']}, power limit {res['power_limit']} "
                 f"(max SM clock {res['sm_max_clock']}).  Workload: {res['workload']}.  One batch per setting; the "
                 f"steps alternate between the six batches, {args.rounds} rounds, order rotated every round.  Step time: "
                 "CUDA events around the call, profiling off (median of the rounds).  Kernel times: summed device time "
                 "per kernel from `crispy_ns_batch_profile`, one profiled step per setting, in a separate pass; the seven "
                 "kernels overlap across chunks, so they do not add up to the step.",
                 "",
                 "| numerics | step ms (median) | all rounds, ms | stream-s / s | vs default | "
                 + " | ".join(k.replace("ns_", "").replace("_kernel", "") + " ms" for k in ks) + " |",
                 "|---|---|---|---|---|" + "---|" * len(ks)]
        for r in rows:
            lines.append(f"| {r['label']} | {r['step_ms_median']:.2f} | " + ", ".join(f"{t:.1f}" for t in r["step_ms_all"])
                         + f" | {r['stream_seconds_per_s'] / 1e3:.1f} K | {r['step_vs_default']:.3f} | "
                         + " | ".join(f"{r['kernel_ms'][k]:.1f}" for k in ks) + " |")
        open(args.md, "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
