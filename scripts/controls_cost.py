#!/usr/bin/env python
"""What the per-stream suppression controls (crispy_ns_batch_set_controls) cost on the c2 workload: 1,024 streams x
60 s, f32 unit scale, device-resident, one call per step.

Three arms: controls off on this tree, controls off on another tree (--parent-root: a checkout of the commit before the
controls with its library built, so that the default path can be compared with the code it replaced), and every stream
floored and gated on this tree.  Two builds of libcrispy_ns cannot share one process, so every measurement is a worker
process of its own, importing crispy_b200 from its arm's tree: it synthesises the input on the device, warms up with one step and times
--steps steps with CUDA events around the call, profiling off.  The workers of the three arms alternate, the order
rotating every round, so that drift of the card or of other work on the host spreads over all of them.  The card's name
and power limit are read in the same run.  Prints the record as one JSON line; --out / --md also write it as JSON and
as a Markdown table (profiles/r3_controls.md is such a table).

    python scripts/controls_cost.py --parent-root PARENT_CHECKOUT --md OUT_DIR/r3_controls.md
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ON = dict(min_gain=0.1, vad_threshold=0.5, hold_frames=20, gate_gain=0.1)  # every stream floored and gated


def worker(args) -> None:
    sys.path.insert(0, args.root)
    import torch
    import crispy_b200 as cb
    from crispy_b200.synth import synth_chunk
    if not torch.cuda.is_available():
        raise SystemExit("controls_cost.py measures on a CUDA device; none is present")
    n, nf = args.streams, args.seconds * 100
    x = torch.cat([synth_chunk(n, min(100, nf - f) * 480, start_sample=f * 480, device="cuda") for f in range(0, nf, 100)], 1)
    out = torch.empty_like(x)
    vad = torch.empty((n, nf), dtype=torch.float32, device="cuda")
    den = cb.BatchDenoiser(n, cb.Model.synthetic(0))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for i in range(args.steps + 1):  # step 0 warms up: module load, first touch of every workspace
        den.reset()
        if args.worker == "on":
            den.set_controls(range(n), **ON)
        torch.cuda.synchronize()
        ev0.record()
        den.process_streams(x, unit_scale=True, out=out, vad=vad)
        ev1.record()
        torch.cuda.synchronize()
        if i:
            times.append(ev0.elapsed_time(ev1))
    print(json.dumps({"step_ms": times}))


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
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=3, help="timed steps per worker")
    ap.add_argument("--parent-root", default=None, help="checkout of the commit before the controls, library built")
    ap.add_argument("--worker", choices=["off", "on"], default=None, help=argparse.SUPPRESS)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None, help="write the JSON record here")
    ap.add_argument("--md", default=None)
    args = ap.parse_args()
    if args.worker:
        return worker(args)

    arms = [("controls off", ROOT, "off"), ("controls off, parent tree", args.parent_root, "off"),
            ("every stream floored and gated", ROOT, "on")]
    arms = [a for a in arms if a[1]]
    times = {a[0]: [] for a in arms}
    for r in range(args.rounds):
        for name, root, mode in arms[r % len(arms):] + arms[:r % len(arms)]:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", mode, "--root", os.path.abspath(root),
                                "--streams", str(args.streams), "--seconds", str(args.seconds), "--steps", str(args.steps)],
                               capture_output=True, text=True,
                               env={k: v for k, v in os.environ.items() if k != "CRISPY_NS_LIB"})  # each tree's own build
            if p.returncode != 0:
                raise SystemExit(f"worker {name} failed ({p.returncode}):\n{p.stderr[-3000:]}")
            times[name] += json.loads(p.stdout.strip().splitlines()[-1])["step_ms"]
    stream_seconds = args.streams * args.seconds
    base = statistics.median(times[arms[0][0]])
    rows = [{"arm": a[0], "step_ms_median": statistics.median(times[a[0]]), "step_ms_all": times[a[0]],
             "stream_seconds_per_s": stream_seconds / (statistics.median(times[a[0]]) / 1e3),
             "step_vs_controls_off": statistics.median(times[a[0]]) / base} for a in arms]
    res = {"workload": f"{args.streams} streams x {args.seconds} s, f32 unit scale, device-resident, one call per step",
           "controls_on": ON, "rounds": args.rounds, "steps_per_worker": args.steps, **card(), "results": rows}
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)
    print(json.dumps(res))
    if args.md:
        lines = ["# Cost of the per-stream suppression controls on the c2 workload", "",
                 f"Measured by `scripts/controls_cost.py` on {res['gpu']}, power limit {res['power_limit']} (max SM clock "
                 f"{res['sm_max_clock']}).  Workload: {res['workload']}.  Controls on: {ON} on every stream.  Each worker "
                 f"process warms up with one step and times {args.steps}; the arms' workers alternate, {args.rounds} rounds, "
                 "order rotated every round.  Step time: CUDA events around the call, profiling off.", "",
                 "| arm | step ms (median) | all steps, ms | stream-s / s | vs controls off |", "|---|---|---|---|---|"]
        for r in rows:
            lines.append(f"| {r['arm']} | {r['step_ms_median']:.2f} | " + ", ".join(f"{t:.1f}" for t in r["step_ms_all"])
                         + f" | {r['stream_seconds_per_s'] / 1e3:.1f} K | {r['step_vs_controls_off']:.3f} |")
        open(args.md, "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
