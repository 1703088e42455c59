#!/usr/bin/env python
"""bench.py -- stream-seconds of 48 kHz audio denoised per wall-second (BASELINE.json metric).

  python bench.py [--gpus N --steps K --warmup W]           our arm: libcrispy_ns.so on N B200s
  python bench.py --impl reference [...]                    reference arm: the CPU implementation
                                                            (oracle port of nnnoiseless 0.5.2; the
                                                            crate itself cannot be built offline)
  python bench.py [...] --dump-outputs DIR                  also write the last timed step's outputs (a seeded
                                                            sample of frames) as DIR/<name>.npy

A "step" is one pass of the whole denoise path over one batch: configs[1] of BASELINE.json --
1,024 independent 60 s 48 kHz mono streams per GPU (6.144 M frames), synthetic speech+noise.
  value : device-resident throughput (inputs already in HBM), CUDA events, max over ranks
  e2e   : same metric through the public host API (BatchDenoiser.process_streams_host): pinned
          host buffers, H2D + kernel + D2H inside the timed region
Streams are independent, so N GPUs each take their own 1,024 streams (weak scaling, no collective
on the data path; torch.distributed is used only for the timing barrier / max).
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
sys.path.insert(0, ROOT)

FRAME = 480
ALG_BYTES_PER_FRAME = 3844          # SURVEY.md 8(d): 480*4 read + 480*4 written + 4 (VAD)
RNN_FLOPS_PER_FRAME = 175006        # SURVEY.md 8(d): 2 * 87,503 MAC
ALL_FLOPS_PER_FRAME = 390000        # SURVEY.md 8(a) whole-pipeline estimate
PITCH_MACS_PER_FRAME = 75000        # K1: multiply-adds per frame that must stay unfused (DESIGN.md section 2)
FP32_PEAK_TFLOPS_NOMINAL = 74.5     # 148 SM * 128 lanes * 2 * 1.965 GHz (not in MEASURED_PEAKS.json)
# the recurrent core (K4) runs on the tensor pipe: 723 bf16 m16n8k16 tiles per 16-stream step, twice (hi + lo plane)
RNN_MMA_FLOPS_PER_FRAME = 2 * 723 * (16 * 8 * 16 * 2) // 16   # executed flops per (stream, frame), padding included
# frames per array --dump-outputs writes: 8,192 x (960 + 1) x 4 B = 31.5 MB for the widest step (c4's stereo mix + VAD)
DUMP_FRAMES = 8192


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=1024, help="streams per GPU")
    ap.add_argument("--seconds", type=float, default=60.0, help="audio seconds per stream per step")
    ap.add_argument("--e2e-seconds", type=float, default=None, help="override the e2e leg's length")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-front-end", action="store_true")
    ap.add_argument("--parity-streams", type=int, default=4)
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"],
                    help="c2 = BASELINE.json configs[1] (default, the headline); c3 = configs[2]: 1,024 streams x 60 s per GPU at "
                         "44.1 kHz through the sinc front end, then denoised; c4 = configs[3]: 4,096 dual-source meetings "
                         "x 10 min, mic PCM16 + app f32 -> dual-mono PCM16; c5 = configs[4]: 8,192 streams x 60 min; both "
                         "partitioned by stream over the N ranks, synthesised on device chunk by chunk, state carried")
    ap.add_argument("--total-streams", type=int, default=None, help="c4/c5: streams (meetings) in the whole job")
    ap.add_argument("--minutes", type=float, default=None, help="c4/c5: recording length (default 10 / 60)")
    ap.add_argument("--chunk-seconds", type=int, default=10, help="c4/c5: audio seconds per call")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what rank 0's last timed step returned (the denoised audio and "
                         "the VAD; c3-c5: of the step's last call) as DIR/<name>.npy, float32, sampled to "
                         f"{DUMP_FRAMES} frames by a fixed seed, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none to write")
    return args


def dump_outputs(dump_dir: str, n_frames: int, arrays: dict) -> None:
    """Writes each [streams, frames x k] output as DIR/<name>.npy, float32 [DUMP_FRAMES, k] (k = 1 is squeezed): the
    frames at the same (stream, frame) pairs, drawn without replacement by numpy's default_rng(0) and sorted, in every
    array and every run."""
    import numpy as np
    import torch
    n_streams = next(iter(arrays.values())).shape[0]
    total = n_streams * n_frames
    pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(total, min(DUMP_FRAMES, total), replace=False)))
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        s, f = (pick // n_frames).to(a.device), (pick % n_frames).to(a.device)
        sample = a.reshape(n_streams, n_frames, -1)[s, f].squeeze(-1)
        np.save(os.path.join(dump_dir, name + ".npy"), sample.float().cpu().numpy())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """dense bf16 TFLOP/s, sustained figure (the kernel is timed inside a long step)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d.get("bf16_tflops_sustained") or d["bf16_tflops"]), "measured sustained (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------------------
class CpuArm:
    """The CPU implementation of the path on all host cores: the oracle port (oracle/rnnoise_oracle.c, the in-repo C
    restatement of nnnoiseless 0.5.2 -- the crate itself cannot be built offline), -O3 -march=native, one DenoiseState
    per stream, pthreads over streams.  The synthetic sample (full-length streams of the same workload) is generated
    ONCE; every step() denoises it again from fresh states."""

    def __init__(self, seconds_per_stream: float, target_step_s: float):
        import numpy as np
        import torch
        from crispy_b200.synth import synth_chunk
        from oracle import pyoracle as po
        self.po, self.np = po, np
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)  # torchrun exports OMP_NUM_THREADS=1: the generator would crawl
        po.build_native()
        self.model = po.Model.synthetic(0)
        # calibrate: one second of audio per thread, on one thread and on all of them
        cal = synth_chunk(self.cores, 48000).numpy()
        po.process_streams(self.model, cal[:1, :4800], unit_scale=True, n_threads=1, native=True)  # tables, page faults
        t0 = time.perf_counter()
        po.process_streams(self.model, cal[:1], unit_scale=True, n_threads=1, native=True)
        self.x_realtime_one_thread = 1.0 / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        po.process_streams(self.model, cal, unit_scale=True, n_threads=self.cores, native=True)
        rate = self.cores / (time.perf_counter() - t0)
        # whole streams of the workload's own length, as many as fit the step budget (a multiple of the thread count)
        self.secs = int(seconds_per_stream) if seconds_per_stream >= 1 else 1
        n = int(target_step_s * rate / self.secs)
        n = max(self.cores, min(1024, n // self.cores * self.cores))
        self.n_streams = n
        t0 = time.perf_counter()
        self.x = np.empty((n, 48000 * self.secs), np.float32)
        for f0 in range(0, self.secs, 10):  # 10 s pieces keep the generator's f64 temporaries small
            nf = min(10, self.secs - f0)
            self.x[:, f0 * 48000:(f0 + nf) * 48000] = synth_chunk(n, nf * 48000, start_sample=f0 * 48000).numpy()
        self.gen_s = time.perf_counter() - t0

    def step(self) -> float:
        """one pass over the sample; returns the wall seconds it took"""
        t0 = time.perf_counter()
        self.po.process_streams(self.model, self.x, unit_scale=True, n_threads=self.cores, native=True)
        return time.perf_counter() - t0

    def describe(self, value: float, wall_s: float) -> dict:
        return {"value": value, "unit": "stream-seconds/s", "cores": self.cores, "kind": "port", "wall_s": wall_s,
                "x_realtime_per_thread_all_threads_busy": value / self.cores,
                "x_realtime_one_thread_alone": self.x_realtime_one_thread,
                "sample": f"{self.n_streams} streams x {self.secs} s of the same synthetic workload (generated once, "
                          f"{self.gen_s:.1f} s, untimed), {self.cores} pthreads over streams, oracle C port "
                          f"(-O3 -march=native: the RNN's sums run one vector lane per neuron, the coarse pitch "
                          f"search eight lags per vector, Stockham FFT) of nnnoiseless 0.5.2; {wall_s:.2f} s wall per pass. "
                          f"RNNoise's paper quotes ~60x real time on one x86 core"}


def cpu_reference_rate(target_seconds: float = 10.0, seconds_per_stream: float = 60.0):
    arm = CpuArm(seconds_per_stream, target_seconds)
    dt = arm.step()
    return arm.describe(arm.n_streams * arm.secs / dt, dt)


def run_reference(args):
    """bench.py --impl reference: rank 0 alone runs the CPU arm (the other ranks exit at once); the whole run is
    sized to end within ~90 s at any K: one calibration, one generated sample, W <= 1 warm-up pass, K timed passes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    arm = CpuArm(args.seconds, max(3.0, min(12.0, 50.0 / (steps + min(args.warmup, 1)))))
    for _ in range(max(0, min(args.warmup, 1))):
        arm.step()
    walls = [arm.step() for _ in range(steps)]
    wall = sum(walls) / len(walls)
    v = arm.n_streams * arm.secs / wall
    line = {
        "impl": "reference", "metric": "stream-seconds of 48 kHz audio denoised per wall-second",
        "value": v, "unit": "stream-seconds/s", "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
        "ms_per_step": 1e3 * wall,  # one step = one pass over the bounded sample (cpu_baseline.sample)
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{args.streams} independent {args.seconds:g} s 48 kHz mono streams per GPU "
                               f"(BASELINE.json configs[1]); the CPU arm times a bounded sample of it: "
                               f"{arm.n_streams} of those streams at full length per step",
                   "same_config": False,
                   "ranks": "rank 0 alone runs the CPU arm with every host thread; a rate, so it does not depend on N",
                   "note": "nnnoiseless itself cannot be built offline (no Rust toolchain, crate not vendored): "
                           "this is the in-repo C restatement, all host cores"},
        "cpu_baseline": arm.describe(v, wall),
        "e2e": {"value": v, "unit": "stream-seconds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import crispy_b200 as cb
    from crispy_b200.synth import synth_chunk

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = []
    if world > 1:  # one process per GPU: keep this rank's pinned host buffers on the GPU's own NUMA node
        from crispy_b200.shard import bind_to_gpu_numa_node
        try:
            pr = torch.cuda.get_device_properties(local)  # CUDA's own enumeration, not NVML's
            numa_cpus = bind_to_gpu_numa_node(f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0")
        except Exception:
            numa_cpus = []
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL only carries the timing barrier / max here; whatever it prints goes to stderr with the rest (main())
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    n_streams = args.streams
    n_frames = int(round(args.seconds * 100))
    first_stream = rank * n_streams  # global stream ids: each GPU denoises its own recordings

    # ---- synthetic input, resident in HBM ------------------------------------------------------
    x = torch.empty((n_streams, n_frames * FRAME), dtype=torch.float32, device=dev)
    chunk = 100  # frames per generation chunk
    for f0 in range(0, n_frames, chunk):
        nf = min(chunk, n_frames - f0)
        x[:, f0 * FRAME:(f0 + nf) * FRAME] = synth_chunk(n_streams, nf * FRAME, first_stream=first_stream,
                                                         start_sample=f0 * FRAME, device=dev)
    out = torch.empty_like(x)
    vad = torch.empty((n_streams, n_frames), dtype=torch.float32, device=dev)
    den = cb.BatchDenoiser(n_streams, device=local)
    info0 = den.info
    fp32 = cb.measure_fp32(local) if rank == 0 else None  # FFMA burst + unfused MAC burst on every SM, ~50 ms

    def step():
        den.reset_async()
        den.process_streams(x, unit_scale=True, out=out, vad=vad)

    # ---- part of the cpu_baseline leg (the one place this arm runs the oracle, as the checker and never inside a
    # timed region): the GPU output of a few streams' first 2 s against the CPU port's (rank 0) ----
    parity = None
    if rank == 0 and args.parity_streams > 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as po
        ns_p, nf_p = min(args.parity_streams, n_streams), min(200, n_frames)
        step()
        torch.cuda.synchronize(dev)
        got = out[:ns_p, :nf_p * FRAME].cpu().numpy()
        gv = vad[:ns_p, :nf_p].cpu().numpy()
        ref, rv = po.process_streams(po.Model.synthetic(0), x[:ns_p, :nf_p * FRAME].cpu().numpy(), unit_scale=True)
        err = got.astype(np.float64) - ref
        parity = {"streams": ns_p, "frames": nf_p, "max_abs_fs": float(np.abs(err).max()),
                  "snr_db": float(10 * np.log10((ref.astype(np.float64) ** 2).mean() / max((err ** 2).mean(), 1e-30))),
                  "vad_max": float(np.abs(gv - rv).max())}
        # SURVEY 8(d): the share of frames the silence gate closes (they still ride through K4, which is batched over
        # 16 streams; RNNoise's gate is E < 0.04 in 16-bit scale, i.e. digital silence: the synthetic streams carry
        # noise through their pauses, so it stays at or near 0 here)
        try:
            den_t = cb.BatchDenoiser(ns_p, device=local)
            _, _, taps_t = den_t.process_streams(x[:ns_p, :nf_p * FRAME], unit_scale=True, return_taps=True)
            parity["silent_fraction"] = float((taps_t[:, :, 133] != 0).float().mean().item())
            del den_t, taps_t
        except Exception as e:  # a reporting extra: never take the bench line down
            parity["silent_fraction"] = None
            parity["silent_fraction_error"] = repr(e)[:200]

    # ---- device-resident timing -----------------------------------------------------------------
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = den.info["launches"]
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for e0, e1 in evs:
        e0.record()
        step()
        e1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = evs[0][0].elapsed_time(evs[-1][1])
    launches = den.info["launches"] - launches0
    if rank == 0 and args.dump_outputs:  # before the profiled step and the serial leg below write into out / vad
        dump_outputs(args.dump_outputs, n_frames, {"out": out, "vad": vad})
    # per-kernel launch durations: one more step of the same workload, OUTSIDE the timed region, with every launch
    # bracketed by CUDA events on the (internal) stream it is launched on; the pipeline runs exactly as above
    # (seven kernels of neighbouring chunks overlap), so these are in-pipeline durations
    den.profile(True)
    step()
    kernel_prof = den.profile_read()
    den.profile(False)
    prof_steps = 1
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    stream_seconds_per_step = world * n_streams * n_frames / 100.0
    value = stream_seconds_per_step * args.steps / (total_ms_max / 1e3)

    # ---- end to end through the host API --------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        import psutil
        e2e_frames = n_frames if args.e2e_seconds is None else int(round(args.e2e_seconds * 100))
        need = 2 * n_streams * e2e_frames * FRAME * 4
        avail = psutil.virtual_memory().available / max(1, world)
        while need > 0.35 * avail and e2e_frames > 100:
            e2e_frames //= 2
            need = 2 * n_streams * e2e_frames * FRAME * 4
        hx = torch.empty((n_streams, e2e_frames * FRAME), dtype=torch.float32).pin_memory()
        hx.copy_(x[:, :e2e_frames * FRAME])
        hout = torch.empty_like(hx).pin_memory()
        hvad = torch.empty((n_streams, e2e_frames), dtype=torch.float32).pin_memory()

        def e2e_step():
            den.reset_async()
            den.process_streams_host(hx, unit_scale=True, out=hout, vad=hvad)

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": world * n_streams * e2e_frames / 100.0 * args.steps / dt, "unit": "stream-seconds/s",
               "h2d_bytes_per_step": n_streams * e2e_frames * FRAME * 4,
               "d2h_bytes_per_step": n_streams * e2e_frames * (FRAME * 4 + 4),
               "seconds_per_stream": e2e_frames / 100.0,
               "api": "BatchDenoiser.process_streams_host -> crispy_ns_process_streams_host (pinned host buffers)",
               "rank0_cpus_bound": len(numa_cpus)}
        if rank == 0:
            e2e["matches_device_path"] = bool(torch.equal(hout[:4], out[:4, :e2e_frames * FRAME].cpu()))
        # the same leg with PCM16 on the link (CRISPY_NS_IN_I16 | CRISPY_NS_OUT_I16: what the recorder stores,
        # recording.rs:101-121): half the bytes per stream-second, so the PCIe ceiling doubles.  Reported beside
        # the f32 figure, not instead of it.
        del hout  # keep the pinned footprint below the f32 leg's
        hx16 = torch.empty((n_streams, e2e_frames * FRAME), dtype=torch.int16).pin_memory()
        hx16.copy_((x[:, :e2e_frames * FRAME] * 32767.0).round().clamp_(-32768, 32767).to(torch.int16))
        del hx
        hout16 = torch.empty_like(hx16).pin_memory()

        def e2e16_step():
            den.reset_async()
            den.process_streams_host(hx16, unit_scale=True, out=hout16, vad=hvad, out_i16=True)

        e2e16_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e16_step()
        barrier()
        dt16 = time.perf_counter() - t0
        tt = torch.tensor([dt16], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e["pcm16_link"] = {"value": world * n_streams * e2e_frames / 100.0 * args.steps / float(tt.item()),
                             "unit": "stream-seconds/s", "h2d_bytes_per_step": n_streams * e2e_frames * FRAME * 2,
                             "d2h_bytes_per_step": n_streams * e2e_frames * (FRAME * 2 + 4),
                             "api": "the same call with CRISPY_NS_IN_I16 | CRISPY_NS_OUT_I16 (PCM16 on the host link, "
                                    "what the recorder stores: recording.rs:101-121)"}
        del hx16, hout16

    # ---- the same kernels one at a time (one stream): isolated durations, comparable with the ncu
    # launch list under profiles/ (inside the timed region above they overlap 7 deep and share SMs) ----
    kernels_isolated = None
    if rank == 0:
        os.environ["CRISPY_NS_SERIAL"] = "1"
        try:
            den_s = cb.BatchDenoiser(n_streams, device=local)
        finally:
            del os.environ["CRISPY_NS_SERIAL"]
        nf_s = min(n_frames, 8 * info0["chunk_frames"])
        den_s.process_streams(x[:, :nf_s * FRAME], unit_scale=True, out=out[:, :nf_s * FRAME], vad=vad[:, :nf_s])
        torch.cuda.synchronize(dev)
        den_s.reset()
        den_s.profile(True)
        den_s.process_streams(x[:, :nf_s * FRAME], unit_scale=True, out=out[:, :nf_s * FRAME], vad=vad[:, :nf_s])
        prof_s = den_s.profile_read()
        den_s.profile(False)
        tot_s = sum(ms for ms, _ in prof_s.values()) or 1.0
        kernels_isolated = {"frames_per_stream": nf_s, "note": "CRISPY_NS_SERIAL=1: all kernels on one stream",
                            "kernels": [{"kernel": k, "launches": n, "avg_launch_us": ms / max(n, 1) * 1e3,
                                         "share_of_kernel_time": ms / tot_s} for k, (ms, n) in prof_s.items()]}
        del den_s

    # ---- configs[2] front ends, timed alone (rank 0): 44.1 -> 48 kHz over n_streams x 10 s ----------
    front_end = None
    if rank == 0 and not args.no_front_end:
        fe_secs = 10
        x44 = torch.zeros((n_streams, 44100 * fe_secs), dtype=torch.float32, device=dev)
        n_cp = min(x.shape[1], x44.shape[1])
        x44[:, :n_cp].copy_(x[:, :n_cp])  # any signal will do: the kernels are data-independent
        front_end = {"input": f"{n_streams} streams x {fe_secs} s at 44.1 kHz -> 48 kHz, device-resident, kernel alone"}
        for name, fn, flops in (("sinc256", lambda: cb.sinc_resample(x44, 44100, 48000), 2 * 256),
                                ("linear", lambda: cb.linear_resample(x44, 44100.0, 48000.0), 3),
                                ("resample_audio", lambda: cb.resample_audio(x44, 44100, 48000), 3)):
            for _ in range(3):
                y48 = fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for _ in range(reps):
                y48 = fn()
            e1.record()
            torch.cuda.synchronize(dev)
            sec = e0.elapsed_time(e1) / 1e3 / reps
            n_out = y48.shape[1]
            front_end[name] = {"ms_per_launch": sec * 1e3, "stream_seconds_per_s": n_streams * fe_secs / sec,
                               "hbm_algorithmic_gbs": n_streams * (x44.shape[1] + n_out) * 4 / sec / 1e9,
                               "fp32_tflops": n_streams * n_out * flops / sec / 1e12}
        # the capture callbacks' downmix (audio.rs:754-755 / :816-818): stereo in, mono out -- the one kernel of the
        # library that IS bound by HBM (12 / 8 bytes per frame, one add and one divide)
        for name, dt, bpf in (("downmix_stereo_f32", torch.float32, 12), ("downmix_stereo_i16", torch.int16, 8)):
            n_fr = 48000 * fe_secs
            st2 = torch.zeros((n_streams, 2 * n_fr), dtype=dt, device=dev)
            for _ in range(3):
                mono = cb.downmix_mono(st2, 2)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            e0.record()
            for _ in range(reps):
                mono = cb.downmix_mono(st2, 2)
            e1.record()
            torch.cuda.synchronize(dev)
            sec = e0.elapsed_time(e1) / 1e3 / reps
            front_end[name] = {"ms_per_launch": sec * 1e3, "stream_seconds_per_s": n_streams * fe_secs / sec,
                               "hbm_algorithmic_gbs": n_streams * n_fr * bpf / sec / 1e9,
                               "frac_hbm": n_streams * n_fr * bpf / sec / 1e9 / measured_peaks()[0],
                               "bytes_per_launch": n_streams * n_fr * bpf,
                               "note": "peak = the driver's copy-measured HBM figure (1 read : 1 write); this kernel reads 2 bytes "
                                       "for every byte it writes, so it can sit above that figure and below the 7.7 TB/s nominal"}
            del st2, mono
        front_end["sinc256"]["frac_fp32_measured"] = front_end["sinc256"]["fp32_tflops"] / fp32["ffma_tflops"]
        front_end["linear"]["frac_hbm"] = front_end["linear"]["hbm_algorithmic_gbs"] / measured_peaks()[0]
        front_end["resample_audio"]["frac_hbm"] = front_end["resample_audio"]["hbm_algorithmic_gbs"] / measured_peaks()[0]
        del y48
        # ---- the other BASELINE.json configs on the same streams, 10 s each, device-resident (rank 0) ----
        def timed(fn, reps=2):
            fn()
            torch.cuda.synchronize(dev)
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b_.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b_) / 1e3 / reps

        nf10 = min(n_frames, fe_secs * 100)

        def c3():
            den.reset_async()
            den.process_streams(x44[:, :441 * nf10], unit_scale=True, input_rate=44100, front_end="sinc")

        xi16 = (x[:, :nf10 * FRAME] * 32767.0).round().clamp(-32768, 32767).to(torch.int16)
        app = torch.roll(x[:, :nf10 * FRAME], 1, 0) * 0.5
        mix = torch.empty((n_streams, nf10 * FRAME, 2), dtype=torch.int16, device=dev)

        def c4():
            den.reset_async()
            den.process_streams(xi16, unit_scale=True, app=app, mix_stereo_i16=True, out=mix)

        front_end["configs"] = {
            "c3_441k_sinc_then_denoise": {"stream_seconds_per_s": n_streams * nf10 / 100.0 / timed(c3),
                                          "what": "configs[2]: 44.1 kHz f32 in -> sinc256 -> denoise -> 48 kHz f32 out"},
            "c4_mic_i16_plus_app_to_stereo_pcm16": {"stream_seconds_per_s": n_streams * nf10 / 100.0 / timed(c4),
                                                    "what": "configs[3] per meeting: mic PCM16 denoised + raw app f32, "
                                                            "clamp(mic+app) -> dual-mono stereo PCM16 (counts meetings)"},
        }
        del x44, xi16, app, mix

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline: per kernel, from the CUDA events taken inside the timed region -----------------
    hbm_peak, peak_src = measured_peaks()
    chunk_frames = info0["chunk_frames"]
    traffic_tab = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic_tab = json.load(open(tp))
        except Exception:
            traffic_tab = {}
    sum_ms = sum(ms for ms, _ in kernel_prof.values()) or 1.0
    kernels = []
    for name, (ms, n) in kernel_prof.items():
        if n == 0:
            continue
        frames_per_launch = n_streams * n_frames * prof_steps / n  # (stream, frame) units one launch processes
        avg_s = ms / n / 1e3
        ent = {"kernel": name, "launches": n, "ms_total": ms, "share_of_kernel_time": ms / sum_ms,
               "avg_launch_us": avg_s * 1e6, "frames_per_launch": frames_per_launch,
               "hbm_algorithmic_gbs": ALG_BYTES_PER_FRAME * frames_per_launch / avg_s / 1e9}
        if name == "ns_rnn_kernel":
            tpeak, tsrc = measured_tensor_peak()
            ent["tensor"] = {"bound": "tensor (latency: 8 dependent products per frame step)",
                             "algorithmic_tflops": RNN_FLOPS_PER_FRAME * frames_per_launch / avg_s / 1e12,
                             "executed_tflops_bf16_hi_lo": RNN_MMA_FLOPS_PER_FRAME * frames_per_launch / avg_s / 1e12,
                             "peak": tpeak, "unit": "TFLOP/s", "peak_source": tsrc}
            ent["tensor"]["frac"] = ent["tensor"]["algorithmic_tflops"] / tpeak
        tr = traffic_tab.get(name)
        if tr and tr.get("streams") == n_streams:
            ent["dram_bytes_per_launch_ncu"] = tr["dram_bytes_per_launch"] * frames_per_launch / tr["frames_per_launch"]
            # what actually limits the kernel (ncu --set full of one isolated launch, profiles/): per cent of peak
            ent["ncu_limiters_pct"] = {k: tr[k] for k in ("issue_active_pct", "smem_wavefronts_pct_of_peak", "fma_pipe_pct",
                                                          "tensor_pipe_pct", "dram_throughput_pct") if tr.get(k) == tr.get(k) and tr.get(k) is not None}
        kernels.append(ent)
    kernels.sort(key=lambda e: -e["ms_total"])
    # The dominant kernel is the one that takes the most SM-time, not the one whose launches last longest: the serial
    # kernels (biquad, recurrent core: one lane or one CTA per group of streams) cover a fraction of the 148 SMs and
    # stretch while they share them with the parallel kernels of the neighbouring chunks.  SM-time = summed launch time
    # x the fraction of the SMs the kernel's grid covers.
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    grid_ctas = {"ns_highpass_kernel": -(-n_streams // 32), "ns_pitchscan_kernel": -(-n_streams // 4),
                 "ns_features_kernel": -(-n_streams // 4), "ns_rnn_kernel": -(-n_streams // info0["rnn_streams_per_cta"])}
    for ent in kernels:
        ent["sm_fraction"] = min(1.0, grid_ctas.get(ent["kernel"], n_sms) / n_sms)
        ent["sm_time_ms"] = ent["ms_total"] * ent["sm_fraction"]
    tot_sm_time = sum(e["sm_time_ms"] for e in kernels) or 1.0
    for ent in kernels:
        ent["share_of_sm_time"] = ent["sm_time_ms"] / tot_sm_time
    dom = max(kernels, key=lambda e: e["sm_time_ms"])
    roofline = {"bound": "hbm", "achieved": dom["hbm_algorithmic_gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": dom["hbm_algorithmic_gbs"] / hbm_peak, "traffic": dom.get("dram_bytes_per_launch_ncu"),
                "peak_source": peak_src, "kernel": dom["kernel"],
                "algorithmic_bytes_per_launch": ALG_BYTES_PER_FRAME * dom["frames_per_launch"],
                "avg_launch_us": dom["avg_launch_us"], "ncu_limiters_pct": dom.get("ncu_limiters_pct"),
                "traffic_source": "profiles/traffic.json: dram bytes and limiter percentages of one `ncu --set full` launch of "
                                  "this kernel at this batch size (profiles/r2_ncu_full.md), scaled to this run's frames per "
                                  "launch; achieved / avg_launch_us are measured live in this run",
                "note": "algorithmic bytes = 3,844 B per (stream, frame) (480 f32 in + 480 f32 out + VAD) x the frames "
                        "one launch covers / that kernel's mean launch time (CUDA events on its own stream, inside the "
                        "timed region, kernels of neighbouring chunks running concurrently). The kernel named is the one "
                        "with the largest share of SM-time (kernels[].share_of_sm_time). No kernel of this path "
                        "is HBM-bound: they are issue/latency bound (profiles/)."}
    roofline_fp32 = {"whole_pipeline_tflops": ALL_FLOPS_PER_FRAME * n_streams * n_frames * args.steps / (total_ms / 1e3) / 1e12,
                     "peak_tflops_measured_ffma_burst": fp32["ffma_tflops"],
                     "unfused_tmacs_measured": fp32["unfused_tmacs"],
                     "peak_tflops_nominal": FP32_PEAK_TFLOPS_NOMINAL,
                     "how": "crispy_ns_measure_fp32: register-resident FFMA chains (fused) and FMUL+FADD chains (the "
                            "unfused multiply-add the pitch kernel's exactness contract requires) on every SM, best of 3"}
    roofline_fp32["frac_whole_pipeline"] = roofline_fp32["whole_pipeline_tflops"] / fp32["ffma_tflops"]
    # K1's own roofline: ~75 K unfused MACs per frame (coarse 35.3 K + candidates <= 28 K + fine 4.8 K + autocorr 4.3 K
    # + downsample / FIR / energies ~3 K) against the measured unfused-MAC rate
    for ent in kernels:
        if ent["kernel"] == "ns_pitch_kernel":
            ent["fp32_unfused"] = {"macs_per_frame": PITCH_MACS_PER_FRAME,
                                   "achieved_tmacs": PITCH_MACS_PER_FRAME * ent["frames_per_launch"] / (ent["avg_launch_us"] * 1e-6) / 1e12,
                                   "peak_tmacs": fp32["unfused_tmacs"]}
            ent["fp32_unfused"]["frac"] = ent["fp32_unfused"]["achieved_tmacs"] / fp32["unfused_tmacs"]

    # ---- north_star: "each phase reported at a stated fraction of its roofline" -------------------------------
    # analysis = K0 + K1 + K2 + K3 + K3b, recurrent = K4, synthesis = K5.  A phase's cost per chunk is its share of the
    # SM-time x the pipeline's period (the kernels of neighbouring chunks overlap, so in-pipeline launch times do not
    # add up to the period; the SM-time shares do).  HBM roofline for analysis and synthesis (algorithmic bytes:
    # analysis reads the 480 f32 of a frame, synthesis writes them + VAD); tensor and FP32 rooflines for the
    # recurrent phase (175,006 algorithmic flop per frame).
    phases = None
    try:
        by = {e["kernel"]: e for e in kernels}
        tpeak, tsrc = measured_tensor_peak()

        fpl = dom["frames_per_launch"]
        period_us = total_ms_max / args.steps * 1e3 / (dom["launches"] / prof_steps)  # one chunk leaves the pipeline every ...

        def sm_us(names):  # the phase's share of the SM-time x the pipeline's period: the shares sum to the period
            return sum(by[k]["share_of_sm_time"] for k in names if k in by) * period_us

        ana = ("ns_highpass_kernel", "ns_highpass_par_kernel", "ns_pitch_kernel", "ns_pitchscan_kernel",
               "ns_spectrum_kernel", "ns_features_kernel")
        t_ana, t_rnn, t_syn = sm_us(ana), sm_us(("ns_rnn_kernel", "ns_rnn_tc5_kernel")), sm_us(("ns_synthesis_kernel",))
        t_all = (t_ana + t_rnn + t_syn) or 1.0
        phases = {
            "how": "the kernels of neighbouring chunks run concurrently, so a phase's cost per chunk is its share of the "
                   "SM-time (in-pipeline launch time x fraction of the 148 SMs its grid covers, kernels[].share_of_sm_time) "
                   "x the pipeline's period (one chunk every period_us); the three add up to the period; achieved = "
                   "algorithmic bytes or flops of one chunk / that time",
            "frames_per_chunk": fpl, "period_us": period_us,
            "analysis": {"kernels": [k for k in ana if k in by], "gpu_time_us_per_chunk": t_ana, "share": t_ana / t_all,
                         "bound": "hbm", "algorithmic_bytes_per_frame": 1920,
                         "achieved_gbs": 1920 * fpl / (t_ana * 1e-6) / 1e9 if t_ana else None,
                         "frac": 1920 * fpl / (t_ana * 1e-6) / 1e9 / hbm_peak if t_ana else None,
                         "limited_by": "issue slots and shared-memory wavefronts (K1 60 % / 64 %, K3 60 % / 58 %), "
                                       "DRAM 2-16 % busy: profiles/r2_ncu_full.md"},
            "recurrent": {"kernels": [k for k in ("ns_rnn_kernel", "ns_rnn_tc5_kernel") if k in by],
                          "gpu_time_us_per_chunk": t_rnn, "share": t_rnn / t_all, "bound": "tensor",
                          "algorithmic_flops_per_frame": RNN_FLOPS_PER_FRAME,
                          "achieved_tflops": RNN_FLOPS_PER_FRAME * fpl / (t_rnn * 1e-6) / 1e12 if t_rnn else None,
                          "frac_of_tensor_peak": RNN_FLOPS_PER_FRAME * fpl / (t_rnn * 1e-6) / 1e12 / tpeak if t_rnn else None,
                          "frac_of_measured_fp32_peak": RNN_FLOPS_PER_FRAME * fpl / (t_rnn * 1e-6) / 1e12 / fp32["ffma_tflops"] if t_rnn else None,
                          "tensor_peak_source": tsrc,
                          "limited_by": "latency of 8 dependent matrix products per frame step, serial in time "
                                        "(HMMA pipe 13 % busy): profiles/r2_k4_tcgen05.md"},
            "synthesis": {"kernels": ["ns_synthesis_kernel"], "gpu_time_us_per_chunk": t_syn, "share": t_syn / t_all,
                          "bound": "hbm", "algorithmic_bytes_per_frame": 1924,
                          "achieved_gbs": 1924 * fpl / (t_syn * 1e-6) / 1e9 if t_syn else None,
                          "frac": 1924 * fpl / (t_syn * 1e-6) / 1e9 / hbm_peak if t_syn else None,
                          "limited_by": "issue slots 59 %, shared-memory wavefronts 54 %, DRAM 23 % busy"},
        }
    except Exception as e:  # a reporting extra: never take the bench line down
        phases = {"error": repr(e)[:200]}

    cpu_baseline = None
    if not args.no_cpu_baseline:
        cpu_baseline = cpu_reference_rate(target_seconds=8.0, seconds_per_stream=args.seconds)

    line = {
        "metric": "stream-seconds of 48 kHz audio denoised per wall-second",
        "value": value, "unit": "stream-seconds/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{n_streams} independent {args.seconds:g} s 48 kHz mono streams per GPU "
                               "(BASELINE.json configs[1]), f32 unit-scale in/out + VAD",
                   "streams_per_gpu": n_streams, "frames_per_stream": n_frames, "parallelism": f"streams/{world}gpu",
                   "chunk_frames": info0["chunk_frames"], "rnn_streams_per_cta": info0["rnn_streams_per_cta"],
                   "l2": f"inputs {x.numel() * 4 / 1e9:.1f} GB + outputs {x.numel() * 4 / 1e9:.1f} GB per step >> 126 MB L2 "
                         "(no flush needed)",
                   "weights": "synthetic seed 0 (nnnoiseless weights are not available offline)"},
        "clocks": clocks, "e2e": e2e, "e2e_pcm16": (e2e or {}).get("pcm16_link"), "gpu_launches": int(launches),
        "roofline": roofline, "kernels": kernels, "kernels_isolated": kernels_isolated, "roofline_fp32": roofline_fp32,
        "phases": phases, "front_end": front_end,
        "cpu_baseline": cpu_baseline,
        "parity_vs_oracle": parity, "wall_s_timed_region": t_wall,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# the long configs at their real size: configs[3] (c4) and configs[4] (c5)
# --------------------------------------------------------------------------------------------------
def run_long(args):
    """c4: 4,096 dual-source meetings x 10 min -- mic PCM16 denoised + raw app f32 -> clamp(mic + app) as dual-mono
    stereo PCM16 (commands/recording.rs:260-264, recording.rs:101-121); counts meetings.  c5: 8,192 streams x 60 min,
    f32 in/out.  Both are partitioned by stream over the N ranks (contiguous blocks, no collective), fed as calls of
    --chunk-seconds of audio with every DenoiseState carried from call to call, the input of each call synthesised on
    the device just before it (the recordings do not fit HBM: SURVEY.md 8(d)).  Only the denoise calls are timed:
    one CUDA event pair per call on the launching stream, summed; max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import crispy_b200 as cb
    from crispy_b200.shard import stream_block
    from crispy_b200.synth import synth_chunk

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    c4 = args.config == "c4"
    c3 = args.config == "c3"
    total_streams = args.total_streams or (4096 if c4 else (1024 * world if c3 else 8192))
    minutes = args.minutes or (10.0 if c4 else (1.0 if c3 else 60.0))
    first, last = stream_block(total_streams, world, rank)
    n = last - first
    if c3:
        args.chunk_seconds = int(round(minutes * 60.0))  # the resamplers keep no state across calls: a whole recording per call
    call_frames = args.chunk_seconds * 100
    n_calls = max(1, int(round(minutes * 60.0 / args.chunk_seconds)))
    den = cb.BatchDenoiser(n, device=local)
    S = call_frames * FRAME
    in_frame = 441 if c3 else FRAME  # input samples per 10 ms
    if c3:
        mic = torch.empty((n, call_frames * in_frame), dtype=torch.float32, device=dev)
        app = None
        out = None
    elif c4:
        mic = torch.empty((n, S), dtype=torch.int16, device=dev)
        app = torch.empty((n, S), dtype=torch.float32, device=dev)
        out = torch.empty((n, S, 2), dtype=torch.int16, device=dev)
    else:
        mic = torch.empty((n, S), dtype=torch.float32, device=dev)
        app = None
        out = torch.empty((n, S), dtype=torch.float32, device=dev)
    vad = torch.empty((n, call_frames), dtype=torch.float32, device=dev)

    def synth(call: int):
        for f0 in range(0, call_frames, 100):
            nf = min(100, call_frames - f0)
            x = synth_chunk(n, nf * FRAME, first_stream=first, start_sample=(call * call_frames + f0) * FRAME, device=dev)
            if c3:  # the same generator read as a 44.1 kHz signal: 441 samples per 10 ms
                mic[:, f0 * 441:(f0 + nf) * 441] = x[:, :nf * 441]
            elif c4:
                mic[:, f0 * FRAME:(f0 + nf) * FRAME] = (x * 32767.0).round().clamp_(-32768, 32767).to(torch.int16)
                app[:, f0 * FRAME:(f0 + nf) * FRAME] = torch.roll(x, 1, 0) * 0.5  # another meeting's voice as app audio
            else:
                mic[:, f0 * FRAME:(f0 + nf) * FRAME] = x

    last_out = [None]

    def call():
        if c3:
            last_out[0] = den.process_streams(mic, unit_scale=True, vad=vad, input_rate=44100, front_end="sinc")[0]
        elif c4:
            den.process_streams(mic, unit_scale=True, app=app, mix_stereo_i16=True, out=out, vad=vad)
        else:
            den.process_streams(mic, unit_scale=True, out=out, vad=vad)

    synth(0)
    parity = None
    if rank == 0 and args.parity_streams > 0 and not args.no_cpu_baseline:  # checker leg: first call, a few streams
        from oracle import pyoracle as po
        k = min(args.parity_streams, n)
        call()
        torch.cuda.synchronize(dev)
        xin = (mic[:k].float() / 32768.0 if c4 else mic[:k]).cpu().numpy()
        if c3:
            xin = np.stack([po.sinc_resample(xin[i], 44100, 48000)[:call_frames * FRAME] for i in range(k)])
        ref, rv = po.process_streams(po.Model.synthetic(0), xin, unit_scale=True, n_threads=k, native=True)
        if c3:
            err = last_out[0][:k].cpu().numpy().astype(np.float64) - ref
            parity = {"streams": k, "frames": call_frames, "max_abs_fs": float(np.abs(err).max()),
                      "vad_max": float(np.abs(vad[:k].cpu().numpy() - rv).max())}
        elif c4:
            want = np.stack([po.mix_dual_mono_i16(ref[i], app[i].cpu().numpy()).reshape(-1, 2) for i in range(k)])
            d = np.abs(out[:k].cpu().numpy().astype(np.int32) - want.astype(np.int32))
            parity = {"streams": k, "frames": call_frames, "max_abs_lsb": int(d.max()), "vad_max": float(np.abs(vad[:k].cpu().numpy() - rv).max())}
        else:
            err = out[:k].cpu().numpy().astype(np.float64) - ref
            parity = {"streams": k, "frames": call_frames, "max_abs_fs": float(np.abs(err).max()),
                      "vad_max": float(np.abs(vad[:k].cpu().numpy() - rv).max())}
    for _ in range(max(3, args.warmup)):
        call()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = den.info["launches"]
    total_ms = 0.0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        den.reset()
        for c in range(n_calls):
            synth(c)  # untimed: the recording "arrives"
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    launches = den.info["launches"] - launches0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, call_frames, {"out": last_out[0] if c3 else out, "vad": vad})
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    units = total_streams * n_calls * call_frames / 100.0  # stream-seconds (c4: meeting-seconds) per step, all ranks
    value = units * args.steps / (total_ms_max / 1e3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_peak, peak_src = measured_peaks()
    bytes_per_frame = (FRAME * 2 + FRAME * 4 + FRAME * 4 + 4) if c4 else ((441 * 4 + FRAME * 4 + 4) if c3 else ALG_BYTES_PER_FRAME)
    achieved = bytes_per_frame * (n * n_calls * call_frames * args.steps) / (total_ms / 1e3) / 1e9
    what = ("4,096 dual-source meetings x 10 min (BASELINE.json configs[3]): mic PCM16 denoised + raw app f32 -> "
            "clamp(mic+app) as dual-mono stereo PCM16; counts meetings" if c4 else
            ("1,024 streams x 60 s per GPU at 44.1 kHz (BASELINE.json configs[2]): windowed-sinc front end (256 taps) to 48 kHz, "
             "then denoised; f32 unit-scale in/out + VAD" if c3 else
             "8,192 streams x 60 min (BASELINE.json configs[4]), f32 unit-scale in/out + VAD"))
    line = {
        "metric": "stream-seconds of 48 kHz audio denoised per wall-second",
        "value": value, "unit": "stream-seconds/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak" if c3 else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{what}; this run: {total_streams} x {minutes:g} min over {world} GPU(s)",
                   "streams_this_rank": n, "calls_per_step": n_calls, "seconds_per_call": args.chunk_seconds,
                   "state": "every DenoiseState carried across the calls of a step (reset between steps)",
                   "timing": "only the denoise calls are timed (one CUDA event pair per call, summed, max over ranks); each "
                             "call's input is synthesised on the device just before it, outside the timed region",
                   "l2": f"{n * call_frames * in_frame * (6 if c4 else 4) / 1e9:.1f} GB in + {n * S * 4 / 1e9:.1f} GB out per call >> 126 MB L2",
                   "chunk_frames": den.info["chunk_frames"], "parallelism": f"streams/{world}gpu, no collective"},
        "clocks": clocks, "e2e": None, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": None, "peak_source": peak_src, "kernel": "whole pipeline (sum over the calls)",
                     "algorithmic_bytes_per_frame": bytes_per_frame},
        "cpu_baseline": None if args.no_cpu_baseline else cpu_reference_rate(8.0, 60.0),
        "parity_vs_oracle": parity, "wall_s_with_synthesis": t_wall,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else printed while the bench runs (NCCL's version
    banner comes from C code, past sys.stdout) was routed to stderr by main()."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())
    else:
        print(json.dumps(line), flush=True)


def main():
    global _REAL_STDOUT
    args = parse_args()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # stdout must hold exactly one JSON line
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "c2":
        run_long(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
