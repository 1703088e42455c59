"""Shared helpers for the test-suite (test plumbing only)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
EMU_LIB = os.path.join(EMU_DIR, "libns_emu.so")
CSRC = os.path.join(ROOT, "crispy_b200", "csrc")

# tolerances stated by BASELINE.json north_star (16-bit scale: full scale = 32768)
TOL_MAX_ABS = 1e-3 * 32768.0
TOL_SNR_DB = 60.0
TOL_VAD = 1e-3
FRAME_LEN = 480


def build_emu(v7: bool = False) -> str:
    """v7: the second-generation pitch kernel (ns_pitch7.cuh, -DNS_PITCH_V7) instead of the product's."""
    lib = EMU_LIB.replace(".so", "_v7.so") if v7 else EMU_LIB
    srcs = [os.path.join(EMU_DIR, "ns_emu.cpp"), os.path.join(CSRC, "ns_host.cpp")]
    deps = srcs + [os.path.join(CSRC, f) for f in ("ns_pipe.cuh", "ns_pitch7.cuh", "ns_common.h", "ns_simt.h", "ns_host.h")]
    if not os.path.exists(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off",
                               "-Wno-unknown-pragmas"] + (["-DNS_PITCH_V7"] if v7 else []) + ["-o", lib] + srcs)
    return lib


_emu = {}


def emu_lib(v7: bool = False):
    if v7 not in _emu:
        L = C.CDLL(build_emu(v7))
        L.ns_emu_process.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                     C.c_longlong, C.c_int, C.c_uint, C.c_float, C.c_int, C.c_uint]
        L.ns_emu_set_controls.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int, C.c_float]
        L.ns_emu_set_controls.restype = None
        L.ns_emu_hp_respeculated.restype = C.c_longlong
        _emu[v7] = L
    return _emu[v7]


def emu_process(blob: bytes, x: np.ndarray, chunk: int = 16, flags: int = 0, volume: float = 1.0, state=None,
                out_dtype=np.float32, out_cols=None, app=None, out_frame_offset: int = 0, v7: bool = False,
                numerics: int = 0):
    """Run the kernel body under the host SIMT emulation.  x: [n_streams, n_frames*480]; numerics: the model's setting
    (crispy_ns_model_set_numerics)."""
    L = emu_lib(v7)
    x = np.ascontiguousarray(x)
    ns, n = x.shape
    nf = n // 480
    out = np.zeros((ns, out_cols if out_cols is not None else n), dtype=out_dtype)
    vad = np.zeros((ns, nf), np.float32)
    dbg = np.zeros((ns, nf, L.ns_emu_dbg_floats()), np.float32)
    if state is None:
        state = np.zeros((ns, L.ns_emu_state_floats()), np.float32)
    app_p, app_stride = None, 0
    if app is not None:
        app = np.ascontiguousarray(app, dtype=np.float32)
        app_p, app_stride = app.ctypes.data, app.shape[1]
    out_stride = out.shape[1] if not (flags & 8) else out.shape[1] // 2
    rc = L.ns_emu_process(blob, len(blob), x.ctypes.data, out.ctypes.data, vad.ctypes.data, app_p,
                          state.ctypes.data, dbg.ctypes.data, ns, nf, n, out_stride, app_stride, chunk, flags,
                          volume, out_frame_offset, numerics)
    assert rc == 0, f"ns_emu_process failed: {rc}"
    return out, vad, dbg, state


def patched_oracle(edits, appended: str) -> C.CDLL:
    """oracle/rnnoise_oracle.c with each (old, new) of `edits` made and `appended` added at its end, compiled as the
    oracle's own build is into a temporary directory of this process (removed at exit), with pyoracle's bindings
    declared.  Each `old` must occur exactly once in the source, so that a changed oracle stops the build."""
    src = open(os.path.join(ROOT, "oracle", "rnnoise_oracle.c")).read()
    for old, _ in edits:
        assert src.count(old) == 1, f"the oracle no longer has exactly one {old!r}: update the patch"
    for old, new in edits:
        src = src.replace(old, new)
    d = tempfile.mkdtemp(prefix="crispy_oracle_patched_")
    atexit.register(shutil.rmtree, d, True)
    c_path, so_path = os.path.join(d, "rnnoise_oracle.c"), os.path.join(d, "librnnoise_oracle.so")
    with open(c_path, "w") as f:
        f.write(src + appended)
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-shared",
                           "-I" + os.path.join(ROOT, "oracle"), "-o", so_path, c_path, "-lm", "-lpthread"])
    return po._declare(C.CDLL(so_path))


def snr_db(ref: np.ndarray, test: np.ndarray) -> float:
    ref = ref.astype(np.float64)
    err = test.astype(np.float64) - ref
    pe = float(np.mean(err ** 2))
    ps = float(np.mean(ref ** 2))
    if pe == 0.0:
        return 200.0
    return 10.0 * np.log10(max(ps, 1e-30) / pe)


def parity_report(ref_out, out, ref_vad, vad) -> dict:
    return {
        "max_abs": float(np.max(np.abs(out.astype(np.float64) - ref_out.astype(np.float64)))),
        "snr_db": snr_db(ref_out, out),
        "vad_max": float(np.max(np.abs(vad - ref_vad))) if vad.size else 0.0,
    }


def assert_parity(ref_out, out, ref_vad, vad, what=""):
    """north_star tolerances, in 16-bit scale: max abs <= 1e-3 FS, SNR >= 60 dB, VAD within 1e-3."""
    r = parity_report(ref_out, out, ref_vad, vad)
    assert r["max_abs"] <= TOL_MAX_ABS, f"{what}: max abs err {r['max_abs']} > {TOL_MAX_ABS}"
    assert r["snr_db"] >= TOL_SNR_DB, f"{what}: SNR {r['snr_db']} dB < {TOL_SNR_DB}"
    assert r["vad_max"] <= TOL_VAD, f"{what}: VAD err {r['vad_max']} > {TOL_VAD}"
    return r


def make_signal(n_streams: int, n_frames: int, seed: int = 0xC0FFEE, first_stream: int = 0) -> np.ndarray:
    """Synthetic speech+noise in 16-bit scale with an exact-silence stretch in stream 1 (if present)."""
    from crispy_b200.synth import synth_chunk
    x = synth_chunk(n_streams, n_frames * 480, seed=seed, first_stream=first_stream).numpy() * 32768.0
    x = x.astype(np.float32)
    if n_streams > 1 and n_frames >= 12:
        # digital silence exercises the E < 0.04 gate and its state rules.  After real audio the
        # high-pass rings for ~9 frames before the gate trips, so short tests put it at the start.
        x[1, : 4 * 480] = 0.0
        if n_frames >= 60:
            x[1, 20 * 480:45 * 480] = 0.0
    return x


ST_SYNTH = 1440  # ns_common.h kStSynth: two 480-float copies of synthesis_mem


def canonical_state(state: np.ndarray) -> np.ndarray:
    """The emulation keeps its chunk counter in the last word of stream 0's state block and
    synthesis_mem is double buffered on that counter's parity (ns_common.h kStSynth).  Return the
    state with the live synthesis_mem copy in slot 0, the stale copy and the counter cleared, so
    that states reached through different chunkings compare equal."""
    st = state.copy()
    sel = int(st.view(np.int32)[0, -1]) & 1
    live = st[:, ST_SYNTH + sel * 480: ST_SYNTH + (sel + 1) * 480].copy()
    st[:, ST_SYNTH: ST_SYNTH + 480] = live
    st[:, ST_SYNTH + 480: ST_SYNTH + 960] = 0.0
    st.view(np.int32)[0, -1] = 0
    return st


def adversarial_signals(n_frames: int) -> dict:
    """Inputs that push the pitch path to its corners (16-bit scale): DC, sparse impulses, loud and tiny noise, tones
    at and beyond the pitch range, clipping, a chirp, silence followed by a step."""
    n = n_frames * 480
    t = np.arange(n) / 48000.0
    rng = np.random.default_rng(1)
    sigs = {
        "dc": np.full(n, 5000.0),
        "impulses": np.where(np.arange(n) % 997 == 0, 30000.0, 0.0),
        "white_loud": rng.standard_normal(n) * 9000,
        "white_tiny": rng.standard_normal(n) * 0.3,
        "sine_60hz": 8000 * np.sin(2 * np.pi * 60 * t),
        "sine_800hz": 8000 * np.sin(2 * np.pi * 800 * t),
        "sine_62_5hz": 8000 * np.sin(2 * np.pi * 62.5 * t),
        "square_clip": np.clip(40000 * np.sin(2 * np.pi * 150 * t), -32768, 32767),
        "chirp": 9000 * np.sin(2 * np.pi * (80 + 4000 * t) * t),
        "zeros_then_step": np.concatenate([np.zeros(n // 2), np.full(n - n // 2, 12000.0)]),
    }
    return {k: v.astype(np.float32) for k, v in sigs.items()}


BRANCH_EPS = 1e-4  # the oracle's branch margin is scaled so that 1e-4 is what two float32 implementations differ by


def long_run_parity(ref, out, rvad, vad, margin, what="") -> dict:
    """Parity over a long recording (unit scale), with RNNoise's own discontinuity set apart.  The pitch filter takes
    r = 1 where the band correlation Exp exceeds the band gain g and a value that is ~0 for small g just below
    (denoise.c pitch_filter), at any magnitude: Exp = 2e-5 against g = 1e-5 takes the branch like 0.9999 against
    0.9998 (mains hum), and the band still reaches the output at 0.6 of its previous gain.  Whether Exp > g holds is
    then decided by the last bits of an FFT butterfly or of the output layer's pre-activation -- two correct
    implementations differ by ~1 % of full scale in such a frame and, through the overlap-add, in the next one
    (DESIGN.md section 3; tests/diag/pitch_filter_conditioning.py reproduces it with the oracle alone).  Frames whose
    oracle-side margin (rnnoise_oracle.c rno_process_frame: |Exp_b - g_b| against min(1e-4, 2e-3 max(|Exp_b|, g_b))
    over the audible bands) is below BRANCH_EPS, and their successors, are reported separately -- a few tenths of a
    per cent of the frames: everything else must meet north_star's max abs <= 1e-3 FS; SNR >= 60 dB and VAD within
    1e-3 must hold over ALL frames."""
    n_streams, n_frames = rvad.shape
    risky = margin < BRANCH_EPS
    risky[:, 1:] |= risky[:, :-1].copy()
    err = np.abs(out.astype(np.float64) - ref).reshape(n_streams, n_frames, FRAME_LEN).max(2)
    r = {"frames": int(rvad.size), "branch_frames_set_apart": int(risky.sum()),
         "max_abs_fs": float(err[~risky].max()) if (~risky).any() else 0.0,
         "max_abs_fs_on_branch_frames": float(err[risky].max()) if risky.any() else 0.0,
         "frames_over_1e-3_fs": int((err > 1e-3).sum()), "frames_over_1e-3_fs_fraction": float((err > 1e-3).mean()),
         "snr_db": snr_db(ref, out), "min_stream_snr_db": float(min(snr_db(ref[s], out[s]) for s in range(n_streams))),
         "vad_max": float(np.abs(vad - rvad).max())}
    assert r["max_abs_fs"] <= 1e-3, (what, r)
    assert r["max_abs_fs_on_branch_frames"] <= 0.05, (what, r)
    assert r["branch_frames_set_apart"] <= max(8, 1e-2 * rvad.size), (what, r)  # they stay the exception (hum streams: ~1 %)
    assert r["snr_db"] >= TOL_SNR_DB and r["min_stream_snr_db"] >= TOL_SNR_DB and r["vad_max"] <= TOL_VAD, (what, r)
    return r
