"""ctypes binding of the CPU oracle (oracle/rnnoise_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under crispy_b200/ imports this module.
PARITY UNPINNED against nnnoiseless itself (see oracle/rnnoise_oracle.h).
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "librnnoise_oracle.so")

FRAME_SIZE = 480
NB_BANDS = 22
NB_FEATURES = 42


class Debug(C.Structure):
    _fields_ = [
        ("features", C.c_float * 42),
        ("gains", C.c_float * 22),
        ("Ex", C.c_float * 22),
        ("Ep", C.c_float * 22),
        ("Exp", C.c_float * 22),
        ("pitch_gain", C.c_float),
        ("vad", C.c_float),
        ("pitch_index", C.c_int32),
        ("silence", C.c_int32),
    ]


class LinRes(C.Structure):
    _fields_ = [
        ("input_rate", C.c_float),
        ("output_rate", C.c_float),
        ("last_sample", C.c_float),
        ("has_last", C.c_int),
        ("input_pos", C.c_double),
        ("next_output_pos", C.c_double),
    ]


def build(force: bool = False) -> str:
    """Compile the oracle with gcc if the .so is missing or stale."""
    src = os.path.join(_HERE, "rnnoise_oracle.c")
    hdr = os.path.join(_HERE, "rnnoise_oracle.h")
    stale = (
        force
        or not os.path.exists(_LIB_PATH)
        or os.path.getmtime(_LIB_PATH) < max(os.path.getmtime(src), os.path.getmtime(hdr))
    )
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _LIB_PATH


_native_path = None


def build_native() -> str:
    """-O3 -march=native build of the same source for the CPU baseline, compiled once per process into a private
    temporary directory that is removed at exit: an -march=native object belongs to the CPU it was built on, and the
    benchmark must run from a read-only tree."""
    global _native_path
    if _native_path is None:
        d = tempfile.mkdtemp(prefix="crispy_oracle_native_")
        atexit.register(shutil.rmtree, d, True)
        path = os.path.join(d, "librnnoise_oracle_native.so")
        subprocess.check_call(["gcc", "-O3", "-march=native", "-fPIC", "-ffp-contract=off", "-fno-fast-math",
                               "-std=c11", "-shared", "-o", path, os.path.join(_HERE, "rnnoise_oracle.c"),
                               "-lm", "-lpthread"])
        _native_path = path
    return _native_path


_lib = None
_libs = {}


def lib(native: bool = False) -> C.CDLL:
    global _lib
    if native:
        if "native" not in _libs:
            _libs["native"] = _declare(C.CDLL(build_native()))
        return _libs["native"]
    if _lib is not None:
        return _lib
    build()
    _lib = _declare(C.CDLL(_LIB_PATH))
    return _lib


def _declare(L: C.CDLL) -> C.CDLL:
    vp, f32p = C.c_void_p, C.POINTER(C.c_float)
    L.rno_model_synthetic.restype = vp
    L.rno_model_synthetic.argtypes = [C.c_uint64]
    L.rno_model_from_bytes.restype = vp
    L.rno_model_from_bytes.argtypes = [C.c_char_p, C.c_size_t]
    L.rno_model_to_bytes.restype = C.c_size_t
    L.rno_model_to_bytes.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.rno_model_free.argtypes = [vp]
    L.rno_create.restype = vp
    L.rno_create.argtypes = [vp]
    L.rno_destroy.argtypes = [vp]
    L.rno_reset.argtypes = [vp]
    L.rno_process_frame.restype = C.c_float
    L.rno_process_frame.argtypes = [vp, f32p, f32p]
    L.rno_get_debug.argtypes = [vp, C.POINTER(Debug)]
    L.rno_process_streams.restype = C.c_int
    L.rno_process_streams.argtypes = [vp, f32p, f32p, f32p, C.c_int, C.c_int, C.c_long, C.c_long,
                                      C.c_uint, C.c_float, C.c_int]
    i32p = C.POINTER(C.c_int32)
    L.rno_process_streams_trace.restype = C.c_int
    L.rno_process_streams_trace.argtypes = [vp, f32p, f32p, f32p, C.c_int, C.c_int, C.c_long, C.c_long,
                                            C.c_uint, C.c_float, C.c_int, i32p, f32p, i32p, f32p]
    L.rno_set_sum_policy.argtypes = [C.c_int]
    L.rno_set_pf_perturb.argtypes = [C.c_float, C.c_float, C.c_float]
    L.rno_set_pf_perturb.restype = None
    L.rno_get_sum_policy.restype = C.c_int
    L.rno_downmix_mono.restype = None
    L.rno_downmix_mono.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_size_t, f32p]
    L.rno_resample_audio.restype = C.c_size_t
    L.rno_resample_audio.argtypes = [f32p, C.c_size_t, C.c_size_t, C.c_size_t, f32p, C.c_size_t]
    L.rno_linres_init.argtypes = [C.POINTER(LinRes), C.c_float, C.c_float]
    L.rno_linres_process.restype = C.c_size_t
    L.rno_linres_process.argtypes = [C.POINTER(LinRes), f32p, C.c_size_t, f32p, C.c_size_t]
    L.rno_sinc_resample_count.restype = C.c_size_t
    L.rno_sinc_resample_count.argtypes = [C.c_int, C.c_int, C.c_size_t]
    L.rno_sinc_resample.restype = C.c_size_t
    L.rno_sinc_resample.argtypes = [f32p, C.c_size_t, f32p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float]
    L.rno_sinc_table.restype = C.c_int
    L.rno_sinc_table.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, f32p, C.c_size_t, C.POINTER(C.c_int)]
    L.rno_processor_run.restype = C.c_size_t
    L.rno_processor_run.argtypes = [vp, C.c_float, C.c_float, f32p, C.c_size_t, f32p, C.c_size_t]
    L.rno_mix_dual_mono_i16.argtypes = [f32p, f32p, C.c_size_t, C.POINTER(C.c_int16)]
    for name in ("rno_half_window", "rno_dct_table", "rno_tansig_table"):
        getattr(L, name).restype = f32p
    L.rno_tansig_approx.restype = C.c_float
    L.rno_tansig_approx.argtypes = [C.c_float]
    L.rno_sigmoid_approx.restype = C.c_float
    L.rno_sigmoid_approx.argtypes = [C.c_float]
    L.rno_forward_transform.argtypes = [f32p, f32p]
    L.rno_inverse_transform.argtypes = [f32p, f32p]
    return L


def _fp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class Model:
    def __init__(self, handle):
        if not handle:
            raise ValueError("oracle: model load failed")
        self.h = handle

    @classmethod
    def synthetic(cls, seed: int = 0) -> "Model":
        return cls(lib().rno_model_synthetic(seed))

    @classmethod
    def from_bytes(cls, blob: bytes) -> "Model":
        return cls(lib().rno_model_from_bytes(blob, len(blob)))

    def to_bytes(self) -> bytes:
        n = lib().rno_model_to_bytes(self.h, None, 0)
        buf = C.create_string_buffer(n)
        lib().rno_model_to_bytes(self.h, buf, n)
        return buf.raw

    def __del__(self):
        try:
            lib().rno_model_free(self.h)
        except Exception:
            pass


class DenoiseState:
    """Mirror of nnnoiseless::DenoiseState (new / process_frame), oracle-backed."""

    def __init__(self, model: Model):
        self.model = model
        self.h = lib().rno_create(model.h)

    def process_frame(self, frame: np.ndarray):
        frame = np.ascontiguousarray(frame, dtype=np.float32)
        assert frame.shape == (FRAME_SIZE,)
        out = np.empty(FRAME_SIZE, dtype=np.float32)
        vad = lib().rno_process_frame(self.h, _fp(out), _fp(frame))
        return out, float(vad)

    def debug(self) -> dict:
        d = Debug()
        lib().rno_get_debug(self.h, C.byref(d))
        return {
            "features": np.array(d.features, dtype=np.float32),
            "gains": np.array(d.gains, dtype=np.float32),
            "Ex": np.array(d.Ex, dtype=np.float32),
            "Ep": np.array(d.Ep, dtype=np.float32),
            "Exp": np.array(d.Exp, dtype=np.float32),
            "pitch_gain": float(d.pitch_gain),
            "vad": float(d.vad),
            "pitch_index": int(d.pitch_index),
            "silence": int(d.silence),
        }

    def reset(self):
        lib().rno_reset(self.h)

    def __del__(self):
        try:
            lib().rno_destroy(self.h)
        except Exception:
            pass


def process_streams(model: Model, x: np.ndarray, unit_scale: bool = False, volume: float = 1.0,
                    n_threads: int = 1, native: bool = False):
    """x: [n_streams, n_frames*480] f32 -> (out same shape, vad [n_streams, n_frames])."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n_streams, n = x.shape
    n_frames = n // FRAME_SIZE
    out = np.zeros_like(x)
    vad = np.zeros((n_streams, n_frames), dtype=np.float32)
    lib(native).rno_process_streams(model.h, _fp(x), _fp(out), _fp(vad), n_streams, n_frames, n, n,
                              1 if unit_scale else 0, volume, n_threads)
    return out, vad


def process_streams_trace(model: Model, x: np.ndarray, unit_scale: bool = False, volume: float = 1.0,
                          n_threads: int = 1, native: bool = False, sum_policy: int = 0, margin: bool = False):
    """As process_streams, additionally returning every frame's discrete decisions:
    (out, vad, pitch_index [n_streams, n_frames] int32, pitch_gain f32, silence int32[, branch margin f32]).
    sum_policy: summation order of the pitch path's inner products (rnnoise_oracle.c rno_set_sum_policy)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n_streams, n = x.shape
    n_frames = n // FRAME_SIZE
    out = np.zeros_like(x)
    vad = np.zeros((n_streams, n_frames), dtype=np.float32)
    pi = np.zeros((n_streams, n_frames), dtype=np.int32)
    pg = np.zeros((n_streams, n_frames), dtype=np.float32)
    sil = np.zeros((n_streams, n_frames), dtype=np.int32)
    mg = np.zeros((n_streams, n_frames), dtype=np.float32) if margin else None
    L = lib(native)
    L.rno_set_sum_policy(int(sum_policy))
    try:
        L.rno_process_streams_trace(model.h, _fp(x), _fp(out), _fp(vad), n_streams, n_frames, n, n,
                                    1 if unit_scale else 0, volume, n_threads,
                                    pi.ctypes.data_as(C.POINTER(C.c_int32)), _fp(pg), sil.ctypes.data_as(C.POINTER(C.c_int32)),
                                    _fp(mg) if margin else None)
    finally:
        L.rno_set_sum_policy(0)
    if margin:  # + the smallest |Exp - g| over the bands per frame: distance of the pitch filter's branch from flipping
        return out, vad, pi, pg, sil, mg
    return out, vad, pi, pg, sil


def downmix_mono(x: np.ndarray, n_channels: int) -> np.ndarray:
    """audio.rs:754-755 / :816-818 / :879-884 on one interleaved buffer (float32, int16 or uint16)."""
    fmt = {np.dtype(np.float32): 0, np.dtype(np.int16): 1, np.dtype(np.uint16): 2}[x.dtype]
    x = np.ascontiguousarray(x)
    n = x.shape[0] // n_channels
    out = np.zeros(n, dtype=np.float32)
    lib().rno_downmix_mono(x.ctypes.data_as(C.c_void_p), fmt, n_channels, n, _fp(out))
    return out


def resample_audio(x: np.ndarray, from_rate: int, to_rate: int) -> np.ndarray:
    """recording.rs:13-39 (the recorder's app-audio resampler) on one buffer."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n = lib().rno_resample_audio(_fp(x), x.shape[0], from_rate, to_rate, None, 0)
    out = np.zeros(n, dtype=np.float32)
    lib().rno_resample_audio(_fp(x), x.shape[0], from_rate, to_rate, _fp(out), n)
    return out


def debug_trace(model: Model, x: np.ndarray):
    """Single stream, frame by frame, with all taps. x: [n_frames*480] (16-bit scale)."""
    st = DenoiseState(model)
    n_frames = x.shape[0] // FRAME_SIZE
    outs, taps = [], []
    for t in range(n_frames):
        o, _ = st.process_frame(x[t * FRAME_SIZE:(t + 1) * FRAME_SIZE])
        outs.append(o)
        taps.append(st.debug())
    return np.concatenate(outs) if outs else np.zeros(0, np.float32), taps


def linear_resample(x: np.ndarray, input_rate: float, output_rate: float) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32)
    r = LinRes()
    lib().rno_linres_init(C.byref(r), input_rate, output_rate)
    cap = int(len(x) * (output_rate / input_rate + 1)) + 16
    out = np.empty(cap, dtype=np.float32)
    n = lib().rno_linres_process(C.byref(r), _fp(x), len(x), _fp(out), cap)
    return out[:n].copy()


def sinc_resample(x: np.ndarray, input_rate: int, output_rate: int, sinc_len: int = 256,
                  f_cutoff: float = 0.95) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32)
    n = lib().rno_sinc_resample_count(int(input_rate), int(output_rate), len(x))
    out = np.empty(n, dtype=np.float32)
    got = lib().rno_sinc_resample(_fp(x), len(x), _fp(out), n, int(input_rate), int(output_rate), int(sinc_len),
                                  float(f_cutoff))
    assert got == n, (got, n)
    return out


def sinc_table(input_rate: int, output_rate: int, sinc_len: int = 256, f_cutoff: float = 0.95):
    """([L, sinc_len] f32 polyphase taps, M)"""
    cap = 1024 * sinc_len
    buf = np.empty(cap, dtype=np.float32)
    M = C.c_int()
    L = lib().rno_sinc_table(int(input_rate), int(output_rate), int(sinc_len), float(f_cutoff), _fp(buf), cap,
                             C.byref(M))
    return buf[:L * sinc_len].reshape(L, sinc_len).copy(), M.value


def processor_run(model: Model, x: np.ndarray, input_rate: float = 48000.0, volume: float = 1.0):
    x = np.ascontiguousarray(x, dtype=np.float32)
    cap = int(len(x) * (48000.0 / input_rate + 1)) + 1024
    out = np.empty(cap, dtype=np.float32)
    n = lib().rno_processor_run(model.h, input_rate, volume, _fp(x), len(x), _fp(out), cap)
    return out[:n].copy()


def mix_dual_mono_i16(mic: np.ndarray, app) -> np.ndarray:
    mic = np.ascontiguousarray(mic, dtype=np.float32)
    out = np.empty(2 * len(mic), dtype=np.int16)
    app_p = None
    if app is not None:
        app = np.ascontiguousarray(app, dtype=np.float32)
        app_p = _fp(app)
    lib().rno_mix_dual_mono_i16(_fp(mic), app_p, len(mic), out.ctypes.data_as(C.POINTER(C.c_int16)))
    return out


def forward_transform(x960: np.ndarray) -> np.ndarray:
    x960 = np.ascontiguousarray(x960, dtype=np.float32)
    out = np.empty(481 * 2, dtype=np.float32)
    lib().rno_forward_transform(_fp(out), _fp(x960))
    return out.view(np.complex64)


def inverse_transform(X481: np.ndarray) -> np.ndarray:
    X = np.ascontiguousarray(X481, dtype=np.complex64).view(np.float32)
    out = np.empty(960, dtype=np.float32)
    lib().rno_inverse_transform(_fp(out), _fp(X))
    return out
