"""ctypes binding of libcrispy_ns.so (include/crispy_ns.h).  There is no fallback: if the library
is missing or no CUDA device is present, the calls raise."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# $CRISPY_NS_LIB selects another build of the same library (kernel tuning experiments, scripts/variants.sh)
LIB_PATH = os.environ.get("CRISPY_NS_LIB") or os.path.join(HERE, "libcrispy_ns.so")

# flags (include/crispy_ns.h)
IN_I16 = 1 << 0
OUT_I16 = 1 << 1
UNIT_SCALE = 1 << 2
MIX_STEREO_I16 = 1 << 3
DROP_FIRST_FRAME = 1 << 8

# numerics of a model (crispy_ns_model_set_numerics): sum order of the pitch path's inner products | biquad arithmetic
SUM_SEQUENTIAL = 0
SUM_DOT4 = 1
SUM_DOT4_XCORR = 2
SUM_MASK = 3
BIQUAD_F32 = 1 << 4

# every symbol include/crispy_ns.h declares
SYMBOLS = [
    "crispy_ns_frame_size", "crispy_ns_last_error", "crispy_ns_device_count",
    "crispy_ns_model_synthetic", "crispy_ns_model_from_bytes", "crispy_ns_model_to_bytes",
    "crispy_ns_model_destroy", "crispy_ns_create", "crispy_ns_process_frame", "crispy_ns_reset",
    "crispy_ns_destroy", "crispy_ns_batch_create", "crispy_ns_batch_reset", "crispy_ns_batch_reset_async", "crispy_ns_batch_n_streams",
    "crispy_ns_process_streams", "crispy_ns_process_streams_host", "crispy_ns_process_streams_debug",
    "crispy_ns_debug_floats", "crispy_ns_batch_state_size", "crispy_ns_batch_save_state",
    "crispy_ns_batch_load_state", "crispy_ns_batch_info", "crispy_ns_batch_destroy",
    "crispy_ns_host_alloc", "crispy_ns_host_free", "crispy_ns_linear_resample_count",
    "crispy_ns_linear_resample", "crispy_ns_resample_audio_count", "crispy_ns_resample_audio", "crispy_ns_downmix_mono", "crispy_ns_sinc_resample_count", "crispy_ns_sinc_resample", "crispy_ns_sinc_resample_needed", "crispy_ns_sinc_resample_chunk",
    "crispy_ns_resample_host",
    "crispy_ns_wav_write_pcm16", "crispy_ns_wav_read_pcm16",
    "crispy_ns_kernel_count", "crispy_ns_kernel_name", "crispy_ns_batch_profile", "crispy_ns_batch_profile_read",
    "crispy_ns_multi_create", "crispy_ns_multi_n_devices", "crispy_ns_multi_stream_range", "crispy_ns_multi_reset",
    "crispy_ns_multi_process_streams_host", "crispy_ns_multi_destroy", "crispy_ns_denoise_wav_files",
    "crispy_ns_measure_fp32",
    "crispy_ns_process_streams_subset", "crispy_ns_process_streams_subset_host", "crispy_ns_batch_reset_streams",
    "crispy_ns_stream_state_size", "crispy_ns_batch_save_streams", "crispy_ns_batch_load_streams",
    "crispy_ns_model_set_numerics", "crispy_ns_model_numerics",
    "crispy_ns_batch_set_controls", "crispy_ns_batch_get_controls", "crispy_ns_set_controls", "crispy_ns_get_controls",
    "crispy_ns_multi_set_controls", "crispy_ns_multi_get_controls",
]


class Controls(C.Structure):
    """crispy_ns_controls (include/crispy_ns.h): per-stream attenuation limit and voice gate; all zero = off"""
    _fields_ = [("min_gain", C.c_float), ("gate_threshold", C.c_float), ("gate_hold", C.c_int32),
                ("gate_gain", C.c_float)]


class CrispyNsError(RuntimeError):
    pass


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CrispyNsError(
            f"{LIB_PATH} is missing: build it with `python -m crispy_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, vpp = C.c_void_p, C.POINTER(C.c_void_p)
    i64, u32, f32 = C.c_int64, C.c_uint32, C.c_float
    L.crispy_ns_frame_size.restype = C.c_int
    L.crispy_ns_last_error.restype = C.c_char_p
    L.crispy_ns_device_count.restype = C.c_int
    L.crispy_ns_model_synthetic.argtypes = [C.c_uint64, vpp]
    L.crispy_ns_model_from_bytes.argtypes = [C.c_char_p, C.c_size_t, vpp]
    L.crispy_ns_model_to_bytes.argtypes = [vp, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.crispy_ns_model_destroy.argtypes = [vp]
    L.crispy_ns_model_destroy.restype = None
    L.crispy_ns_model_set_numerics.argtypes = [vp, u32]
    L.crispy_ns_model_numerics.argtypes = [vp]
    L.crispy_ns_model_numerics.restype = u32
    L.crispy_ns_create.argtypes = [vp, C.c_int, vpp]
    L.crispy_ns_process_frame.argtypes = [vp, vp, vp, C.POINTER(f32)]
    L.crispy_ns_reset.argtypes = [vp]
    L.crispy_ns_destroy.argtypes = [vp]
    L.crispy_ns_destroy.restype = None
    L.crispy_ns_batch_create.argtypes = [vp, C.c_int, C.c_int, vpp]
    L.crispy_ns_batch_reset.argtypes = [vp]
    L.crispy_ns_batch_reset_async.argtypes = [vp, vp]
    L.crispy_ns_batch_n_streams.argtypes = [vp]
    L.crispy_ns_process_streams.argtypes = [vp, vp, vp, vp, vp, C.c_int, i64, i64, i64, i64, u32, f32, vp]
    L.crispy_ns_process_streams_host.argtypes = [vp, vp, vp, vp, vp, C.c_int, i64, i64, i64, i64, u32, f32]
    L.crispy_ns_process_streams_debug.argtypes = [vp, vp, vp, vp, vp, C.c_int, i64, i64, u32, f32, vp]
    L.crispy_ns_debug_floats.restype = C.c_int
    L.crispy_ns_batch_state_size.argtypes = [vp]
    L.crispy_ns_batch_state_size.restype = C.c_size_t
    L.crispy_ns_batch_save_state.argtypes = [vp, vp, C.c_size_t]
    L.crispy_ns_batch_load_state.argtypes = [vp, vp, C.c_size_t]
    ip = C.POINTER(C.c_int)
    L.crispy_ns_process_streams_subset.argtypes = [vp, ip, C.c_int, vp, vp, vp, vp, C.c_int, i64, i64, i64, i64, u32, f32, vp]
    L.crispy_ns_process_streams_subset_host.argtypes = [vp, ip, C.c_int, vp, vp, vp, vp, C.c_int, i64, i64, i64, i64, u32, f32]
    L.crispy_ns_batch_reset_streams.argtypes = [vp, ip, C.c_int, vp]
    L.crispy_ns_stream_state_size.restype = C.c_size_t
    L.crispy_ns_batch_save_streams.argtypes = [vp, ip, C.c_int, vp, C.c_size_t]
    L.crispy_ns_batch_load_streams.argtypes = [vp, ip, C.c_int, vp, C.c_size_t]
    cp = C.POINTER(Controls)
    L.crispy_ns_batch_set_controls.argtypes = [vp, ip, C.c_int, cp, vp]
    L.crispy_ns_batch_get_controls.argtypes = [vp, ip, C.c_int, cp]
    L.crispy_ns_set_controls.argtypes = [vp, cp]
    L.crispy_ns_get_controls.argtypes = [vp, cp]
    L.crispy_ns_multi_set_controls.argtypes = [vp, ip, C.c_int, cp]
    L.crispy_ns_multi_get_controls.argtypes = [vp, ip, C.c_int, cp]
    L.crispy_ns_batch_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(i64), C.POINTER(i64)]
    L.crispy_ns_kernel_count.restype = C.c_int
    L.crispy_ns_kernel_name.argtypes = [C.c_int]
    L.crispy_ns_kernel_name.restype = C.c_char_p
    L.crispy_ns_batch_profile.argtypes = [vp, C.c_int]
    L.crispy_ns_batch_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64), C.c_int]
    L.crispy_ns_batch_destroy.argtypes = [vp]
    L.crispy_ns_batch_destroy.restype = None
    L.crispy_ns_host_alloc.argtypes = [vpp, C.c_size_t]
    L.crispy_ns_host_free.argtypes = [vp]
    L.crispy_ns_host_free.restype = None
    L.crispy_ns_linear_resample_count.argtypes = [f32, f32, i64]
    L.crispy_ns_linear_resample_count.restype = i64
    L.crispy_ns_linear_resample.argtypes = [C.c_int, vp, vp, C.c_int, i64, i64, i64, f32, f32, vp]
    L.crispy_ns_downmix_mono.argtypes = [C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, i64, i64, i64, vp]
    L.crispy_ns_resample_audio_count.argtypes = [i64, C.c_int, C.c_int]
    L.crispy_ns_resample_audio_count.restype = i64
    L.crispy_ns_resample_audio.argtypes = [C.c_int, vp, vp, C.c_int, i64, i64, i64, C.c_int, C.c_int, vp]
    L.crispy_ns_sinc_resample_count.argtypes = [C.c_int, C.c_int, i64]
    L.crispy_ns_sinc_resample_count.restype = i64
    L.crispy_ns_sinc_resample.argtypes = [C.c_int, vp, vp, C.c_int, i64, i64, i64, C.c_int, C.c_int, C.c_int, f32, vp]
    L.crispy_ns_sinc_resample_needed.argtypes = [C.c_int, C.c_int, C.c_int, i64, i64, i64, C.POINTER(i64), C.POINTER(i64)]
    L.crispy_ns_sinc_resample_chunk.argtypes = [C.c_int, vp, i64, i64, i64, vp, i64, i64, C.c_int, i64, i64, C.c_int, C.c_int,
                                                C.c_int, f32, vp]
    L.crispy_ns_resample_host.argtypes = [C.c_int, vp, vp, C.c_int, i64, i64, i64, C.c_int, C.c_int, C.c_int]
    L.crispy_ns_wav_write_pcm16.argtypes = [C.c_char_p, vp, i64, C.c_int, C.c_int]
    L.crispy_ns_wav_read_pcm16.argtypes = [C.c_char_p, vp, i64, C.POINTER(i64), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.crispy_ns_multi_create.argtypes = [vp, C.POINTER(C.c_int), C.c_int, C.c_int, vpp]
    L.crispy_ns_multi_n_devices.argtypes = [vp]
    L.crispy_ns_multi_stream_range.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.crispy_ns_multi_reset.argtypes = [vp]
    L.crispy_ns_multi_process_streams_host.argtypes = [vp, vp, vp, vp, vp, C.c_int, i64, i64, i64, i64, u32, f32]
    L.crispy_ns_multi_destroy.argtypes = [vp]
    L.crispy_ns_multi_destroy.restype = None
    L.crispy_ns_denoise_wav_files.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_int, u32, f32,
                                              C.POINTER(f32)]
    L.crispy_ns_measure_fp32.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().crispy_ns_last_error()
        raise CrispyNsError(f"libcrispy_ns error {rc}: {msg.decode() if msg else ''}")
