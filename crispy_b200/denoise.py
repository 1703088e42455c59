"""Host-side mirror of the reference's noise-suppression interface, over libcrispy_ns.so.

The reference is Rust (`src-tauri/src/audio.rs`); no Rust toolchain exists in this image, so the
verified host layer is Python over the C ABI (include/crispy_ns.h).  Names, argument meaning and
error behaviour follow the reference:

  DenoiseState.new() / .process_frame(out, inp) -> vad   nnnoiseless surface used at audio.rs:229, :268
  RnnNoiseProcessor(input_rate, output_rate, volume)      audio.rs:202-315 (push_sample / next_sample)
  LinearResampler(input_rate, output_rate)                audio.rs:73-134
  BatchDenoiser(n_streams).process_streams(...)           the batched surface north_star adds

PyTorch is used only to own device / pinned memory and CUDA streams; all arithmetic on the path is
in the hand-written sm_100a kernels.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import deque
from typing import Optional, Tuple

import numpy as np

from . import _lib
from ._lib import (DROP_FIRST_FRAME, IN_I16, MIX_STEREO_I16, OUT_I16, UNIT_SCALE, CrispyNsError,
                   check)

FRAME_SIZE = 480  # nnnoiseless::FRAME_SIZE (audio.rs:4)
SAMPLE_RATE = 48000


def device_count() -> int:
    return int(_lib.lib().crispy_ns_device_count())


class Model:
    """The six int8 RNN layers.  nnnoiseless embeds its weights in the crate; here they are data."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)

    @classmethod
    def synthetic(cls, seed: int = 0) -> "Model":
        h = C.c_void_p()
        check(_lib.lib().crispy_ns_model_synthetic(seed, C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_bytes(cls, blob: bytes) -> "Model":
        h = C.c_void_p()
        check(_lib.lib().crispy_ns_model_from_bytes(blob, len(blob), C.byref(h)))
        return cls(h.value)

    @property
    def numerics(self) -> int:
        """Which float32 arithmetic the pitch path's decisions follow: a SUM_* order | BIQUAD_F32 (crispy_b200._lib;
        include/crispy_ns.h crispy_ns_model_set_numerics).  0, the default, is xiph's C.  Handles copy it when they are
        created; to_bytes / from_bytes do not carry it."""
        return int(_lib.lib().crispy_ns_model_numerics(self._h))

    @numerics.setter
    def numerics(self, value: int) -> None:
        check(_lib.lib().crispy_ns_model_set_numerics(self._h, int(value)))

    def to_bytes(self) -> bytes:
        n = C.c_size_t()
        check(_lib.lib().crispy_ns_model_to_bytes(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        check(_lib.lib().crispy_ns_model_to_bytes(self._h, buf, n.value, C.byref(n)))
        return buf.raw

    def __del__(self):
        try:
            _lib.lib().crispy_ns_model_destroy(self._h)
        except Exception:
            pass


class DenoiseState:
    """Mirror of nnnoiseless::DenoiseState as the reference uses it (audio.rs:203, :229, :268)."""

    FRAME_SIZE = FRAME_SIZE

    def __init__(self, model: Optional[Model] = None, device: int = 0):
        self._model = model
        self._h = C.c_void_p()
        check(_lib.lib().crispy_ns_create(model._h if model else None, device, C.byref(self._h)))

    @classmethod
    def new(cls, model: Optional[Model] = None, device: int = 0) -> "DenoiseState":
        return cls(model, device)

    def process_frame(self, out: np.ndarray, inp: np.ndarray) -> float:
        """out, inp: 480 f32 in 16-bit scale.  Returns the VAD probability.  Like upstream, a slice
        of the wrong length is a programming error (upstream asserts)."""
        if inp.shape != (FRAME_SIZE,) or out.shape != (FRAME_SIZE,):
            raise AssertionError("process_frame needs two 480-sample frames")
        if inp.dtype != np.float32 or out.dtype != np.float32 or not out.flags.c_contiguous:
            raise AssertionError("process_frame needs contiguous float32 frames")
        inp = np.ascontiguousarray(inp)
        vad = C.c_float()
        check(_lib.lib().crispy_ns_process_frame(self._h, out.ctypes.data, inp.ctypes.data, C.byref(vad)))
        return float(vad.value)

    def reset(self) -> None:
        check(_lib.lib().crispy_ns_reset(self._h))

    def __del__(self):
        try:
            if self._h:
                _lib.lib().crispy_ns_destroy(self._h)
        except Exception:
            pass


class LinearResampler:
    """audio.rs:73-134, sample for sample (f64 positions, f32 samples)."""

    def __init__(self, input_rate: float, output_rate: float):
        self.set_rates(input_rate, output_rate)

    def rates(self) -> Tuple[float, float]:
        return float(self.input_rate), float(self.output_rate)

    def set_rates(self, input_rate: float, output_rate: float) -> None:
        self.input_rate = np.float32(input_rate)
        self.output_rate = np.float32(output_rate)
        self.last_sample = np.float32(0.0)
        self.has_last = False
        self.input_pos = 0.0
        self.next_output_pos = 0.0

    def process_sample(self, sample: float, emit) -> None:
        sample = np.float32(sample)
        if abs(self.input_rate - self.output_rate) < 1.0:
            emit(sample)
            return
        if not self.has_last:
            self.last_sample = sample
            self.has_last = True
            self.input_pos = 0.0
            self.next_output_pos = 0.0
            return
        self.input_pos += 1.0
        step = float(np.float32(self.input_rate / self.output_rate))
        while self.next_output_pos <= self.input_pos:
            t = np.float32(self.next_output_pos - (self.input_pos - 1.0))
            t = np.float32(min(max(t, np.float32(0.0)), np.float32(1.0)))
            emit(np.float32(self.last_sample + np.float32(np.float32(sample - self.last_sample) * t)))
            self.next_output_pos += step
        self.last_sample = sample


def linear_resample(x, input_rate: float, output_rate: float):
    """Batched LinearResampler on the GPU: x is a CUDA f32 tensor [n_streams, n_in]; returns
    [n_streams, n_out], bit-identical to feeding every row through LinearResampler."""
    import torch
    if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise CrispyNsError("linear_resample needs a CUDA float32 [n_streams, n_in] tensor")
    n_streams, n_in = x.shape
    n_out = int(_lib.lib().crispy_ns_linear_resample_count(input_rate, output_rate, n_in))
    out = torch.empty((n_streams, n_out), dtype=torch.float32, device=x.device)
    st = torch.cuda.current_stream(x.device).cuda_stream
    check(_lib.lib().crispy_ns_linear_resample(x.device.index or 0, x.data_ptr(), out.data_ptr(), n_streams,
                                               n_in, x.stride(0), out.stride(0) if n_out else 0,
                                               input_rate, output_rate, st))
    return out


def downmix_mono(x, n_channels: int):
    """The capture callbacks' downmix (audio.rs:754-755, :816-818, :879-884) on the device.  x: CUDA tensor
    [n_streams, n_frames * n_channels] of interleaved float32, int16 or uint16 samples -> float32 [n_streams, n_frames]."""
    import torch
    fmts = {torch.float32: 0, torch.int16: 1, torch.uint16: 2}
    if not x.is_cuda or x.dim() != 2 or x.stride(1) != 1 or x.dtype not in fmts or n_channels < 1:
        raise CrispyNsError("downmix_mono needs a CUDA [n_streams, n_frames * n_channels] tensor of float32, int16 or uint16")
    n_streams, n_frames = x.shape[0], x.shape[1] // int(n_channels)
    out = torch.empty((n_streams, n_frames), dtype=torch.float32, device=x.device)
    if n_streams and n_frames:
        check(_lib.lib().crispy_ns_downmix_mono(x.device.index or 0, x.data_ptr(), fmts[x.dtype], int(n_channels), out.data_ptr(),
                                                n_streams, n_frames, x.stride(0), out.stride(0),
                                                torch.cuda.current_stream(x.device).cuda_stream))
    return out


def resample_audio(x, from_rate: int, to_rate: int):
    """recording.rs:13-39 on the device: the recorder's whole-buffer linear interpolator for captured app audio
    (what reaches the dual-mono mix beside the denoised microphone).  x: CUDA float32 [n_streams, n_in]."""
    import torch
    if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise CrispyNsError("resample_audio needs a CUDA float32 [n_streams, n_in] tensor")
    n_streams, n_in = x.shape
    n_out = int(_lib.lib().crispy_ns_resample_audio_count(n_in, int(from_rate), int(to_rate)))
    out = torch.empty((n_streams, n_out), dtype=torch.float32, device=x.device)
    if n_streams and n_out:
        check(_lib.lib().crispy_ns_resample_audio(x.device.index or 0, x.data_ptr(), out.data_ptr(), n_streams, n_in,
                                                  x.stride(0), out.stride(0), int(from_rate), int(to_rate),
                                                  torch.cuda.current_stream(x.device).cuda_stream))
    return out


def sinc_resample(x, input_rate: int, output_rate: int, sinc_len: int = 256, f_cutoff: float = 0.95):
    """Batched windowed-sinc resampler on the GPU (north_star item 4: the rubato-equivalent
    44.1 -> 48 kHz front end; rubato 0.16.2 pinned at Cargo.lock:4166).  x is a CUDA f32 tensor
    [n_streams, n_in]; returns [n_streams, ceil(n_in*L/M)].  Asynchronous on the current stream."""
    import torch
    if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise CrispyNsError("sinc_resample needs a CUDA float32 [n_streams, n_in] tensor")
    n_streams, n_in = x.shape
    n_out = int(_lib.lib().crispy_ns_sinc_resample_count(int(input_rate), int(output_rate), n_in))
    out = torch.empty((n_streams, n_out), dtype=torch.float32, device=x.device)
    st = torch.cuda.current_stream(x.device).cuda_stream
    check(_lib.lib().crispy_ns_sinc_resample(x.device.index or 0, x.data_ptr(), out.data_ptr(), n_streams,
                                             n_in, x.stride(0), out.stride(0) if n_out else 0,
                                             int(input_rate), int(output_rate), int(sinc_len), float(f_cutoff), st))
    return out


def sinc_needed(input_rate: int, output_rate: int, n_total: int, first_out: int, n_out: int, sinc_len: int = 256):
    """(in_first, n_in): the input samples the taps of outputs first_out .. first_out + n_out touch."""
    a, b = C.c_int64(), C.c_int64()
    check(_lib.lib().crispy_ns_sinc_resample_needed(int(input_rate), int(output_rate), int(sinc_len), int(n_total),
                                                    int(first_out), int(n_out), C.byref(a), C.byref(b)))
    return a.value, b.value


def sinc_resample_chunk(x_window, in_first: int, n_total: int, first_out: int, n_out: int, input_rate: int,
                        output_rate: int, sinc_len: int = 256, f_cutoff: float = 0.95):
    """Outputs first_out .. first_out + n_out of a long recording from the window of it that is on the GPU
    (x_window[:, 0] is the recording's sample in_first).  Chunked calls reproduce sinc_resample bit for bit."""
    import torch
    if not x_window.is_cuda or x_window.dtype != torch.float32 or x_window.dim() != 2 or x_window.stride(1) != 1:
        raise CrispyNsError("sinc_resample_chunk needs a CUDA float32 [n_streams, n_in] tensor")
    n_streams, n_in = x_window.shape
    out = torch.empty((n_streams, n_out), dtype=torch.float32, device=x_window.device)
    st = torch.cuda.current_stream(x_window.device).cuda_stream
    check(_lib.lib().crispy_ns_sinc_resample_chunk(x_window.device.index or 0, x_window.data_ptr(), int(in_first), n_in,
                                                   int(n_total), out.data_ptr(), int(first_out), int(n_out), n_streams,
                                                   x_window.stride(0), out.stride(0) if n_out else 0, int(input_rate),
                                                   int(output_rate), int(sinc_len), float(f_cutoff), st))
    return out


def resample_host(x, input_rate: int, output_rate: int, kind: str = "sinc", device: int = 0):
    """Host-array front end (crispy_ns_resample_host): x is a host f32 array [n_streams, n_in]; returns a numpy
    array [n_streams, n_out].  kind: "linear" (audio.rs:108-133), "sinc", or "audio" (recording.rs:13-39)."""
    xa = np.ascontiguousarray(x, dtype=np.float32)
    if xa.ndim != 2:
        raise CrispyNsError("resample_host needs a [n_streams, n_in] array")
    L = _lib.lib()
    k = {"linear": 0, "sinc": 1, "audio": 2}[kind]
    n_streams, n_in = xa.shape
    n_out = int(L.crispy_ns_linear_resample_count(float(input_rate), float(output_rate), n_in) if k == 0 else
                L.crispy_ns_sinc_resample_count(int(input_rate), int(output_rate), n_in) if k == 1 else
                L.crispy_ns_resample_audio_count(n_in, int(input_rate), int(output_rate)))
    out = np.empty((n_streams, n_out), dtype=np.float32)
    check(L.crispy_ns_resample_host(device, xa.ctypes.data, out.ctypes.data, n_streams, n_in, n_in, max(n_out, 1),
                                    int(input_rate), int(output_rate), k))
    return out


class BatchDenoiser:
    """n independent DenoiseStates on one GPU; state persists across calls (chunked recordings)."""

    def __init__(self, n_streams: int, model: Optional[Model] = None, device: int = 0):
        self.n_streams = int(n_streams)
        self.device = int(device)
        self._model = model
        self._h = C.c_void_p()
        check(_lib.lib().crispy_ns_batch_create(model._h if model else None, device, n_streams, C.byref(self._h)))

    # ---- device-resident path -------------------------------------------------------------------
    def process_streams(self, x, *, unit_scale: bool = True, volume: float = 1.0,
                        drop_first_frame: bool = False, out=None, vad=None, out_i16: bool = False,
                        app=None, mix_stereo_i16: bool = False, return_taps: bool = False,
                        input_rate: float = SAMPLE_RATE, front_end: str = "linear"):
        """x: CUDA tensor [n_streams, n_frames*480], f32 (unit scale by default, i.e. the
        RnnNoiseProcessor convention) or int16.  Returns (out, vad[, taps]).  Asynchronous on the
        current torch CUDA stream.  With input_rate != 48 kHz (f32 only) the front end runs first on
        the same stream: "linear" = the reference's LinearResampler (audio.rs:217-221), "sinc" = the
        windowed-sinc kernel; a whole recording per call (the resamplers keep no state across calls)."""
        import torch
        if abs(float(input_rate) - SAMPLE_RATE) >= 1.0:
            if front_end == "sinc":
                x = sinc_resample(x, int(round(input_rate)), int(SAMPLE_RATE))
            elif front_end == "linear":
                x = linear_resample(x, float(input_rate), float(SAMPLE_RATE))
            else:
                raise CrispyNsError("front_end must be 'linear' or 'sinc'")
        if not x.is_cuda or x.dim() != 2 or x.stride(1) != 1 or x.shape[0] != self.n_streams:
            raise CrispyNsError("process_streams needs a CUDA [n_streams, n_samples] tensor")
        if x.dtype not in (torch.float32, torch.int16):
            raise CrispyNsError("process_streams input must be float32 or int16")
        n_frames = x.shape[1] // FRAME_SIZE
        flags = 0
        if x.dtype == torch.int16:
            flags |= IN_I16
        if unit_scale:
            flags |= UNIT_SCALE
        first = drop_first_frame and self.frames_done == 0
        if drop_first_frame:
            flags |= DROP_FIRST_FRAME
        n_out_frames = n_frames - (1 if first else 0)
        dev = x.device
        if mix_stereo_i16:
            flags |= MIX_STEREO_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE, 2), dtype=torch.int16, device=dev)
            out_stride = out.stride(0) // 2
        elif out_i16:
            flags |= OUT_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE), dtype=torch.int16, device=dev)
            out_stride = out.stride(0)
        else:
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE), dtype=torch.float32, device=dev)
            out_stride = out.stride(0)
        if vad is None:
            vad = torch.zeros((self.n_streams, n_frames), dtype=torch.float32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        L = _lib.lib()
        if return_taps:
            taps = torch.zeros((self.n_streams, n_frames, L.crispy_ns_debug_floats()), dtype=torch.float32, device=dev)
            check(L.crispy_ns_process_streams_debug(self._h, x.data_ptr(), out.data_ptr(), vad.data_ptr(),
                                                    taps.data_ptr(), n_frames, x.stride(0), out_stride, flags,
                                                    volume, st))
            return out, vad, taps
        app_ptr, app_stride = None, 0
        if app is not None:
            if not app.is_cuda or app.dtype != torch.float32 or app.stride(1) != 1:
                raise CrispyNsError("app audio must be a CUDA float32 tensor")
            app_ptr, app_stride = app.data_ptr(), app.stride(0)
        check(L.crispy_ns_process_streams(self._h, x.data_ptr(), out.data_ptr(), vad.data_ptr(), app_ptr,
                                          n_frames, x.stride(0), out_stride, vad.stride(0), app_stride, flags,
                                          volume, st))
        return out, vad

    # ---- host path (what a caller with recordings in RAM uses) ------------------------------------
    def process_streams_host(self, x, *, unit_scale: bool = True, volume: float = 1.0,
                             drop_first_frame: bool = False, out=None, vad=None, out_i16: bool = False,
                             app=None, mix_stereo_i16: bool = False):
        """x: host tensor/array [n_streams, n_frames*480] (pinned for copy/compute overlap).
        Synchronous; H2D, kernel and D2H are pipelined in time chunks inside the library."""
        import torch
        xt = torch.as_tensor(x)
        if xt.is_cuda or xt.dim() != 2 or xt.stride(1) != 1 or xt.shape[0] != self.n_streams:
            raise CrispyNsError("process_streams_host needs a host [n_streams, n_samples] tensor")
        n_frames = xt.shape[1] // FRAME_SIZE
        flags = 0
        if xt.dtype == torch.int16:
            flags |= IN_I16
        elif xt.dtype != torch.float32:
            raise CrispyNsError("process_streams_host input must be float32 or int16")
        if unit_scale:
            flags |= UNIT_SCALE
        first = drop_first_frame and self.frames_done == 0
        if drop_first_frame:
            flags |= DROP_FIRST_FRAME
        n_out_frames = n_frames - (1 if first else 0)
        if mix_stereo_i16:
            flags |= MIX_STEREO_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE, 2), dtype=torch.int16)
            out_stride = out.stride(0) // 2
        elif out_i16:
            flags |= OUT_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE), dtype=torch.int16)
            out_stride = out.stride(0)
        else:
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE), dtype=torch.float32)
            out_stride = out.stride(0)
        if vad is None:
            vad = torch.zeros((self.n_streams, n_frames), dtype=torch.float32)
        app_ptr, app_stride = None, 0
        if app is not None:
            app = torch.as_tensor(app)
            app_ptr, app_stride = app.data_ptr(), app.stride(0)
        check(_lib.lib().crispy_ns_process_streams_host(self._h, xt.data_ptr(), out.data_ptr(), vad.data_ptr(),
                                                        app_ptr, n_frames, xt.stride(0), out_stride,
                                                        vad.stride(0), app_stride, flags, volume))
        return out, vad

    # ---- streams that advance independently (include/crispy_ns.h, per-stream section) -------------
    def _ids(self, streams):
        ids = np.ascontiguousarray(np.asarray(streams, dtype=np.int64).reshape(-1))
        if ids.size and (ids.min() < 0 or ids.max() >= self.n_streams):
            raise CrispyNsError("stream id out of range")
        ids = ids.astype(np.int32)
        return ids, ids.ctypes.data_as(C.POINTER(C.c_int))

    def _subset_io(self, n_rows, n_frames, in_dtype, unit_scale, drop_first_frame, out, vad, out_i16, mix_stereo_i16,
                   device):
        import torch
        flags = (IN_I16 if in_dtype == torch.int16 else 0) | (UNIT_SCALE if unit_scale else 0)
        if drop_first_frame:
            flags |= DROP_FIRST_FRAME  # refused by the library: the caller drops a stream's first frame itself
        n_samples = n_frames * FRAME_SIZE
        if mix_stereo_i16:
            flags |= MIX_STEREO_I16
            if out is None:
                out = torch.zeros((n_rows, n_samples, 2), dtype=torch.int16, device=device)
            out_stride = out.stride(0) // 2
        else:
            if out_i16:
                flags |= OUT_I16
            if out is None:
                out = torch.zeros((n_rows, n_samples), dtype=torch.int16 if out_i16 else torch.float32, device=device)
            out_stride = out.stride(0)
        if vad is None:
            vad = torch.zeros((n_rows, n_frames), dtype=torch.float32, device=device)
        return flags, out, out_stride, vad

    def process_streams_subset(self, streams, x, *, unit_scale: bool = True, volume: float = 1.0,
                               drop_first_frame: bool = False, out=None, vad=None, out_i16: bool = False,
                               app=None, mix_stereo_i16: bool = False, input_rate: float = SAMPLE_RATE,
                               front_end: str = "linear"):
        """As process_streams for the listed streams only: row i of x (CUDA tensor [len(streams), n_frames*480]) is
        stream streams[i]; every other stream's state stays as it was.  Asynchronous on the current torch stream.
        drop_first_frame is refused (the caller drops a stream's first frame)."""
        import torch
        if abs(float(input_rate) - SAMPLE_RATE) >= 1.0:
            if front_end not in ("linear", "sinc"):
                raise CrispyNsError("front_end must be 'linear' or 'sinc'")
            x = (sinc_resample(x, int(round(input_rate)), int(SAMPLE_RATE)) if front_end == "sinc"
                 else linear_resample(x, float(input_rate), float(SAMPLE_RATE)))
        ids, ptr = self._ids(streams)
        if not x.is_cuda or x.dim() != 2 or x.stride(1) != 1 or x.shape[0] != ids.size:
            raise CrispyNsError("process_streams_subset needs a CUDA [len(streams), n_samples] tensor")
        if x.dtype not in (torch.float32, torch.int16):
            raise CrispyNsError("process_streams_subset input must be float32 or int16")
        n_frames = x.shape[1] // FRAME_SIZE
        flags, out, out_stride, vad = self._subset_io(ids.size, n_frames, x.dtype, unit_scale, drop_first_frame, out,
                                                      vad, out_i16, mix_stereo_i16, x.device)
        app_ptr, app_stride = None, 0
        if app is not None:
            if not app.is_cuda or app.dtype != torch.float32 or app.stride(1) != 1:
                raise CrispyNsError("app audio must be a CUDA float32 tensor")
            app_ptr, app_stride = app.data_ptr(), app.stride(0)
        st = torch.cuda.current_stream(x.device).cuda_stream
        check(_lib.lib().crispy_ns_process_streams_subset(self._h, ptr, int(ids.size), x.data_ptr(), out.data_ptr(),
                                                          vad.data_ptr(), app_ptr, n_frames, x.stride(0), out_stride,
                                                          vad.stride(0), app_stride, flags, volume, st))
        return out, vad

    def process_streams_subset_host(self, streams, x, *, unit_scale: bool = True, volume: float = 1.0,
                                    drop_first_frame: bool = False, out=None, vad=None, out_i16: bool = False,
                                    app=None, mix_stereo_i16: bool = False):
        """As process_streams_host for the listed streams only (row i of the host tensor x is stream streams[i])."""
        import torch
        ids, ptr = self._ids(streams)
        xt = torch.as_tensor(x)
        if xt.is_cuda or xt.dim() != 2 or xt.stride(1) != 1 or xt.shape[0] != ids.size:
            raise CrispyNsError("process_streams_subset_host needs a host [len(streams), n_samples] tensor")
        if xt.dtype not in (torch.float32, torch.int16):
            raise CrispyNsError("process_streams_subset_host input must be float32 or int16")
        n_frames = xt.shape[1] // FRAME_SIZE
        flags, out, out_stride, vad = self._subset_io(ids.size, n_frames, xt.dtype, unit_scale, drop_first_frame, out,
                                                      vad, out_i16, mix_stereo_i16, "cpu")
        app_ptr, app_stride = None, 0
        if app is not None:
            app = torch.as_tensor(app)
            app_ptr, app_stride = app.data_ptr(), app.stride(0)
        check(_lib.lib().crispy_ns_process_streams_subset_host(self._h, ptr, int(ids.size), xt.data_ptr(), out.data_ptr(),
                                                               vad.data_ptr(), app_ptr, n_frames, xt.stride(0),
                                                               out_stride, vad.stride(0), app_stride, flags, volume))
        return out, vad

    def reset_streams(self, streams) -> None:
        """Fresh DenoiseStates for the listed streams, on the current torch CUDA stream (no host sync)."""
        import torch
        ids, ptr = self._ids(streams)
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(_lib.lib().crispy_ns_batch_reset_streams(self._h, ptr, int(ids.size), st))

    def save_streams(self, streams) -> bytes:
        """One self-describing record per listed stream (stream_state_size() bytes each), concatenated."""
        ids, ptr = self._ids(streams)
        n = int(ids.size) * stream_state_size()
        buf = C.create_string_buffer(max(n, 1))
        check(_lib.lib().crispy_ns_batch_save_streams(self._h, ptr, int(ids.size), buf, n))
        return buf.raw[:n]

    def load_streams(self, streams, blob: bytes) -> None:
        """Put the records of save_streams (from any batch of this build) into the listed streams."""
        ids, ptr = self._ids(streams)
        check(_lib.lib().crispy_ns_batch_load_streams(self._h, ptr, int(ids.size), blob, len(blob)))

    # ---- bookkeeping ----------------------------------------------------------------------------
    @property
    def info(self) -> dict:
        s, c, l, f = C.c_int(), C.c_int(), C.c_int64(), C.c_int64()
        check(_lib.lib().crispy_ns_batch_info(self._h, C.byref(s), C.byref(c), C.byref(l), C.byref(f)))
        return {"rnn_streams_per_cta": s.value, "chunk_frames": c.value, "launches": l.value, "frames_done": f.value}

    @property
    def frames_done(self) -> int:
        return self.info["frames_done"]

    def profile(self, enable: bool = True) -> None:
        """Bracket every kernel launch with CUDA events on its own stream (measurement aid)."""
        check(_lib.lib().crispy_ns_batch_profile(self._h, 1 if enable else 0))

    def profile_read(self) -> dict:
        """{kernel name: (summed device ms, launches)} since the last read; synchronises."""
        L = _lib.lib()
        n = L.crispy_ns_kernel_count()
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        check(L.crispy_ns_batch_profile_read(self._h, ms, cnt, n))
        return {L.crispy_ns_kernel_name(k).decode(): (float(ms[k]), int(cnt[k])) for k in range(n)}

    def save_state(self) -> bytes:
        n = _lib.lib().crispy_ns_batch_state_size(self._h)
        buf = C.create_string_buffer(n)
        check(_lib.lib().crispy_ns_batch_save_state(self._h, buf, n))
        return buf.raw

    def load_state(self, blob: bytes) -> None:
        check(_lib.lib().crispy_ns_batch_load_state(self._h, blob, len(blob)))

    def reset(self) -> None:
        check(_lib.lib().crispy_ns_batch_reset(self._h))

    def reset_async(self) -> None:
        """Fresh DenoiseStates, as a memset on the current torch CUDA stream (no host sync)."""
        import torch
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(_lib.lib().crispy_ns_batch_reset_async(self._h, st))

    def __del__(self):
        try:
            if self._h:
                _lib.lib().crispy_ns_batch_destroy(self._h)
        except Exception:
            pass


def stream_state_size() -> int:
    """Bytes of one stream record of BatchDenoiser.save_streams."""
    return int(_lib.lib().crispy_ns_stream_state_size())


class MultiDenoiser:
    """n independent DenoiseStates over several GPUs of one box, driven from this one process
    (crispy_ns_multi_*: contiguous blocks of streams per device, one host thread per device, no exchange)."""

    def __init__(self, n_streams: int, devices=None, model: Optional[Model] = None):
        self.n_streams = int(n_streams)
        devs = list(range(device_count())) if devices is None else [int(d) for d in devices]
        arr = (C.c_int * len(devs))(*devs)
        self._model = model
        self._h = C.c_void_p()
        check(_lib.lib().crispy_ns_multi_create(model._h if model else None, arr, len(devs), n_streams, C.byref(self._h)))

    @property
    def ranges(self):
        """[(device, first_stream, n_streams), ...] -- the partition (== shard.stream_block)."""
        L = _lib.lib()
        out = []
        for i in range(L.crispy_ns_multi_n_devices(self._h)):
            d, f, n = C.c_int(), C.c_int(), C.c_int()
            check(L.crispy_ns_multi_stream_range(self._h, i, C.byref(d), C.byref(f), C.byref(n)))
            out.append((d.value, f.value, n.value))
        return out

    def reset(self) -> None:
        check(_lib.lib().crispy_ns_multi_reset(self._h))

    def process_streams_host(self, x, *, unit_scale: bool = True, volume: float = 1.0, drop_first_frame: bool = False,
                             out=None, vad=None, out_i16: bool = False, app=None, mix_stereo_i16: bool = False,
                             first_call: bool = True):
        """As BatchDenoiser.process_streams_host over all n_streams rows; returns when every device is done."""
        import torch
        xt = torch.as_tensor(x)
        if xt.is_cuda or xt.dim() != 2 or xt.stride(1) != 1 or xt.shape[0] != self.n_streams:
            raise CrispyNsError("process_streams_host needs a host [n_streams, n_samples] tensor")
        n_frames = xt.shape[1] // FRAME_SIZE
        flags = 0
        if xt.dtype == torch.int16:
            flags |= IN_I16
        elif xt.dtype != torch.float32:
            raise CrispyNsError("process_streams_host input must be float32 or int16")
        if unit_scale:
            flags |= UNIT_SCALE
        if drop_first_frame:
            flags |= DROP_FIRST_FRAME
        n_out_frames = n_frames - (1 if (drop_first_frame and first_call) else 0)
        if mix_stereo_i16:
            flags |= MIX_STEREO_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE, 2), dtype=torch.int16)
            out_stride = out.stride(0) // 2
        else:
            if out_i16:
                flags |= OUT_I16
            if out is None:
                out = torch.zeros((self.n_streams, n_out_frames * FRAME_SIZE), dtype=torch.int16 if out_i16 else torch.float32)
            out_stride = out.stride(0)
        if vad is None:
            vad = torch.zeros((self.n_streams, n_frames), dtype=torch.float32)
        app_ptr, app_stride = None, 0
        if app is not None:
            app = torch.as_tensor(app)
            app_ptr, app_stride = app.data_ptr(), app.stride(0)
        check(_lib.lib().crispy_ns_multi_process_streams_host(self._h, xt.data_ptr(), out.data_ptr(), vad.data_ptr(), app_ptr,
                                                              n_frames, xt.stride(0), out_stride, vad.stride(0), app_stride,
                                                              flags, volume))
        return out, vad

    def __del__(self):
        try:
            if self._h:
                _lib.lib().crispy_ns_multi_destroy(self._h)
        except Exception:
            pass


def measure_fp32(device: int = 0) -> dict:
    """Register-resident FP32 bursts on every SM: {'ffma_tflops': fused multiply-add throughput,
    'unfused_tmacs': rounded product + rounded add pairs per second / 1e12}."""
    a, b = C.c_double(), C.c_double()
    check(_lib.lib().crispy_ns_measure_fp32(device, C.byref(a), C.byref(b)))
    return {"ffma_tflops": a.value, "unfused_tmacs": b.value}


class RnnNoiseProcessor:
    """audio.rs:202-315: per-sample operator around DenoiseState (frame assembly, x32768, /32768,
    clamp, volume, first frame dropped, linear resampling on either side)."""

    def __init__(self, input_rate: float, output_rate: float, volume: float,
                 model: Optional[Model] = None, device: int = 0):
        if abs(input_rate - 48000.0) >= 1.0:  # audio.rs:217-221
            self.input_resampler: Optional[LinearResampler] = LinearResampler(input_rate, 48000.0)
            effective = 48000.0
        else:
            self.input_resampler = None
            effective = float(input_rate)
        self.max_output_len = int(effective)
        self.denoise = DenoiseState.new(model, device)
        self.input_buf: deque = deque()
        self.output_buf: deque = deque()
        self.resample_pos = 0.0
        self.input_rate = effective
        self.output_rate = float(output_rate)
        self.volume = min(max(float(volume), 0.0), 1.0)
        self.first_frame = True

    def push_sample(self, sample: float):
        """Returns None or the list of newly denoised samples (audio.rs:242-295)."""
        todo = []
        if self.input_resampler is not None:
            self.input_resampler.process_sample(sample, todo.append)
        else:
            todo.append(np.float32(sample))
        acc = []
        for s in todo:
            if len(self.input_buf) >= self.max_output_len:
                self.input_buf.popleft()
            self.input_buf.append(s)
            if len(self.input_buf) >= FRAME_SIZE:
                frame = np.array([self.input_buf.popleft() for _ in range(FRAME_SIZE)], dtype=np.float32)
                frame *= np.float32(32768.0)
                out = np.zeros(FRAME_SIZE, dtype=np.float32)
                self.denoise.process_frame(out, frame)
                out = np.clip(out / np.float32(32768.0), -1.0, 1.0).astype(np.float32) * np.float32(self.volume)
                if self.first_frame:
                    self.first_frame = False
                    continue
                for o in out:
                    if len(self.output_buf) >= self.max_output_len:
                        self.output_buf.popleft()
                    self.output_buf.append(o)
                acc.extend(out.tolist())
        return acc or None

    def next_sample(self) -> float:
        """audio.rs:297-314: linear interpolation of output_buf toward the device rate."""
        if len(self.output_buf) < 2:
            return 0.0
        step = self.input_rate / self.output_rate
        while self.resample_pos >= 1.0:
            self.output_buf.popleft()
            self.resample_pos -= 1.0
            if len(self.output_buf) < 2:
                return 0.0
        s0, s1 = self.output_buf[0], self.output_buf[1]
        frac = np.float32(self.resample_pos)
        self.resample_pos += step
        return float(np.float32(s0 + (s1 - s0) * frac))


# ---- f3: WAV PCM16 -----------------------------------------------------------------------------------
def wav_write_pcm16(path: str, interleaved: np.ndarray, channels: int = 2, sample_rate: int = SAMPLE_RATE) -> None:
    a = np.ascontiguousarray(interleaved, dtype=np.int16).reshape(-1)
    if a.size % channels:
        raise CrispyNsError("Left and right channel length mismatch")  # recording.rs:103
    check(_lib.lib().crispy_ns_wav_write_pcm16(path.encode(), a.ctypes.data, a.size // channels, channels, sample_rate))


def denoise_wav_files(paths_in, paths_out, *, model: Optional[Model] = None, device: int = 0, volume: float = 1.0,
                      drop_first_frame: bool = False):
    """Finished recordings in, denoised dual-mono recordings out (crispy_ns_denoise_wav_files): 48 kHz PCM16 files
    as the recorder writes them (recording.rs:83-99); channel 0 is denoised (commands/transcription.rs:310-312) and
    written to both channels through the recorder's quantiser (recording.rs:108-110).  Returns each file's mean VAD."""
    n = len(paths_in)
    if n != len(paths_out) or n == 0:
        raise CrispyNsError("denoise_wav_files needs as many output as input paths (at least one)")
    pin = (C.c_char_p * n)(*[os.fsencode(p) for p in paths_in])
    pout = (C.c_char_p * n)(*[os.fsencode(p) for p in paths_out])
    vad = (C.c_float * n)()
    check(_lib.lib().crispy_ns_denoise_wav_files(model._h if model else None, device, pin, pout, n,
                                                 DROP_FIRST_FRAME if drop_first_frame else 0, volume, vad))
    return [float(v) for v in vad]


def wav_read_pcm16(path: str):
    n, ch, sr = C.c_int64(), C.c_int(), C.c_int()
    check(_lib.lib().crispy_ns_wav_read_pcm16(path.encode(), None, 0, C.byref(n), C.byref(ch), C.byref(sr)))
    a = np.empty(n.value * ch.value, dtype=np.int16)
    check(_lib.lib().crispy_ns_wav_read_pcm16(path.encode(), a.ctypes.data, a.size, C.byref(n), C.byref(ch), C.byref(sr)))
    return a.reshape(-1, ch.value), sr.value
