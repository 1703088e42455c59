"""crispy_b200 -- B200-native (sm_100a) drop-in for the RNNoise noise-suppression path of
sleep3r/crispy (nnnoiseless::DenoiseState behind src-tauri/src/audio.rs:268).

The product is crispy_b200/libcrispy_ns.so (hand-written CUDA + the C ABI of include/crispy_ns.h);
this package is the thin host mirror of the reference's interface.  No CPU fallback exists.
"""
from .denoise import (FRAME_SIZE, SAMPLE_RATE, BatchDenoiser, DenoiseState, LinearResampler, Model,  # noqa: F401
                      RnnNoiseProcessor, MultiDenoiser, denoise_wav_files, device_count, downmix_mono, linear_resample, measure_fp32, resample_audio, resample_host, sinc_needed, sinc_resample, sinc_resample_chunk, stream_state_size, wav_read_pcm16, wav_write_pcm16)
from ._lib import CrispyNsError  # noqa: F401
