/*
 * crispy_ns.h -- C ABI of libcrispy_ns.so: a B200-native (sm_100a) drop-in for the RNNoise
 * noise-suppression path of sleep3r/crispy.
 *
 * What it replaces in the reference (/root/reference/src-tauri/src/...):
 *   - `use nnnoiseless::{DenoiseState, FRAME_SIZE}`                      audio.rs:4
 *   - `DenoiseState::new() -> Box<DenoiseState<'static>>`               audio.rs:203, :229
 *   - `denoise.process_frame(&mut out[..], &in[..]) -> f32 (VAD)`        audio.rs:268
 *   - the wrapper arithmetic around it (x32768, /32768, clamp, volume,
 *     first frame dropped)                                               audio.rs:261-278
 *   - LinearResampler in front of it when the input is not 48 kHz        audio.rs:73-134, :217-221
 *   - the recorder's dual-mono mix + PCM16 quantiser                     commands/recording.rs:260-264,
 *                                                                        recording.rs:101-121
 * plus the batched `process_streams` surface BASELINE.json's north_star adds (many independent
 * recordings at once; streams are independent, so batches shard over GPUs with no exchange).
 *
 * Conventions
 *   - Every function returns 0 on success or a negative CRISPY_NS_E* code; it never throws or
 *     unwinds across the boundary (the reference builds with panic = "abort", Cargo.toml:10-20).
 *     crispy_ns_last_error() returns a thread-local message for the last failure.
 *   - Plain pointers and sizes only.  `void *cuda_stream` is a cudaStream_t (NULL = the legacy
 *     default stream).  Device-pointer entry points are asynchronous on that stream; host-pointer
 *     entry points are synchronous.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with
 *     CRISPY_NS_ENODEV.
 *   - A handle is not thread-safe (the reference guards its DenoiseState with a Mutex,
 *     audio.rs:693); distinct handles are independent.
 */
#ifndef CRISPY_NS_H
#define CRISPY_NS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRISPY_NS_FRAME_SIZE 480 /* nnnoiseless::FRAME_SIZE (audio.rs:4) */

enum {
  CRISPY_NS_OK = 0,
  CRISPY_NS_EINVAL = -1, /* bad argument */
  CRISPY_NS_ENODEV = -2, /* no CUDA device / device index out of range */
  CRISPY_NS_ECUDA = -3,  /* CUDA runtime error (message in crispy_ns_last_error) */
  CRISPY_NS_EMODEL = -4, /* malformed model blob */
  CRISPY_NS_ENOMEM = -5,
  CRISPY_NS_EIO = -6
};

/* flags for the batched calls */
enum {
  CRISPY_NS_IN_I16 = 1u << 0,     /* input samples are int16 (16-bit scale) instead of f32 */
  CRISPY_NS_OUT_I16 = 1u << 1,    /* output samples are int16 in 16-bit scale (round-to-nearest, saturating);
                                     UNIT_SCALE's clamp and `volume` do not apply to this format: a call
                                     with OUT_I16 and volume != 1 is rejected with CRISPY_NS_EINVAL */
  CRISPY_NS_UNIT_SCALE = 1u << 2, /* f32 I/O in [-1,1]: x32768 on load, /32768 + clamp(-1,1) + *volume
                                     on store -- RnnNoiseProcessor::push_sample, audio.rs:261-273.
                                     Without it f32 I/O is in 16-bit scale, as process_frame itself. */
  CRISPY_NS_MIX_STEREO_I16 = 1u << 3, /* output = interleaved stereo PCM16 of clamp(denoised + app):
                                         commands/recording.rs:260-264 + recording.rs:108-110 */
  CRISPY_NS_DROP_FIRST_FRAME = 1u << 8 /* discard the very first output frame of each stream
                                          (audio.rs:275-278); the first call then yields n_frames-1 */
};

typedef struct crispy_ns_model crispy_ns_model; /* the six RNN layers (int8 weights) */
typedef struct crispy_ns_state crispy_ns_state; /* one stream: mirrors nnnoiseless::DenoiseState */
typedef struct crispy_ns_batch crispy_ns_batch; /* n independent streams on one GPU */
typedef struct crispy_ns_multi crispy_ns_multi; /* n independent streams over several GPUs of one box */

int crispy_ns_frame_size(void); /* 480 */
const char *crispy_ns_last_error(void);
int crispy_ns_device_count(void); /* number of CUDA devices, 0 if none */

/* ---- model: nnnoiseless embeds its weights in the crate; they are not redistributable here, so
 * the model is an explicit object.  Blob formats: "CRNSMDL1" binary (DESIGN.md) or the rnnoise-nu
 * text format.  crispy_ns_model_synthetic gives seeded int8 weights of the same topology. ---- */
int crispy_ns_model_synthetic(uint64_t seed, crispy_ns_model **out);
int crispy_ns_model_from_bytes(const void *blob, size_t len, crispy_ns_model **out);
int crispy_ns_model_to_bytes(const crispy_ns_model *m, void *buf, size_t cap, size_t *needed);
void crispy_ns_model_destroy(crispy_ns_model *m);

/* ---- numerics: which float32 arithmetic the pitch path's discrete decisions follow.  The product reproduces one
 * arithmetic bit for bit; which one nnnoiseless itself computes is not pinned (DESIGN.md section 6, points 1 and 4), so
 * the alternatives are a setting of the model, the object that names the reference being matched.
 *   sum order (CRISPY_NS_SUM_MASK): the inner products of pitch_search / remove_doubling (celt_inner_prod,
 *     dual_inner_prod) and the cross-correlations (celt_pitch_xcorr: coarse search, autocorrelation) summed in xiph's
 *     sequential order (0, the default), as four interleaved partial sums ((s0 + s1) + s2) + s3 in the inner products
 *     only (DOT4), or in the cross-correlations as well (DOT4_XCORR);
 *   CRISPY_NS_BIQUAD_F32: the high-pass biquad in f32 arithmetic, every product and sum rounded separately, instead
 *     of f32 state with f64 intermediates as the C computes it.
 * Every handle copies the model's setting when it is created (crispy_ns_create, _batch_create, _multi_create,
 * _denoise_wav_files); changing the model later does not affect it; model == NULL means 0.  The CRNSMDL1 blob does not
 * carry the setting: crispy_ns_model_to_bytes / _from_bytes leave it out, and a model from bytes starts at 0.
 * set_numerics returns CRISPY_NS_EINVAL for a null model, unknown bits or sum order 3.  Builds whose pitch kernel
 * knows only the sequential order (-DNS_PITCH_V7) refuse a nonzero sum order at handle creation (CRISPY_NS_EINVAL).
 * A stream record (crispy_ns_batch_save_streams) carries the batch's numerics; a whole-batch state
 * (crispy_ns_batch_save_state) does not, and is only meaningful in a batch of the same numerics. ---- */
enum {
  CRISPY_NS_SUM_SEQUENTIAL = 0u, /* xiph order: the default */
  CRISPY_NS_SUM_DOT4 = 1u,       /* four partial sums in celt_inner_prod / dual_inner_prod */
  CRISPY_NS_SUM_DOT4_XCORR = 2u, /* DOT4, and in celt_pitch_xcorr as well */
  CRISPY_NS_SUM_MASK = 3u,
  CRISPY_NS_BIQUAD_F32 = 1u << 4 /* biquad in f32 arithmetic, no f64 intermediates, no contraction */
};
int crispy_ns_model_set_numerics(crispy_ns_model *m, uint32_t numerics);
uint32_t crispy_ns_model_numerics(const crispy_ns_model *m);

/* ---- DenoiseState::new (audio.rs:229).  model == NULL selects the built-in default: the blob
 * named by $CRISPY_NS_WEIGHTS if set, else synthetic seed 0. ---- */
int crispy_ns_create(const crispy_ns_model *model, int device, crispy_ns_state **out);
/* ---- DenoiseState::process_frame (audio.rs:268): 480 f32 in 16-bit scale in and out (host
 * pointers); *vad receives the voice-activity probability the reference discards.  Synchronous; the seven
 * kernels of the frame are replayed as a CUDA graph (about 0.1 ms per call on a B200). ---- */
int crispy_ns_process_frame(crispy_ns_state *st, float *out480, const float *in480, float *vad);
int crispy_ns_reset(crispy_ns_state *st); /* fresh DenoiseState (audio.rs:955-965 model switch) */
void crispy_ns_destroy(crispy_ns_state *st);

/* ---- batched process_streams (north_star).  Geometry: stream s, frame t, sample i lives at
 * base + s*stride + t*480 + i (strides in samples; for MIX_STEREO_I16 output, in stereo pairs).
 * State (all of DenoiseState) persists across calls, so a long recording can be fed in chunks. ---- */
int crispy_ns_batch_create(const crispy_ns_model *model, int device, int n_streams, crispy_ns_batch **out);
int crispy_ns_batch_reset(crispy_ns_batch *b);
/* same, as an asynchronous memset on cuda_stream (no device synchronisation) */
int crispy_ns_batch_reset_async(crispy_ns_batch *b, void *cuda_stream);
int crispy_ns_batch_n_streams(const crispy_ns_batch *b);
/* device pointers, asynchronous on cuda_stream.  vad may be NULL.  app (unit-scale f32, same
 * geometry as the output frames) is only read with CRISPY_NS_MIX_STEREO_I16 and may be NULL. */
int crispy_ns_process_streams(crispy_ns_batch *b, const void *d_in, void *d_out, float *d_vad,
                              const float *d_app, int n_frames, int64_t in_stride, int64_t out_stride,
                              int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume,
                              void *cuda_stream);
/* host pointers, synchronous; copies are chunked in time and overlapped with the kernel.  Pinned
 * host memory (crispy_ns_host_alloc) is needed for the overlap to materialise. */
int crispy_ns_process_streams_host(crispy_ns_batch *b, const void *h_in, void *h_out, float *h_vad,
                                   const float *h_app, int n_frames, int64_t in_stride,
                                   int64_t out_stride, int64_t vad_stride, int64_t app_stride,
                                   uint32_t flags, float volume);
/* test hook: as crispy_ns_process_streams, additionally writing per-frame taps
 * ([n_streams][n_frames][crispy_ns_debug_floats()] f32, device pointer). */
int crispy_ns_process_streams_debug(crispy_ns_batch *b, const void *d_in, void *d_out, float *d_vad,
                                    float *d_taps, int n_frames, int64_t in_stride, int64_t out_stride,
                                    uint32_t flags, float volume, void *cuda_stream);
int crispy_ns_debug_floats(void);

/* checkpoint / resume of every stream's DenoiseState (host buffers); the state does not record the batch's numerics
 * and is only meaningful when loaded into a batch of the same numerics */
size_t crispy_ns_batch_state_size(const crispy_ns_batch *b);
int crispy_ns_batch_save_state(crispy_ns_batch *b, void *buf, size_t len);
int crispy_ns_batch_load_state(crispy_ns_batch *b, const void *buf, size_t len);

/* ---- streams that advance independently: calls over a subset of the batch, and reset / checkpoint / resume of
 * single streams (recordings of different lengths sharing slots, live streams that have a frame now, a recording
 * moved to another batch or GPU).  A stream's results do not depend on which other streams share a call.
 *   - streams[i] (host array, distinct ids, each in [0, n_streams)) is the batch stream whose samples are row i of
 *     d_in / d_out / d_vad / d_app; every other stream's DenoiseState is left bit for bit as it was.  The array may
 *     be reused as soon as the call returns.
 *   - Geometry, flags and volume as crispy_ns_process_streams / _host, except that CRISPY_NS_DROP_FIRST_FRAME is
 *     refused (the caller drops a stream's first frame itself).
 *   - Arguments are checked before anything is enqueued: a null handle, n_active outside [0, n_streams], an id out of
 *     range or listed twice, CRISPY_NS_DROP_FIRST_FRAME, or a record of the wrong length or magic give
 *     CRISPY_NS_EINVAL and change no state.  n_active == 0 or n_frames == 0 touches nothing.
 *   - frames_done (crispy_ns_batch_info) counts full-batch frames only: subset calls and per-stream resets and loads
 *     leave it alone.  After any of them a full-batch call with CRISPY_NS_DROP_FIRST_FRAME is refused
 *     (CRISPY_NS_EINVAL) until the next crispy_ns_batch_reset, _reset_async or _load_state.
 *   - Ordering: the state rows are copied on the batch's own streams, after every call already enqueued and before
 *     the next one, whichever CUDA stream that call is made on.  The device call is asynchronous on cuda_stream,
 *     which waits for the call's last kernel; a subset call ends with its pipeline drained.
 * ---- */
int crispy_ns_process_streams_subset(crispy_ns_batch *b, const int *streams, int n_active, const void *d_in,
                                     void *d_out, float *d_vad, const float *d_app, int n_frames,
                                     int64_t in_stride, int64_t out_stride, int64_t vad_stride,
                                     int64_t app_stride, uint32_t flags, float volume, void *cuda_stream);
/* host pointers, synchronous, copies pipelined as in crispy_ns_process_streams_host */
int crispy_ns_process_streams_subset_host(crispy_ns_batch *b, const int *streams, int n_active, const void *h_in,
                                          void *h_out, float *h_vad, const float *h_app, int n_frames,
                                          int64_t in_stride, int64_t out_stride, int64_t vad_stride,
                                          int64_t app_stride, uint32_t flags, float volume);
/* fresh DenoiseState for the listed streams only; asynchronous: ordered after the work already on cuda_stream and
 * every call already enqueued, and before the batch's next call; cuda_stream waits for it */
int crispy_ns_batch_reset_streams(crispy_ns_batch *b, const int *streams, int n, void *cuda_stream);
/* one self-describing record per listed stream (host buffers, synchronous): a 16-byte header ("CRNSSTR1", the state's
 * float count, the batch's numerics) and the stream's DenoiseState -- 11,152 bytes in this build.  A record loads into
 * any stream of any batch of this build with the same numerics (else CRISPY_NS_EINVAL); save_streams needs len >= n
 * records, load_streams exactly n records. */
size_t crispy_ns_stream_state_size(void);
int crispy_ns_batch_save_streams(crispy_ns_batch *b, const int *streams, int n, void *buf, size_t len);
int crispy_ns_batch_load_streams(crispy_ns_batch *b, const int *streams, int n, const void *buf, size_t len);

/* ---- per-stream suppression controls: an attenuation limit and a voice gate.  They act only on what leaves the
 * pipeline: no pitch decision, VAD or recurrent state depends on them.
 *   Attenuation limit: on non-silent frames the band gains applied to the spectrum are max(g, min_gain), where
 *     g = max(g_raw, 0.6 lastg) is the smoothed gain; lastg keeps the unfloored g and the pitch filter uses g_raw.
 *     Silent frames pass through as without it.  The floor changes synthesis_mem.
 *   Voice gate: frame t is voiced if its returned VAD (0 on silent frames) >= gate_threshold.  A voiced frame sets
 *     left = gate_hold and the gate is open; otherwise, if left > 0, left -= 1 and the gate is open; otherwise it is
 *     closed.  G_t = 1 while open, else gate_gain.  Output sample i of frame t is the 16-bit-scale denoised sample
 *     times G_{t-1} + (G_t - G_{t-1}) * ((float)(i + 1) / 480.0f), every operation rounded separately, taken after
 *     the overlap-add and before the output conversion (unit scale, clamp, volume, i16, and the dual-mono mix, whose
 *     app audio is not gated).  The gate never writes synthesis_mem; CRISPY_NS_DROP_FIRST_FRAME drops a gated frame
 *     and the gate still advances.  A fresh stream has G_{-1} = 1.
 *   All zeros (a fresh stream) is no floor and the gate off; gate_gain matters only while gate_threshold > 0.
 * The controls and the gate's carry (left, G of the last frame) belong to the recording in the slot: they are part of
 * the stream's state, so subset calls, stream records and whole-batch states carry them, records saved before the
 * controls existed load with them off, and every reset (crispy_ns_reset, _batch_reset, _reset_async, _reset_streams)
 * turns them off.  Setting the controls keeps the gate's carry: they take effect from the stream's next frame.
 * set_controls is ordered as crispy_ns_batch_reset_streams: after every call already enqueued and before the next one,
 * whichever CUDA stream that call is made on; cuda_stream waits for it.  get_controls is synchronous.  A value out of
 * range or NaN, a null handle or array, or a stream id out of range or listed twice gives CRISPY_NS_EINVAL and changes
 * no state. ---- */
typedef struct {
  float min_gain;        /* [0, 1]; floor on every band gain applied to the spectrum; 0 = no limit (today) */
  float gate_threshold;  /* [0, 1]; a frame is voiced if its VAD >= threshold; 0 = every frame voiced = gate off */
  int32_t gate_hold;     /* [0, 1<<20] frames the gate stays open after the last voiced frame */
  float gate_gain;       /* [0, 1]; output gain while the gate is closed; 0 = mute */
} crispy_ns_controls;
/* controls / out point to n crispy_ns_controls structs, one for the single-stream calls.  The prototypes spell them as void
 * pointers because every prototype of this header uses only scalar, handle and void pointer types, which the Rust
 * shim's extern block (bindings/rust/ns_gpu.rs) is checked against type by type; the shim's methods take the
 * #[repr(C)] struct. */
int crispy_ns_batch_set_controls(crispy_ns_batch *b, const int *streams, int n, const void *controls, void *cuda_stream);
int crispy_ns_batch_get_controls(crispy_ns_batch *b, const int *streams, int n, void *out);
/* the same for the one stream of a crispy_ns_state handle, synchronously */
int crispy_ns_set_controls(crispy_ns_state *st, const void *controls);
int crispy_ns_get_controls(crispy_ns_state *st, void *out);

/* launch geometry + bookkeeping: streams per recurrent-core CTA, frames per engine chunk
 * ($CRISPY_NS_CHUNK_FRAMES overrides the default at batch_create), kernels launched so far,
 * frames processed per stream */
int crispy_ns_batch_info(const crispy_ns_batch *b, int *rnn_streams_per_cta, int *chunk_frames,
                         int64_t *launches, int64_t *frames_done);
/* measurement aid: with profiling enabled every kernel launch is bracketed by CUDA events on the
 * stream it is launched on; profile_read synchronises, returns the summed device time (ms) and the
 * launch count per kernel (index < crispy_ns_kernel_count()) since the last read, and clears them. */
int crispy_ns_kernel_count(void);
const char *crispy_ns_kernel_name(int k);
int crispy_ns_batch_profile(crispy_ns_batch *b, int enable);
int crispy_ns_batch_profile_read(crispy_ns_batch *b, double *ms_total, int64_t *n_launches, int n_kernels);
void crispy_ns_batch_destroy(crispy_ns_batch *b);


/* ---- (e) several GPUs from one process (SURVEY.md 8(e)).  The reference keeps one DenoiseState per stream
 * and no shared mutable state (audio.rs:203), so the n_streams of a multi handle are cut into contiguous blocks
 * of ceil/floor(n_streams / n_devices) streams, device i taking block i (crispy_ns_multi_stream_range); a
 * meeting's mic and app audio share one stream index, so its dual-mono mix never crosses devices.  Each device
 * has its own crispy_ns_batch, weights copy, host thread and CUDA streams; nothing is exchanged between
 * devices (no collective).  The host call has crispy_ns_process_streams_host's geometry over all n_streams
 * rows; it returns when every device has finished. ---- */
int crispy_ns_multi_create(const crispy_ns_model *model, const int *devices, int n_devices, int n_streams,
                           crispy_ns_multi **out);
int crispy_ns_multi_n_devices(const crispy_ns_multi *m);
int crispy_ns_multi_stream_range(const crispy_ns_multi *m, int i, int *device, int *first_stream, int *n_streams);
int crispy_ns_multi_reset(crispy_ns_multi *m);
int crispy_ns_multi_process_streams_host(crispy_ns_multi *m, const void *h_in, void *h_out, float *h_vad,
                                         const float *h_app, int n_frames, int64_t in_stride, int64_t out_stride,
                                         int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume);
/* crispy_ns_batch_set_controls / _get_controls over the multi handle's global stream ids (synchronous) */
int crispy_ns_multi_set_controls(crispy_ns_multi *m, const int *streams, int n, const void *controls);
int crispy_ns_multi_get_controls(crispy_ns_multi *m, const int *streams, int n, void *out);
void crispy_ns_multi_destroy(crispy_ns_multi *m);

/* pinned host memory for the host-pointer path */
int crispy_ns_host_alloc(void **ptr, size_t bytes);
void crispy_ns_host_free(void *ptr);

/* ---- a4 / f2: LinearResampler (audio.rs:73-134), data-parallel on the device.  The output
 * positions depend only on the two rates, so they are tabulated once on the host in f64 exactly as
 * the reference accumulates them; the device then interpolates every (stream, sample) at once and
 * is bit-identical to LinearResampler::process_sample.  n_out = crispy_ns_linear_resample_count. */
int64_t crispy_ns_linear_resample_count(float input_rate, float output_rate, int64_t n_in);
int crispy_ns_linear_resample(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in,
                              int64_t in_stride, int64_t out_stride, float input_rate,
                              float output_rate, void *cuda_stream);

/* ---- the caller's side of the path: the capture callbacks downmix interleaved device frames to mono before
 * RnnNoiseProcessor::push_sample sees them -- f32: sum(frame) / channels (audio.rs:754-755); i16: sum(s / 32768) /
 * channels (audio.rs:816-818); u16: sum((s - 32768) / 32768) / channels (audio.rs:879-884); f32 sums in channel
 * order.  One kernel, bit-identical, bound by HBM.  d_in: [n_streams][n_frames * n_channels] interleaved samples of
 * sample_format (strides in elements), d_out: [n_streams][n_frames] f32 unit scale. */
enum { CRISPY_NS_FMT_F32 = 0, CRISPY_NS_FMT_I16 = 1, CRISPY_NS_FMT_U16 = 2 };
int crispy_ns_downmix_mono(int device, const void *d_in, int sample_format, int n_channels, float *d_out,
                           int n_streams, int64_t n_frames, int64_t in_stride, int64_t out_stride,
                           void *cuda_stream);

/* ---- f2, the app-audio side: resample_audio (recording.rs:13-39), the whole-buffer linear interpolator the recorder
 * applies to captured app audio before it is mixed with the denoised microphone (recording.rs:356-360):
 * ratio = from_rate / to_rate in f64, out[i] = s[j] + (s[j + 1] - s[j]) * (frac as f32) with j = floor(i * ratio),
 * the last sample repeated where j + 1 runs off the end.  Data-parallel and bit-identical on the device (the
 * position of every output is one f64 multiply).  n_out = crispy_ns_resample_audio_count; equal rates copy. */
int64_t crispy_ns_resample_audio_count(int64_t n_in, int from_rate, int to_rate);
int crispy_ns_resample_audio(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in,
                             int64_t in_stride, int64_t out_stride, int from_rate, int to_rate,
                             void *cuda_stream);

/* ---- f2 (BASELINE.json north_star item 4, configs[2]): windowed-sinc 44.1 -> 48 kHz front end,
 * "rubato-equivalent".  The reference's own front end on this path is the linear interpolator above;
 * rubato 0.16.2 (Cargo.lock:4166) is in its tree ahead of transcription
 * (commands/transcription.rs:201-207).  Polyphase form of rubato's synchronous sinc resampler:
 * sinc_len taps (0 = 256), f_cutoff relative to Nyquist (0 = 0.95; scaled by the ratio when
 * downsampling), BlackmanHarris2 window, one tabulated phase per L of the reduced ratio
 * L/M = output_rate/input_rate (L <= 1024), delay-compensated, zeros outside [0, n_in):
 *   out[s][n] = sum_k h[(n*M)%L][k] * in[s][floor(n*M/L) - sinc_len/2 + 1 + k],  n < ceil(n_in*L/M)
 * 441 input samples give exactly one 480-sample frame.  Device pointers, asynchronous. */
int64_t crispy_ns_sinc_resample_count(int input_rate, int output_rate, int64_t n_in);
int crispy_ns_sinc_resample(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in,
                            int64_t in_stride, int64_t out_stride, int input_rate, int output_rate,
                            int sinc_len, float f_cutoff, void *cuda_stream);

/* the same for a recording that does not fit one call: the recording has n_total input samples, d_in[s][0] is its
 * sample in_first and n_in samples are present; outputs first_out .. first_out + n_out (first_out a whole number of
 * periods, i.e. a multiple of L: any multiple of 480 for 44.1 -> 48 kHz) go to d_out[s][0 ..).  Samples outside
 * [0, n_total) count as zeros; crispy_ns_sinc_resample_needed gives the input range the outputs' taps touch.
 * Chunked calls reproduce the whole-recording call bit for bit. */
int crispy_ns_sinc_resample_needed(int input_rate, int output_rate, int sinc_len, int64_t n_total, int64_t first_out,
                                   int64_t n_out, int64_t *in_first, int64_t *n_in);
int crispy_ns_sinc_resample_chunk(int device, const float *d_in, int64_t in_first, int64_t n_in, int64_t n_total,
                                  float *d_out, int64_t first_out, int64_t n_out, int n_streams, int64_t in_stride,
                                  int64_t out_stride, int input_rate, int output_rate, int sinc_len, float f_cutoff,
                                  void *cuda_stream);
/* host-pointer convenience over the two front ends (what the Rust side calls for recordings in RAM):
 * kind 0 = linear (audio.rs:108-133), 1 = windowed sinc (defaults 256 taps, cutoff 0.95), 2 = the recorder's
 * resample_audio (recording.rs:13-39).  Synchronous; h_out must hold crispy_ns_{linear,sinc}_resample_count /
 * crispy_ns_resample_audio_count samples per stream. */
int crispy_ns_resample_host(int device, const float *h_in, float *h_out, int n_streams, int64_t n_in,
                            int64_t in_stride, int64_t out_stride, int input_rate, int output_rate, int kind);

/* ---- f3: RIFF/WAVE PCM16 I/O (recording.rs:83-121 writer; commands/recording.rs:385-460 parser).
 * The reader walks the chunks as get_wav_duration does (unknown chunks skipped, pad bytes honoured), accepts the plain
 * PCM header hound writes for the recorder's spec, fmt chunks of 18 or 40 bytes, WAVE_FORMAT_EXTENSIBLE with the PCM
 * sub-format, and a data size of 0xFFFFFFFF (a writer that could not seek back: the data runs to the end of the
 * file); anything that is not 16-bit PCM is refused with CRISPY_NS_EIO.  Call it with interleaved = NULL first to
 * learn n_frames / channels / sample_rate. */
int crispy_ns_wav_write_pcm16(const char *path, const int16_t *interleaved, int64_t n_frames,
                              int channels, int sample_rate);
int crispy_ns_wav_read_pcm16(const char *path, int16_t *interleaved, int64_t cap_samples,
                             int64_t *n_frames, int *channels, int *sample_rate);


/* ---- f3 end to end: batch-denoise finished recordings.  Every paths_in[i] is a 48 kHz PCM16 RIFF/WAVE file as
 * the recorder writes it (recording.rs:83-99: stereo, both channels carry the same mix); channel 0 is taken
 * (as the transcription reader does, commands/transcription.rs:310-312), denoised with PCM16 on the host link,
 * and written to paths_out[i] as dual-mono stereo PCM16 through the recorder's quantiser
 * (clamp(x,-1,1)*32767 truncated, recording.rs:108-110).  Files may differ in length: all n_files run as one
 * batch, shorter ones are padded with silence internally and written back at their own length.  flags:
 * CRISPY_NS_DROP_FIRST_FRAME mirrors audio.rs:275-278 (the output is then 480 samples shorter).  mean_vad
 * (n_files floats, may be NULL) receives each file's mean voice-activity probability (f4). ---- */
int crispy_ns_denoise_wav_files(const crispy_ns_model *model, int device, const char *const *paths_in,
                                const char *const *paths_out, int n_files, uint32_t flags, float volume,
                                float *mean_vad);

/* ---- measurement aid: a register-resident burst on every SM for ~10 ms.  *ffma_tflops receives the FP32
 * throughput of fused multiply-adds (2 flop each), *unfused_tmacs the rate of rounded-product + rounded-add
 * pairs (10^12 MAC/s), the form the pitch kernel's exactness contract requires.  Either may be NULL. ---- */
int crispy_ns_measure_fp32(int device, double *ffma_tflops, double *unfused_tmacs);

#ifdef __cplusplus
}
#endif
#endif /* CRISPY_NS_H */
