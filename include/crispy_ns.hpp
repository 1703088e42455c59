// crispy_ns.hpp -- C++17 host layer above the C ABI of libcrispy_ns.so (include/crispy_ns.h).
//
// The reference's host code on this path is Rust (src-tauri/src/audio.rs, recording.rs); this image has no Rust
// toolchain, so the compiled host side a native caller uses is this header (the same shape as the Rust shim in
// bindings/rust/ns_gpu.rs, which cannot be built here).  It mirrors the reference's operator interface for the
// path -- same names, argument meaning and error behaviour -- so tests/cpp/host_mirror_test.cpp reads like the
// reference's own unit tests (audio.rs:1040-1096, recording.rs:406-520):
//
//   crispy::DenoiseState::new_() / process_frame(out, in)        nnnoiseless surface at audio.rs:4, :203, :229, :268
//   crispy::LinearResampler                                      audio.rs:73-134
//   crispy::RnnNoiseProcessor::{new_, push_sample, next_sample}  audio.rs:202-315
//   crispy::WavWriter::{new_, write_samples, finalize}           recording.rs:78-127
//   crispy::resample_audio                                       recording.rs:13-39 (many buffers at once)
//   crispy::BatchDenoiser / MultiDenoiser / denoise_wav_files    the batched surface BASELINE.json's north_star adds
//
// Header-only; needs nothing but the C header and -lcrispy_ns.  All arithmetic of the denoiser runs in the library's
// sm_100a kernels; there is no CPU fallback (without a CUDA device the constructors throw crispy::Error with
// CRISPY_NS_ENODEV).  What stays on the host is what the reference also does per sample around process_frame:
// frame assembly, the wrapper's scalings and the two streaming linear interpolators.  Those follow the reference
// operation for operation in float / double, and the products that feed an addition are kept from being contracted
// into fused multiply-adds (unfused_lerp), so a build with -march=native gives the same bits as the Rust code.
#ifndef CRISPY_NS_HPP
#define CRISPY_NS_HPP

#include <cmath>
#include <cstdint>
#include <cstring>
#include <deque>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "crispy_ns.h"

namespace crispy {

constexpr std::size_t FRAME_SIZE = CRISPY_NS_FRAME_SIZE;  // nnnoiseless::FRAME_SIZE (audio.rs:4)
constexpr std::size_t SAMPLE_RATE = 48000;                // recording.rs:8
constexpr std::size_t CHANNELS = 2;                       // recording.rs:9

// A failed library call: code() is the CRISPY_NS_E* value, what() the library's thread-local message.  The Rust side
// returns Result<_, String> (recording.rs) or panics (nnnoiseless asserts); here both are this exception.
class Error : public std::runtime_error {
 public:
  Error(int code, const std::string &msg) : std::runtime_error(msg), code_(code) {}
  int code() const noexcept { return code_; }

 private:
  int code_;
};

namespace detail {
inline void check(int rc) {
  if (rc != CRISPY_NS_OK) throw Error(rc, crispy_ns_last_error());
}
// f32 `clamp` of the Rust standard library: NaN stays NaN
inline float clampf(float x, float lo, float hi) { return x < lo ? lo : (x > hi ? hi : x); }
// a + (b - a) * t with the product rounded before the addition, whatever -ffp-contract / -march say
inline float unfused_lerp(float a, float b, float t) {
  float p = (b - a) * t;
#if defined(__GNUC__) && (defined(__x86_64__) || defined(__i386__))
  __asm__ volatile("" : "+x"(p));
#elif defined(__GNUC__) && defined(__aarch64__)
  __asm__ volatile("" : "+w"(p));
#else
  volatile float q = p;
  p = q;
#endif
  return a + p;
}
// Rust's `f32 as i16`: toward zero, saturating, NaN -> 0
inline std::int16_t f32_as_i16(float v) {
  if (!(v == v)) return 0;
  if (v >= 32767.0f) return 32767;
  if (v <= -32768.0f) return -32768;
  return (std::int16_t)(std::int32_t)v;
}
// Rust's `f32 as usize`
inline std::size_t f32_as_usize(float v) {
  if (!(v > 0.0f)) return 0;
  if (v >= 18446744073709551616.0f) return ~(std::size_t)0;
  return (std::size_t)v;
}
}  // namespace detail

inline int device_count() { return crispy_ns_device_count(); }

// Per-stream suppression controls (crispy_ns_controls): a floor on the applied band gains and a voice gate with hold.
// Value-initialised, they are off.  The setters throw crispy::Error for a value out of range or NaN.
using Controls = crispy_ns_controls;

// The six int8 layers of the recurrent network.  nnnoiseless embeds its weights in the crate; here they are data
// (crispy_ns_model_*): a CRNSMDL1 / rnnoise-nu blob, or seeded synthetic weights of the same topology.
class Model {
 public:
  static Model synthetic(std::uint64_t seed = 0) {
    crispy_ns_model *m = nullptr;
    detail::check(crispy_ns_model_synthetic(seed, &m));
    return Model(m);
  }
  static Model from_bytes(const void *blob, std::size_t len) {
    crispy_ns_model *m = nullptr;
    detail::check(crispy_ns_model_from_bytes(blob, len, &m));
    return Model(m);
  }
  std::vector<std::uint8_t> to_bytes() const {
    std::size_t n = 0;
    detail::check(crispy_ns_model_to_bytes(h_, nullptr, 0, &n));
    std::vector<std::uint8_t> b(n);
    detail::check(crispy_ns_model_to_bytes(h_, b.data(), b.size(), &n));
    return b;
  }
  // CRISPY_NS_SUM_* | CRISPY_NS_BIQUAD_F32 (crispy_ns.h): the arithmetic the handles created from this model follow
  void set_numerics(std::uint32_t numerics) { detail::check(crispy_ns_model_set_numerics(h_, numerics)); }
  std::uint32_t numerics() const { return crispy_ns_model_numerics(h_); }
  Model(Model &&o) noexcept : h_(std::exchange(o.h_, nullptr)) {}
  Model &operator=(Model &&o) noexcept {
    if (this != &o) {
      crispy_ns_model_destroy(h_);
      h_ = std::exchange(o.h_, nullptr);
    }
    return *this;
  }
  Model(const Model &) = delete;
  Model &operator=(const Model &) = delete;
  ~Model() { crispy_ns_model_destroy(h_); }
  const crispy_ns_model *get() const { return h_; }

 private:
  explicit Model(crispy_ns_model *h) : h_(h) {}
  crispy_ns_model *h_;
};

// nnnoiseless::DenoiseState as audio.rs uses it: `Box<DenoiseState<'static>>` (audio.rs:203) from
// `DenoiseState::new()` (:229), `process_frame(&mut out[..], &in[..]) -> f32` (:268).
class DenoiseState {
 public:
  static constexpr std::size_t FRAME_SIZE = crispy::FRAME_SIZE;

  // audio.rs:229.  model == nullptr: the built-in default ($CRISPY_NS_WEIGHTS, else synthetic seed 0).  nnnoiseless'
  // new() cannot fail; this one needs a CUDA device and throws Error(CRISPY_NS_ENODEV) without one.
  static std::unique_ptr<DenoiseState> new_(const Model *model = nullptr, int device = 0) {
    crispy_ns_state *h = nullptr;
    detail::check(crispy_ns_create(model ? model->get() : nullptr, device, &h));
    return std::unique_ptr<DenoiseState>(new DenoiseState(h));
  }
  // audio.rs:268: 480 f32 in 16-bit scale in and out; returns the VAD probability (the reference discards it).
  float process_frame(float *output, std::size_t output_len, const float *input, std::size_t input_len) {
    if (input_len != FRAME_SIZE || output_len != FRAME_SIZE)  // upstream: assert_eq!(input.len(), FRAME_SIZE)
      throw std::invalid_argument("process_frame needs two 480-sample frames");
    float vad = 0.f;
    detail::check(crispy_ns_process_frame(h_, output, input, &vad));
    return vad;
  }
  template <class Out, class In>
  float process_frame(Out &output, const In &input) {
    return process_frame(output.data(), output.size(), input.data(), input.size());
  }
  void reset() { detail::check(crispy_ns_reset(h_)); }  // a fresh state, as the model switch at audio.rs:955-965 builds
  void set_controls(const Controls &c) { detail::check(crispy_ns_set_controls(h_, &c)); }
  Controls controls() {
    Controls c{};
    detail::check(crispy_ns_get_controls(h_, &c));
    return c;
  }
  DenoiseState(const DenoiseState &) = delete;
  DenoiseState &operator=(const DenoiseState &) = delete;
  ~DenoiseState() { crispy_ns_destroy(h_); }

 private:
  explicit DenoiseState(crispy_ns_state *h) : h_(h) {}
  crispy_ns_state *h_;
};

// audio.rs:73-134, field for field (f64 positions, f32 samples).
class LinearResampler {
 public:
  LinearResampler(float input_rate, float output_rate) : input_rate_(input_rate), output_rate_(output_rate) {}
  static LinearResampler new_(float input_rate, float output_rate) { return LinearResampler(input_rate, output_rate); }

  std::pair<float, float> rates() const { return {input_rate_, output_rate_}; }

  void set_rates(float input_rate, float output_rate) {  // audio.rs:97-105: the state restarts with the rates
    input_rate_ = input_rate;
    output_rate_ = output_rate;
    last_sample_ = 0.0f;
    has_last_ = false;
    input_pos_ = 0.0;
    next_output_pos_ = 0.0;
  }

  template <class Emit>
  void process_sample(float sample, Emit &&emit) {  // audio.rs:108-133
    if (std::fabs(input_rate_ - output_rate_) < 1.0f) {
      emit(sample);
      return;
    }
    if (!has_last_) {
      last_sample_ = sample;
      has_last_ = true;
      input_pos_ = 0.0;
      next_output_pos_ = 0.0;
      return;
    }
    input_pos_ += 1.0;
    const double step = (double)(input_rate_ / output_rate_);  // the quotient is an f32 first
    while (next_output_pos_ <= input_pos_) {
      const float t = detail::clampf((float)(next_output_pos_ - (input_pos_ - 1.0)), 0.0f, 1.0f);
      emit(detail::unfused_lerp(last_sample_, sample, t));
      next_output_pos_ += step;
    }
    last_sample_ = sample;
  }

 private:
  float input_rate_, output_rate_;
  float last_sample_ = 0.0f;
  bool has_last_ = false;
  double input_pos_ = 0.0, next_output_pos_ = 0.0;
};

// audio.rs:202-315: the per-sample operator around DenoiseState -- frame assembly, x32768, /32768, clamp, volume,
// first frame dropped, linear interpolation on either side.
class RnnNoiseProcessor {
 public:
  RnnNoiseProcessor(float input_rate, float output_rate, float volume, const Model *model = nullptr, int device = 0)
      : denoise_(DenoiseState::new_(model, device)) {
    if (std::fabs(input_rate - 48000.0f) >= 1.0f) {  // audio.rs:217-225
      input_resampler_.emplace(input_rate, 48000.0f);
      input_rate_ = 48000.0f;
    } else {
      input_rate_ = input_rate;
    }
    max_output_len_ = detail::f32_as_usize(input_rate_);
    output_rate_ = output_rate;
    volume_ = detail::clampf(volume, 0.0f, 1.0f);
  }
  static RnnNoiseProcessor new_(float input_rate, float output_rate, float volume) {
    return RnnNoiseProcessor(input_rate, output_rate, volume);
  }

  // audio.rs:242-295: nullopt, or the samples denoised by this push
  std::optional<std::vector<float>> push_sample(float sample) {
    scratch_.clear();
    if (input_resampler_)
      input_resampler_->process_sample(sample, [this](float s) { scratch_.push_back(s); });
    else
      scratch_.push_back(sample);

    std::vector<float> output_accumulator;
    for (float s : scratch_) {
      if (input_buf_.size() >= max_output_len_ && !input_buf_.empty()) input_buf_.pop_front();
      input_buf_.push_back(s);
      if (input_buf_.size() >= FRAME_SIZE) {
        float input_frame[FRAME_SIZE], output_frame[FRAME_SIZE] = {};
        for (std::size_t i = 0; i < FRAME_SIZE; i++) {
          input_frame[i] = input_buf_.front() * 32768.0f;
          input_buf_.pop_front();
        }
        denoise_->process_frame(output_frame, FRAME_SIZE, input_frame, FRAME_SIZE);
        if (first_frame_) {  // audio.rs:275-278
          first_frame_ = false;
          continue;
        }
        for (std::size_t i = 0; i < FRAME_SIZE; i++) {
          const float out = detail::clampf(output_frame[i] / 32768.0f, -1.0f, 1.0f) * volume_;
          if (output_buf_.size() >= max_output_len_ && !output_buf_.empty()) output_buf_.pop_front();
          output_buf_.push_back(out);
          output_accumulator.push_back(out);
        }
      }
    }
    if (output_accumulator.empty()) return std::nullopt;
    return output_accumulator;
  }

  // audio.rs:297-314: the playback side pulls samples at the device rate
  float next_sample() {
    if (output_buf_.size() < 2) return 0.0f;
    const double step = (double)input_rate_ / (double)output_rate_;
    while (resample_pos_ >= 1.0) {
      output_buf_.pop_front();
      resample_pos_ -= 1.0;
      if (output_buf_.size() < 2) return 0.0f;
    }
    const float s0 = output_buf_[0], s1 = output_buf_[1];
    const float frac = (float)resample_pos_;
    resample_pos_ += step;
    return detail::unfused_lerp(s0, s1, frac);
  }

  float volume() const { return volume_; }
  std::size_t buffered_output() const { return output_buf_.size(); }

 private:
  std::unique_ptr<DenoiseState> denoise_;
  std::deque<float> input_buf_, output_buf_;
  std::vector<float> scratch_;
  double resample_pos_ = 0.0;
  float input_rate_ = 48000.0f, output_rate_ = 48000.0f, volume_ = 1.0f;
  bool first_frame_ = true;
  std::size_t max_output_len_ = 48000;
  std::optional<LinearResampler> input_resampler_;
};

// Many independent recordings at once (north_star `process_streams`): n_streams rows of n_frames * 480 samples,
// `stride` samples apart, host pointers (pinned memory from host_alloc lets the copies overlap the kernels).  The
// arithmetic of RnnNoiseProcessor::push_sample (audio.rs:261-278) is fused into the kernels' loads and stores.  The
// DenoiseStates persist across calls, so a long recording can be fed in pieces.
class BatchDenoiser {
 public:
  explicit BatchDenoiser(int n_streams, const Model *model = nullptr, int device = 0) : n_streams_(n_streams) {
    detail::check(crispy_ns_batch_create(model ? model->get() : nullptr, device, n_streams, &h_));
  }
  BatchDenoiser(const BatchDenoiser &) = delete;
  BatchDenoiser &operator=(const BatchDenoiser &) = delete;
  ~BatchDenoiser() { crispy_ns_batch_destroy(h_); }

  int n_streams() const { return n_streams_; }
  // unit-scale f32 in and out; vad (n_streams x n_frames, may be null) receives the voice-activity probabilities
  void process_streams(const float *input, float *output, float *vad, int n_frames, std::int64_t stride,
                       float volume = 1.0f, bool drop_first_frame = false) {
    const std::uint32_t flags = (std::uint32_t)CRISPY_NS_UNIT_SCALE | (drop_first_frame ? (std::uint32_t)CRISPY_NS_DROP_FIRST_FRAME : 0u);
    detail::check(crispy_ns_process_streams_host(h_, input, output, vad, nullptr, n_frames, stride, stride,
                                                 vad ? n_frames : 0, 0, flags, volume));
  }
  // PCM16 in and out (what the recorder stores, recording.rs:101-121): half the bytes on the host link
  void process_streams_pcm16(const std::int16_t *input, std::int16_t *output, float *vad, int n_frames,
                             std::int64_t stride) {
    detail::check(crispy_ns_process_streams_host(h_, input, output, vad, nullptr, n_frames, stride, stride,
                                                 vad ? n_frames : 0, 0, CRISPY_NS_IN_I16 | CRISPY_NS_OUT_I16, 1.0f));
  }
  // recorder path (commands/recording.rs:260-264 + recording.rs:108-110): mic denoised + app raw -> clamp ->
  // interleaved dual-mono PCM16 (out_pcm16: n_streams rows of 2 * n_frames * 480 samples, 2 * stride apart)
  void process_and_mix(const float *mic, const float *app, std::int16_t *out_pcm16, int n_frames, std::int64_t stride) {
    detail::check(crispy_ns_process_streams_host(h_, mic, out_pcm16, nullptr, app, n_frames, stride, stride, 0, stride,
                                                 CRISPY_NS_UNIT_SCALE | CRISPY_NS_MIX_STEREO_I16, 1.0f));
  }
  std::vector<std::uint8_t> save_state() {
    std::vector<std::uint8_t> b(crispy_ns_batch_state_size(h_));
    detail::check(crispy_ns_batch_save_state(h_, b.data(), b.size()));
    return b;
  }
  void load_state(const std::vector<std::uint8_t> &b) { detail::check(crispy_ns_batch_load_state(h_, b.data(), b.size())); }
  void reset() { detail::check(crispy_ns_batch_reset(h_)); }

  // Streams that advance independently: row i of input / output / vad (n_frames per row) is batch stream streams[i];
  // every other stream is left as it was.  Unit-scale f32, host pointers, synchronous.
  void process_streams_subset(const std::vector<int> &streams, const float *input, float *output, float *vad,
                              int n_frames, std::int64_t stride, float volume = 1.0f) {
    detail::check(crispy_ns_process_streams_subset_host(h_, streams.data(), (int)streams.size(), input, output, vad,
                                                        nullptr, n_frames, stride, stride, vad ? n_frames : 0, 0,
                                                        CRISPY_NS_UNIT_SCALE, volume));
  }
  // fresh DenoiseStates for the listed streams (ordered before the next call; cuda_stream waits for it)
  void reset_streams(const std::vector<int> &streams, void *cuda_stream = nullptr) {
    detail::check(crispy_ns_batch_reset_streams(h_, streams.data(), (int)streams.size(), cuda_stream));
  }
  // one record of crispy_ns_stream_state_size() bytes per listed stream; loads into any stream of any batch
  std::vector<std::uint8_t> save_streams(const std::vector<int> &streams) {
    std::vector<std::uint8_t> b(streams.size() * crispy_ns_stream_state_size());
    detail::check(crispy_ns_batch_save_streams(h_, streams.data(), (int)streams.size(), b.data(), b.size()));
    return b;
  }
  void load_streams(const std::vector<int> &streams, const std::vector<std::uint8_t> &b) {
    detail::check(crispy_ns_batch_load_streams(h_, streams.data(), (int)streams.size(), b.data(), b.size()));
  }
  // controls[i] for streams[i]; ordered as reset_streams
  void set_controls(const std::vector<int> &streams, const std::vector<Controls> &controls, void *cuda_stream = nullptr) {
    if (controls.size() != streams.size()) throw Error(CRISPY_NS_EINVAL, "set_controls: one Controls per stream");
    detail::check(crispy_ns_batch_set_controls(h_, streams.data(), (int)streams.size(), controls.data(), cuda_stream));
  }
  std::vector<Controls> controls(const std::vector<int> &streams) {
    std::vector<Controls> c(streams.size());
    detail::check(crispy_ns_batch_get_controls(h_, streams.data(), (int)streams.size(), c.data()));
    return c;
  }
  crispy_ns_batch *get() { return h_; }

 private:
  crispy_ns_batch *h_ = nullptr;
  int n_streams_;
};

// The same batch over several GPUs of the box from this one process (crispy_ns_multi_*: contiguous blocks of streams
// per device, one host thread per device inside the library, nothing exchanged between devices).
class MultiDenoiser {
 public:
  MultiDenoiser(int n_streams, const std::vector<int> &devices, const Model *model = nullptr) {
    detail::check(crispy_ns_multi_create(model ? model->get() : nullptr, devices.data(), (int)devices.size(), n_streams, &h_));
  }
  MultiDenoiser(const MultiDenoiser &) = delete;
  MultiDenoiser &operator=(const MultiDenoiser &) = delete;
  ~MultiDenoiser() { crispy_ns_multi_destroy(h_); }

  struct Range {
    int device, first_stream, n_streams;
  };
  std::vector<Range> ranges() const {
    std::vector<Range> r((std::size_t)crispy_ns_multi_n_devices(h_));
    for (std::size_t i = 0; i < r.size(); i++)
      detail::check(crispy_ns_multi_stream_range(h_, (int)i, &r[i].device, &r[i].first_stream, &r[i].n_streams));
    return r;
  }
  void process_streams(const float *input, float *output, float *vad, int n_frames, std::int64_t stride,
                       float volume = 1.0f) {
    detail::check(crispy_ns_multi_process_streams_host(h_, input, output, vad, nullptr, n_frames, stride, stride,
                                                       vad ? n_frames : 0, 0, CRISPY_NS_UNIT_SCALE, volume));
  }
  void process_streams_pcm16(const std::int16_t *input, std::int16_t *output, int n_frames, std::int64_t stride) {
    detail::check(crispy_ns_multi_process_streams_host(h_, input, output, nullptr, nullptr, n_frames, stride, stride, 0, 0,
                                                       CRISPY_NS_IN_I16 | CRISPY_NS_OUT_I16, 1.0f));
  }
  void reset() { detail::check(crispy_ns_multi_reset(h_)); }
  // global stream ids; synchronous
  void set_controls(const std::vector<int> &streams, const std::vector<Controls> &controls) {
    if (controls.size() != streams.size()) throw Error(CRISPY_NS_EINVAL, "set_controls: one Controls per stream");
    detail::check(crispy_ns_multi_set_controls(h_, streams.data(), (int)streams.size(), controls.data()));
  }
  std::vector<Controls> controls(const std::vector<int> &streams) {
    std::vector<Controls> c(streams.size());
    detail::check(crispy_ns_multi_get_controls(h_, streams.data(), (int)streams.size(), c.data()));
    return c;
  }

 private:
  crispy_ns_multi *h_ = nullptr;
};

// recording.rs:78-127: the recorder's 48 kHz stereo PCM16 writer.  new_ creates the file (an unwritable path fails
// there, as hound::WavWriter::create does), write_samples quantises and interleaves, finalize writes the RIFF sizes.
class WavWriter {
 public:
  static WavWriter new_(const std::string &output_path) {
    if (crispy_ns_wav_write_pcm16(output_path.c_str(), nullptr, 0, (int)CHANNELS, (int)SAMPLE_RATE) != CRISPY_NS_OK)
      throw Error(CRISPY_NS_EIO, std::string("Failed to create WAV writer: ") + crispy_ns_last_error());
    return WavWriter(output_path);
  }
  void write_samples(const std::vector<float> &left, const std::vector<float> &right) {
    write_samples(left.data(), left.size(), right.data(), right.size());
  }
  void write_samples(const float *left, std::size_t n_left, const float *right, std::size_t n_right) {
    if (n_left != n_right) throw Error(CRISPY_NS_EINVAL, "Left and right channel length mismatch");  // recording.rs:103
    pcm_.reserve(pcm_.size() + 2 * n_left);
    for (std::size_t i = 0; i < n_left; i++) {  // recording.rs:108-110
      pcm_.push_back(detail::f32_as_i16(detail::clampf(left[i], -1.0f, 1.0f) * 32767.0f));
      pcm_.push_back(detail::f32_as_i16(detail::clampf(right[i], -1.0f, 1.0f) * 32767.0f));
    }
  }
  // already quantised interleaved stereo, e.g. the output of BatchDenoiser::process_and_mix
  void write_interleaved(const std::int16_t *lr, std::size_t n_frames) { pcm_.insert(pcm_.end(), lr, lr + 2 * n_frames); }
  const std::string &output_path() const { return path_; }
  std::string finalize() && {
    if (crispy_ns_wav_write_pcm16(path_.c_str(), pcm_.data(), (std::int64_t)(pcm_.size() / CHANNELS), (int)CHANNELS,
                                  (int)SAMPLE_RATE) != CRISPY_NS_OK)
      throw Error(CRISPY_NS_EIO, std::string("Failed to finalize WAV: ") + crispy_ns_last_error());
    return std::move(path_);
  }

 private:
  explicit WavWriter(std::string p) : path_(std::move(p)) {}
  std::string path_;
  std::vector<std::int16_t> pcm_;
};

struct WavData {
  std::vector<std::int16_t> interleaved;
  int channels = 0, sample_rate = 0;
  std::int64_t n_frames = 0;
};
// what the tests read back with hound::WavReader (recording.rs:441-452); the chunk walk of get_wav_duration
inline WavData wav_read_pcm16(const std::string &path) {
  WavData w;
  detail::check(crispy_ns_wav_read_pcm16(path.c_str(), nullptr, 0, &w.n_frames, &w.channels, &w.sample_rate));
  w.interleaved.resize((std::size_t)(w.n_frames * w.channels));
  detail::check(crispy_ns_wav_read_pcm16(path.c_str(), w.interleaved.data(), (std::int64_t)w.interleaved.size(), &w.n_frames,
                                         &w.channels, &w.sample_rate));
  return w;
}

// recording.rs:13-39 `resample_audio(samples, from_rate, to_rate)` on the device, for n_streams buffers of one length
// at once (row-major in and out); bit-identical to the recorder's loop.
inline std::vector<float> resample_audio(const std::vector<float> &samples, std::size_t from_rate, std::size_t to_rate,
                                         int n_streams = 1, int device = 0) {
  if (n_streams < 1 || samples.size() % (std::size_t)n_streams) throw std::invalid_argument("resample_audio: ragged rows");
  const std::int64_t n_in = (std::int64_t)(samples.size() / (std::size_t)n_streams);
  const std::int64_t n_out = crispy_ns_resample_audio_count(n_in, (int)from_rate, (int)to_rate);
  std::vector<float> out((std::size_t)(n_out * n_streams));
  if (n_out)
    detail::check(crispy_ns_resample_host(device, samples.data(), out.data(), n_streams, n_in, n_in, n_out, (int)from_rate,
                                          (int)to_rate, 2));
  return out;
}

// Front end for recordings that are not at 48 kHz: the reference's LinearResampler (audio.rs:217-221) or, with `sinc`,
// the windowed-sinc kernel (north_star item 4).  Row-major [n_streams][n_in] in, [n_streams][n_out] out.
inline std::vector<float> resample_to_48k(const std::vector<float> &input, int n_streams, int input_rate, bool sinc,
                                          int device = 0) {
  if (n_streams < 1 || input.size() % (std::size_t)n_streams) throw std::invalid_argument("resample_to_48k: ragged rows");
  const std::int64_t n_in = (std::int64_t)(input.size() / (std::size_t)n_streams);
  const std::int64_t n_out = sinc ? crispy_ns_sinc_resample_count(input_rate, 48000, n_in)
                                  : crispy_ns_linear_resample_count((float)input_rate, 48000.0f, n_in);
  std::vector<float> out((std::size_t)(n_out * n_streams));
  if (n_out)
    detail::check(crispy_ns_resample_host(device, input.data(), out.data(), n_streams, n_in, n_in, n_out, input_rate, 48000,
                                          sinc ? 1 : 0));
  return out;
}

// Finished recordings (recording.rs:83-99 files) in, denoised dual-mono files out; returns each file's mean VAD.
inline std::vector<float> denoise_wav_files(const std::vector<std::string> &paths_in, const std::vector<std::string> &paths_out,
                                            const Model *model = nullptr, int device = 0, bool drop_first_frame = false,
                                            float volume = 1.0f) {
  if (paths_in.size() != paths_out.size() || paths_in.empty())
    throw std::invalid_argument("denoise_wav_files needs as many output as input paths (at least one)");
  std::vector<const char *> pin, pout;
  for (const auto &p : paths_in) pin.push_back(p.c_str());
  for (const auto &p : paths_out) pout.push_back(p.c_str());
  std::vector<float> vad(paths_in.size());
  detail::check(crispy_ns_denoise_wav_files(model ? model->get() : nullptr, device, pin.data(), pout.data(), (int)pin.size(),
                                            drop_first_frame ? (std::uint32_t)CRISPY_NS_DROP_FIRST_FRAME : 0u, volume, vad.data()));
  return vad;
}

// pinned host memory for the host-pointer calls
template <class T>
struct PinnedBuffer {
  explicit PinnedBuffer(std::size_t n) : n_(n) {
    void *p = nullptr;
    detail::check(crispy_ns_host_alloc(&p, n * sizeof(T)));
    p_ = static_cast<T *>(p);
  }
  PinnedBuffer(const PinnedBuffer &) = delete;
  PinnedBuffer &operator=(const PinnedBuffer &) = delete;
  ~PinnedBuffer() { crispy_ns_host_free(p_); }
  T *data() { return p_; }
  const T *data() const { return p_; }
  std::size_t size() const { return n_; }
  T &operator[](std::size_t i) { return p_[i]; }

 private:
  T *p_ = nullptr;
  std::size_t n_;
};

}  // namespace crispy
#endif  // CRISPY_NS_HPP
