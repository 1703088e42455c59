// ns_common.h -- constants, table and parameter structs shared by the sm_100a kernels, the host
// library and the host-side SIMT emulation used by the CPU tests.
//
// Domain vocabulary follows the reference path (nnnoiseless::DenoiseState behind
// /root/reference/src-tauri/src/audio.rs:268): frames of 480 samples at 48 kHz, a 960-sample
// analysis window, 481 frequency bins, 22 bands, 42 features, a 1728-sample pitch buffer.
#pragma once
#include <stdint.h>

namespace ns {

constexpr int kFrame = 480;
constexpr int kWindow = 960;
constexpr int kFreq = 481;
constexpr int kBands = 22;
constexpr int kFeatures = 42;
constexpr int kCepsMem = 8;
constexpr int kDeltaCeps = 6;
constexpr int kPitchMin = 60;
constexpr int kPitchMax = 768;
constexpr int kPitchBuf = 1728;
constexpr int kGroupThreads = 128;   // threads cooperating on one frame's spectra

// ---- pipeline geometry ---------------------------------------------------------------------------
// A call is cut into chunks of <= chunk_cap frames.  Per chunk and stream the engine keeps, in HBM:
//   hp  : the high-passed signal, kHist samples of history + chunk*480 new samples (f32)
//   tab : per frame, the pitch candidate table remove_doubling's serial decision walks (kTabWords)
//   rec : per frame, the small record passed between phases (kRecFloats)
//   spec: per frame, the spectra X and P (K3 -> K5)
//   featq: per (16-stream group, frame), the 42 features pre-split for the tensor pipe (K3b -> K4)
constexpr int kHist = 1440;          // >= 1248 (pitch_buf history) and a multiple of 480
constexpr int kLpLen = 864;          // pitch_buf downsampled by 2
constexpr int kLpStride = 872;       // padded row of the per-frame downsampled buffers
constexpr int kMaxK = 15;            // remove_doubling examines T0/k for k = 1..15
constexpr int kTabWords = 48;
//   word 0      : T0 | n_k << 16      (n_k = candidates present, k = 1..n_k)
//   word 1      : unused
//   word 2+3(k-1): T_k | pitch_index_k << 16 ; g_k (f32 bits) ; pitch_gain_k (f32 bits)
constexpr int kRecFloats = 148;      // a multiple of 4: K5 stages the record with 16-byte bulk copies
constexpr int kRecPitchIndex = 0;    // int bits
constexpr int kRecSilence = 1;       // int bits
constexpr int kRecPitchGain = 2;
constexpr int kRecVad = 3;
constexpr int kRecExp = 4;           // 22 (normalised band correlation)
constexpr int kRecCeps = 26;         // 22 (DCT of log band energy, offsets applied)
constexpr int kRecTail = 48;         // 7: features[34..40]
constexpr int kRecGatePrev = 55;     // the voice gate's output gain G of the previous frame (K4 -> K5)
constexpr int kRecGRaw = 56;         // 22: band gains as the RNN emits them (the pitch filter uses these)
constexpr int kRecG = 78;            // 22: band gains after the 0.6*lastg smoothing
constexpr int kRecEx = 100;          // 22: band energy of the frame
constexpr int kRecEp = 122;          // 22: band energy of the pitch-lagged window
constexpr int kRecGate = 144;        // the voice gate's output gain G of this frame (K4 -> K5)
static_assert(kRecGate + 1 <= kRecFloats && kRecFloats % 4 == 0, "record overflow");
constexpr int kSpecStride = 482;     // complex bins per stored spectrum (481 used); per frame: X then P

struct alignas(8) cf {
  float x, y;
};
struct alignas(16) f4 {
  float x, y, z, w;
};

// ---- per-stream persistent state (the fields of nnnoiseless::DenoiseState), one block of
// kStateFloats f32 per stream in HBM.
constexpr int kStHist = 0;                        // 1440: last high-passed samples (pitch_buf + analysis_mem)
constexpr int kStSynth = kStHist + kHist;         // 2x480: synthesis_mem, double buffered: a chunk reads copy
                                                  //        synth_sel and writes the other (its runs are concurrent)
constexpr int kStCeps = kStSynth + 2 * kFrame;    // 176 : cepstral_mem[8][22]
constexpr int kStLastG = kStCeps + 176;           // 22  : lastg
constexpr int kStHVad = kStLastG + 22;            // 24  : vad_gru_state
constexpr int kStHNoise = kStHVad + 24;           // 48  : noise_gru_state
constexpr int kStHDen = kStHNoise + 48;           // 96  : denoise_gru_state
constexpr int kStHp = kStHDen + 96;               // 2   : mem_hp_x (f32, as upstream)
constexpr int kStLastGain = kStHp + 2;            // 1
constexpr int kStLastPeriod = kStLastGain + 1;    // 1 (int bits)
constexpr int kStMemId = kStLastPeriod + 1;       // 1 (int bits)
constexpr int kStFrameCount = kStMemId + 1;       // 1 (int bits, informational)
// per-stream suppression controls (crispy_ns_controls) and the voice gate's carry.  Every field is encoded so that a
// zeroed row -- a fresh, reset or pre-controls stream -- means no floor and an open gate.
constexpr int kStCtlMinGain = kStFrameCount + 1;  // 1   : floor on the applied band gains; 0 = none
constexpr int kStCtlGateThr = kStCtlMinGain + 1;  // 1   : VAD threshold; 0 = every frame voiced = gate off
constexpr int kStCtlGateHold = kStCtlGateThr + 1; // 1   : frames the gate stays open after a voiced frame (int bits)
constexpr int kStCtlGateGain = kStCtlGateHold + 1;// 1   : output gain while closed (moot while the threshold is 0)
constexpr int kStGateLeft = kStCtlGateGain + 1;   // 1   : hold frames left (int bits)
constexpr int kStGateShut = kStGateLeft + 1;      // 1   : 1 if the previous frame's G was a closed gate's (int bits)
constexpr int kStGateShutGain = kStGateShut + 1;  // 1   : that G (the gate gain in force then)
constexpr int kStateFloats = 2784;                // padded to a multiple of 32 floats
static_assert(kStGateShutGain + 1 <= kStateFloats, "state layout overflow");

// ---- per-frame debug taps (optional), mirrors oracle rno_debug
constexpr int kDbgFeatures = 0;
constexpr int kDbgGains = 42;
constexpr int kDbgEx = 64;
constexpr int kDbgEp = 86;
constexpr int kDbgExp = 108;
constexpr int kDbgPitchGain = 130;
constexpr int kDbgVad = 131;
constexpr int kDbgPitchIndex = 132;  // stored as float
constexpr int kDbgSilence = 133;
constexpr int kDbgGRaw = 136;        // 22: band gains as the RNN emitted them (what the pitch filter compares Exp with)
constexpr int kDbgFloats = 160;

// ---- constant tables, generated on the host in f64 and copied to shared memory per CTA
struct Tables {
  cf w480[480];          // exp(-2 pi i k/480)
  cf w960[244];          // exp(-2 pi i k/960), k <= 240
  float win[480];        // Vorbis power-complementary half window
  float dct[484];        // dct_table[j*22+i] = cos((j+.5) i pi/22) (* sqrt(.5) for i == 0)
  float tansig[204];     // tanh(0.04 i) rounded to 6 decimals, i <= 200
  float bin_frac[400];   // j / band_size for bin k inside band interval bin_band[k]
  int32_t bin_band[400]; // band interval index (0..20) of bin k
  int32_t eband[24];     // band edges in bins (eband5ms * 4), 22 used
};

// ---- recurrent core (K4) on the tensor pipe: mma.sync m16n8k16, bf16 x bf16 -> f32.
// One CTA carries 16 streams (the M dimension of one MMA tile).  Every activation vector lives in
// shared memory already split into bf16 hi + bf16 lo (x = hi + lo to 2^-17 relative) and already in
// the MMA A-fragment order, one "k-tile" = 16 consecutive inputs x 16 streams = 32 lanes x 4 words:
//   element (stream row r, input kk) of a k-tile -> lane (r%8)*4 + (kk%8)/2, word (r/8) + 2*(kk/8),
//   halfword kk%2.
// The accumulator (C) fragment of an n-tile of 8 outputs has the same lane/word pattern as half a
// k-tile, so an epilogue lane writes its own activations straight back as the next job's A operand.
// Weights (int8, exact in bf16) are packed on the host as B fragments per (job, k-tile, n-tile):
// 32 lanes x 2 words, lane = n*4 + (kk%8)/2, word kk/8, halfword kk%2.
constexpr int kMmaStreams = 16;
constexpr int kMmaWarps = 8;
constexpr int kMmaThreads = 32 * kMmaWarps;
constexpr int kKtWords = 128;            // 32 lanes x 4 words per k-tile (per hi / lo plane)
// resident k-tiles (segments); the feature k-tiles are double buffered separately
constexpr int kKtDV = 0;                 // [dense 24 | vad state 24]            3 k-tiles
constexpr int kKtDVR = 3;                // [dense 24 | r*h of the vad GRU 24]   3
constexpr int kKtNH = 6;                 // noise state 48                        3
constexpr int kKtNR = 9;                 // r*h of the noise GRU                  3
constexpr int kKtDH = 12;                // denoise state 96                      6
constexpr int kKtDR = 18;                // r*h of the denoise GRU                6
constexpr int kKtResident = 24;
constexpr int kKtF = 24;                 // virtual index of the 3 feature k-tiles (42 features + 6 zeros)
constexpr int kFeatKt = 3;
// per (16-stream group, frame) block K3b hands to K4: hi plane, lo plane, 16 silence flags
constexpr int kFeatBlockWords = 2 * kFeatKt * kKtWords + kMmaStreams;  // 784 words = 3136 B
enum MmaJob : int32_t {
  kJDense = 0,   // input_dense            K = F            N = 24
  kJVadZR = 1,   // vad_gru z | r          K = DV           N = 48
  kJVadC = 2,    // vad_gru candidate      K = DVR          N = 24
  kJNoiseZR = 3, // noise_gru z | r        K = DV, F, NH    N = 96
  kJNoiseC = 4,  // noise_gru candidate    K = DV, F, NR    N = 48
  kJDenZR = 5,   // denoise_gru z | r      K = DV[1..2], NH, F, DH   N = 192
  kJDenC = 6,    // denoise_gru candidate  K = DV[1..2], NH, F, DR   N = 96
  kJOut = 7,     // denoise_output         K = DH           N = 22 (24)
  kJVadOut = 8,  // vad_output             K = DV           N = 1 (8)
  kNumMmaJobs = 9
};
// compile-time shape of every product: its k-tile list (virtual k-tile indices) and n-tile count.
// The kernel unrolls over it (every shared-memory offset becomes an immediate); the host packer
// (ns_host.cpp pack_rnn) walks the same lists.
template <int V>
struct IntC {
  static constexpr int value = V;
};
template <int... KT>
struct KtList {
  static constexpr int n = (int)sizeof...(KT);
};
template <int J>
struct MmaShape;
template <> struct MmaShape<kJDense>   { using Kt = KtList<24, 25, 26>; static constexpr int nnt = 3; };
template <> struct MmaShape<kJVadZR>   { using Kt = KtList<0, 1, 2>; static constexpr int nnt = 6; };
template <> struct MmaShape<kJVadC>    { using Kt = KtList<3, 4, 5>; static constexpr int nnt = 3; };
template <> struct MmaShape<kJNoiseZR> { using Kt = KtList<0, 1, 2, 24, 25, 26, 6, 7, 8>; static constexpr int nnt = 12; };
template <> struct MmaShape<kJNoiseC>  { using Kt = KtList<0, 1, 2, 24, 25, 26, 9, 10, 11>; static constexpr int nnt = 6; };
template <> struct MmaShape<kJDenZR>   { using Kt = KtList<1, 2, 6, 7, 8, 24, 25, 26, 12, 13, 14, 15, 16, 17>; static constexpr int nnt = 24; };
template <> struct MmaShape<kJDenC>    { using Kt = KtList<1, 2, 6, 7, 8, 24, 25, 26, 18, 19, 20, 21, 22, 23>; static constexpr int nnt = 12; };
template <> struct MmaShape<kJOut>     { using Kt = KtList<12, 13, 14, 15, 16, 17>; static constexpr int nnt = 3; };
template <> struct MmaShape<kJVadOut>  { using Kt = KtList<0, 1, 2>; static constexpr int nnt = 1; };
// B fragments of job J start at word MmaOff<J>::w ([i][nt][32 lanes][2 words]); its nnt*8 biases at MmaOff<J>::b
template <int J>
struct MmaOff {
  static constexpr int w = MmaOff<J - 1>::w + MmaShape<J - 1>::Kt::n * MmaShape<J - 1>::nnt * 64;
  static constexpr int b = MmaOff<J - 1>::b + MmaShape<J - 1>::nnt * 8;
};
template <>
struct MmaOff<0> {
  static constexpr int w = 0, b = 0;
};
struct RnnHeader {
  int32_t activation[kNumMmaJobs];  // 0 tanh, 1 sigmoid, 2 relu (of the layer behind each product)
  int32_t n_words;
  int32_t n_bias;
  int32_t pad;
};
constexpr int kMmaWords = MmaOff<kNumMmaJobs>::w;  // 723 B-fragment tiles x 64 words = 46,272
constexpr int kMmaBias = MmaOff<kNumMmaJobs>::b;   // 560
static_assert(kMmaWords == 46272 && kMmaBias == 560, "RNNoise topology");

// ---- launch parameters
enum Flags : uint32_t {
  kFlagInI16 = 1u << 0,       // input samples are int16 (16-bit scale)
  kFlagOutI16 = 1u << 1,      // output samples are int16 (round to nearest, saturate)
  kFlagUnitScale = 1u << 2,   // audio.rs:261-273 wrapper arithmetic: x32768 in, /32768 + clamp + *volume out
  kFlagMixStereoI16 = 1u << 3 // f1: out = interleaved stereo i16 of clamp(dn + app) * 32767 (trunc)
};

// One chunk of one call.  Caller pointers (in/out/vad/app/dbg) address frame 0 of the CALL; the
// kernels add frame0.  Engine pointers (hp/tab/rec) address the chunk's workspace slot.
struct Params {
  const void *in;
  void *out;
  float *vad;             // [n_streams][vad_stride] or null
  const float *app;       // f1: app audio, unit scale, same geometry as out frames; may be null
  float *dbg;             // [n_streams][n_frames_call][kDbgFloats] or null
  float *state;           // [n_streams][kStateFloats]
  float *hp;              // [n_streams][hp_stride]
  uint32_t *tab;          // [n_streams][chunk_cap][kTabWords]
  float *rec;             // [n_streams][chunk_cap][kRecFloats]
  cf *spec;               // [n_streams][chunk_cap][2][kSpecStride]: X and P of every frame
  uint32_t *featq;        // [ceil(n_streams/16)][chunk_cap][kFeatBlockWords]: features as bf16 hi/lo A fragments
  const Tables *tables;
  const RnnHeader *rnn_hdr;
  const uint32_t *rnn_words;
  const float *rnn_bias;
  long long in_stride;    // samples between streams
  long long out_stride;   // samples (mono) or stereo pairs between streams
  long long vad_stride;
  long long app_stride;
  long long hp_stride;    // kHist + chunk_cap*480
  int n_streams;
  int n_frames;           // frames in this chunk
  int frame0;             // index of the chunk's first frame within the call
  int n_frames_call;      // frames in the whole call (debug tap geometry)
  int chunk_cap;
  int synth_sel;          // which synthesis_mem copy this chunk reads (chunk counter & 1)
  int out_frame_offset;   // output frame t is stored at frame slot t + out_frame_offset (skipped if < 0)
  int syn_run;            // K5: consecutive frames of one stream per task (>= 1; the host picks it per chunk)
  uint32_t flags;
  float volume;
};

}  // namespace ns
