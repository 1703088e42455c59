// ns_rnn_tc5.cuh -- K4 on the fifth-generation tensor cores: the recurrent core (a14: dense -> VAD GRU -> noise GRU ->
// denoise GRU -> dense) of 128 streams per CTA as tcgen05.mma (UTCHMMA) products with every operand where Blackwell
// wants it:
//   * A (activations, 128 streams x K): TENSOR MEMORY.  Lane = stream, 32-bit column c holds the bf16 pair of inputs
//     (2c, 2c + 1); two planes, hi at columns [0, 208) and lo = bf16(x - hi) at [208, 416), so x = hi + lo to 2^-17.
//     The epilogue threads write them with tcgen05.st and the MMA reads them in place (the .ts form: A from TMEM).
//   * B (weights, int8 exact in bf16): SHARED MEMORY, 188.5 KB resident for the whole launch, one block per product in
//     the canonical K-major no-swizzle layout a UMMA shared-memory descriptor addresses (8 x 16 B core matrices).
//   * D (f32 accumulators, 128 x N): TENSOR MEMORY columns [416, 512), read back with tcgen05.ld for the epilogue.
// One frame step is nine rounds.  A tcgen05.mma issued by one thread costs ~77 cycles whatever N <= 128 is
// (scripts/micro/tc5_rate.cu: 77 cycles at N = 16 .. 128, 97 at 192, 128 at 256), so a round is made as wide as the
// 96 accumulator columns allow (z | r of the noise GRU in one round; z, r, candidate of the denoise GRU 96 columns
// each) and takes 2 MMAs (hi and lo plane into the same accumulator) per k-tile of its inputs: 152 MMAs per frame.
// One thread issues the round's MMAs and commits them to an mbarrier; the 512 epilogue threads (four per stream: warp w
// owns the tensor-memory lanes 32 (w % 4) .. + 31 and the column quarter w / 4) wait on it, load their quarter of the
// columns of their stream's row, apply bias / table tanh / GRU algebra in registers (the GRU states themselves stay in
// f32 registers) and store the next products' operands straight back into tensor memory.
// 1,024 streams take 8 CTAs instead of the 64 the warp-level mma.sync core occupies (ns_pipe.cuh rnn_body).
//
// Device-only (no host emulation: tensor memory has no CPU stand-in); parity is checked on the GPU against the oracle
// and against the mma.sync core (tests/test_gpu_parity.py).
#pragma once
#include "ns_common.h"

namespace ns {
namespace tc5 {

constexpr int kStreams = 128;
constexpr int kThreads = 512;   // thread = (stream row m = tid & 127, column quarter hs = tid >> 7)
constexpr int kParts = 4;
constexpr int kColLo = 208;     // first column of the lo plane
constexpr int kColD = 416;      // accumulator columns
constexpr int kTmemCols = 512;
constexpr int kNumRounds = 9;
constexpr int kMaxKt = 14;

// positions of the activation vectors in the A element space (k-tile v = elements 16 v .. 16 v + 15); every vector
// starts a k-tile except the VAD state, which shares k-tiles 0..2 with the dense layer's output
constexpr int kPosDense = 0, kPosVadH = 24, kPosVadR = 48, kPosNoiseH = 80, kPosNoiseR = 128, kPosDenH = 176,
              kPosDenR = 272, kPosFeat = 368;
static_assert(kPosFeat + 48 == 2 * kColLo, "the A planes");

struct Round {
  int n_kt;
  int kt[kMaxKt];
  int n;      // columns of the round (a multiple of 16): quarter h takes columns [h n/4, (h + 1) n/4)
  int boff;   // byte offset of the round's weight block
};
// weight block of a round: [k-tile][K half][n / 8][8 columns][8 inputs] bf16 = n * 32 bytes per k-tile
constexpr Round kRounds[kNumRounds] = {
    {3, {23, 24, 25}, 32, 0},                                                  // 0 input_dense
    {3, {0, 1, 2}, 48, 3072},                                                  // 1 vad z | r
    {4, {0, 1, 3, 4}, 32, 7680},                                               // 2 vad candidate
    {9, {0, 1, 2, 23, 24, 25, 5, 6, 7}, 96, 11776},                            // 3 noise z | r
    {9, {0, 1, 2, 23, 24, 25, 8, 9, 10}, 64, 39424},                           // 4 noise candidate (+ vad_output)
    {14, {1, 2, 5, 6, 7, 23, 24, 25, 11, 12, 13, 14, 15, 16}, 96, 57856},      // 5 denoise z
    {14, {1, 2, 5, 6, 7, 23, 24, 25, 11, 12, 13, 14, 15, 16}, 96, 100864},     // 6 denoise r
    {14, {1, 2, 5, 6, 7, 23, 24, 25, 17, 18, 19, 20, 21, 22}, 96, 143872},     // 7 denoise candidate
    {6, {11, 12, 13, 14, 15, 16}, 32, 186880},                                 // 8 denoise_output
};
constexpr int kWeightBytes = 186880 + 6 * 32 * 32;  // 193,024
constexpr int kBiasPerRound = 96;
constexpr bool rounds_consistent() {
  int off = 0;
  for (int r = 0; r < kNumRounds; r++) {
    if (kRounds[r].boff != off || kRounds[r].n % 16 != 0 || kRounds[r].n > kBiasPerRound || kRounds[r].n > kTmemCols - kColD) return false;
    off += kRounds[r].n_kt * kRounds[r].n * 32;
  }
  return off == kWeightBytes;
}
static_assert(rounds_consistent(), "weight block offsets");

// what column `col` of round `r` computes: layer 0 dense, 1 vad GRU, 2 noise GRU, 3 denoise GRU, 4 output, 5 vad_output;
// gate 0 z, 1 r, 2 candidate; unit index; layer -1 = padding.  Shared by the host packer and (implicitly) the epilogues.
struct ColInfo {
  int layer, gate, unit;
};
inline ColInfo col_info(int r, int col) {
  const int part_n = kRounds[r].n / kParts, h = col / part_n, j = col % part_n;
  switch (r) {
    case 0: return j < 6 ? ColInfo{0, 0, 6 * h + j} : ColInfo{-1, 0, 0};
    case 1: return j < 6 ? ColInfo{1, 0, 6 * h + j} : ColInfo{1, 1, 6 * h + j - 6};
    case 2: return j < 6 ? ColInfo{1, 2, 6 * h + j} : ColInfo{-1, 0, 0};
    case 3: return j < 12 ? ColInfo{2, 0, 12 * h + j} : ColInfo{2, 1, 12 * h + j - 12};
    case 4: return j < 12 ? ColInfo{2, 2, 12 * h + j} : ((h == 0 && j == 12) ? ColInfo{5, 0, 0} : ColInfo{-1, 0, 0});
    case 5: return ColInfo{3, 0, 24 * h + j};
    case 6: return ColInfo{3, 1, 24 * h + j};
    case 7: return ColInfo{3, 2, 24 * h + j};
    default: return (j < 6 && 6 * h + j < 22) ? ColInfo{4, 0, 6 * h + j} : ColInfo{-1, 0, 0};
  }
}

#if defined(__CUDACC__) && !defined(NS_HOST_EMU)

struct Smem {
  alignas(128) unsigned char w[kWeightBytes];
  float bias[kNumRounds * kBiasPerRound];
  float tansig[204];
  alignas(8) unsigned long long mbar;
  unsigned tmem_base;
};
static_assert(sizeof(Smem) <= 227 * 1024, "tcgen05 recurrent core exceeds the shared memory of a CTA");

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

template <int N>
struct TmemIo;
template <>
struct TmemIo<1> {
  static __device__ __forceinline__ void ld(unsigned a, unsigned *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v[0]) : "r"(a));
  }
  static __device__ __forceinline__ void st(unsigned a, const unsigned *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(a), "r"(v[0]));
  }
};
template <>
struct TmemIo<2> {
  static __device__ __forceinline__ void ld(unsigned a, unsigned *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(a));
  }
  static __device__ __forceinline__ void st(unsigned a, const unsigned *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(a), "r"(v[0]), "r"(v[1]));
  }
};
template <>
struct TmemIo<4> {
  static __device__ __forceinline__ void ld(unsigned a, unsigned *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(a));
  }
  static __device__ __forceinline__ void st(unsigned a, const unsigned *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]));
  }
};
template <>
struct TmemIo<8> {
  static __device__ __forceinline__ void ld(unsigned a, unsigned *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(a));
  }
  static __device__ __forceinline__ void st(unsigned a, const unsigned *v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(a), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]));
  }
};
// N consecutive columns in pieces of P columns (every piece starts at a multiple of P columns: callers choose P so)
template <int N, int P>
__device__ __forceinline__ void tmem_ld(unsigned a, unsigned *v) {
  static_assert(N % P == 0, "whole pieces");
#pragma unroll
  for (int i = 0; i < N; i += P) TmemIo<P>::ld(a + i, v + i);
}
template <int N, int P>
__device__ __forceinline__ void tmem_st(unsigned a, const unsigned *v) {
  static_assert(N % P == 0, "whole pieces");
#pragma unroll
  for (int i = 0; i < N; i += P) TmemIo<P>::st(a + i, v + i);
}

// NV values of this thread's stream -> hi / lo bf16 pairs at A position `pos` (pos / 2 a multiple of P) of both planes
template <int NV, int P>
__device__ __forceinline__ void store_act(unsigned lane_base, int pos, const float *v) {
  unsigned hi[NV / 2], lo[NV / 2];
#pragma unroll
  for (int i = 0; i < NV / 2; i++) bf16_split2(v[2 * i], v[2 * i + 1], hi[i], lo[i]);
  tmem_st<NV / 2, P>(lane_base + (unsigned)(pos >> 1), hi);
  tmem_st<NV / 2, P>(lane_base + (unsigned)(kColLo + (pos >> 1)), lo);
}

__device__ __forceinline__ void rnn_tc5_body(const Params &p, Smem &s) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hs = warp >> 2;        // TMEM lane quarter of this warp, column quarter
  const int m = 32 * q + lane;                   // stream row within the CTA
  const int stream = blockIdx.x * kStreams + m;
  const bool live = stream < p.n_streams;
  // ---- weights, biases, tables -> shared memory; tensor memory; the mbarrier
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(p.rnn_words);
    uint4 *dst = reinterpret_cast<uint4 *>(s.w);
    for (int i = tid; i < kWeightBytes / 16; i += kThreads) dst[i] = src[i];
    for (int i = tid; i < kNumRounds * kBiasPerRound; i += kThreads) s.bias[i] = p.rnn_bias[i];
    for (int i = tid; i < 204; i += kThreads) s.tansig[i] = p.tables->tansig[i];
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s.mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the weights, written through the generic proxy, for the MMAs
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const unsigned tbase = s.tmem_base;
  const unsigned lane_base = tbase + ((unsigned)(32 * q) << 16);
  const float *tab = s.tansig;
  const RnnHeader &H = *p.rnn_hdr;
  const int act_dense = H.activation[kJDense], act_vad = H.activation[kJVadC], act_noise = H.activation[kJNoiseC],
            act_den = H.activation[kJDenC], act_out = H.activation[kJOut], act_vadout = H.activation[kJVadOut];
  // ---- recurrent state of this thread's units: vad 6 hs + 0..5, noise 12 hs + 0..11, denoise 24 hs + 0..23,
  //      lastg 6 hs + 0..5 (22 bands: the last quarter owns four)
  float hv[6], hn[12], hd[24], lastg[6];
  {
    const float *st = p.state + (long long)(live ? stream : 0) * kStateFloats;
#pragma unroll
    for (int j = 0; j < 6; j++) hv[j] = live ? st[kStHVad + 6 * hs + j] : 0.f;
#pragma unroll
    for (int j = 0; j < 12; j++) hn[j] = live ? st[kStHNoise + 12 * hs + j] : 0.f;
#pragma unroll
    for (int j = 0; j < 24; j++) hd[j] = live ? st[kStHDen + 24 * hs + j] : 0.f;
#pragma unroll
    for (int j = 0; j < 6; j++) lastg[j] = (live && 6 * hs + j < kBands) ? st[kStLastG + 6 * hs + j] : 0.f;
  }
  // the voice gate (ns_pipe.cuh gate_step) runs on the thread that writes the stream's VAD
  GateState gate = {};
  if (live && hs == 0) gate = gate_load(p.state + (long long)stream * kStateFloats);
  store_act<6, 1>(lane_base, kPosVadH + 6 * hs, hv);
  store_act<12, 2>(lane_base, kPosNoiseH + 12 * hs, hn);
  store_act<24, 4>(lane_base, kPosDenH + 24 * hs, hd);
  if (hs == 0) {  // the padding behind r * h of the VAD GRU (elements 72..79) meets zero weights: it must be finite
    const unsigned zero[4] = {0u, 0u, 0u, 0u};
    tmem_st<4, 4>(lane_base + (unsigned)((kPosVadR + 24) >> 1), zero);
    tmem_st<4, 4>(lane_base + (unsigned)(kColLo + ((kPosVadR + 24) >> 1)), zero);
  }
  // feature words of (16-stream group, frame): K3b's layout (ns_pipe.cuh features_body): pair qq of row r at word widx;
  // quarter hs stores pairs 12 (hs & 1) .. + 11 of plane hs >> 1
  const int row16 = m & 15, fplane = hs >> 1, fhalf = hs & 1;
  const uint32_t *fq_src = p.featq + (long long)(stream >> 4) * p.chunk_cap * kFeatBlockWords;
  unsigned fw[12];
  unsigned silw = 1u;
  auto fetch_features = [&](int t) {  // issued a frame ahead: the loads fly under the previous frame's rounds
    const uint32_t *blk = fq_src + (long long)t * kFeatBlockWords + fplane * (kFeatKt * kKtWords);
#pragma unroll
    for (int i = 0; i < 12; i++) {
      const int qq = 12 * fhalf + i;
      const int widx = ((qq >> 3) * 32 + (row16 & 7) * 4 + (qq & 3)) * 4 + (row16 >> 3) + 2 * ((qq & 7) >> 2);
      fw[i] = live ? __ldg(blk + widx) : 0u;
    }
    silw = live ? __ldg(fq_src + (long long)t * kFeatBlockWords + 2 * kFeatKt * kKtWords + row16) : 1u;
  };
  unsigned parity = 0;
  unsigned err = 0;
  auto round_mma = [&](auto ri_tag) {  // one thread: every k-tile of the round, hi then lo plane, into the accumulator columns
    constexpr Round R = kRounds[decltype(ri_tag)::value];
    const unsigned idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(R.n >> 3) << 17) | ((unsigned)(128 >> 4) << 24);
    const unsigned lbo = (unsigned)(R.n / 8 * 128);
    const unsigned b0 = smem_u32(s.w) + (unsigned)R.boff;
    unsigned first = 1;
#pragma unroll
    for (int i = 0; i < R.n_kt; i++) {
      const unsigned long long bdesc = (unsigned long long)(((b0 + (unsigned)(i * R.n * 32)) & 0x3FFFFu) >> 4) |
                                       ((unsigned long long)(lbo >> 4) << 16) | ((unsigned long long)(128 >> 4) << 32) | (1ull << 46);
#pragma unroll
      for (int plane = 0; plane < 2; plane++) {
        const unsigned a = tbase + (unsigned)(plane * kColLo + 8 * R.kt[i]);
        const unsigned acc = first ? 0u : 1u;
        first = 0;
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tbase + kColD),
            "r"(a), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u));
      }
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&s.mbar)) : "memory");
  };
#ifdef NS_TC5_CLOCKS
  // measurement build: where a frame step's cycles go, seen by the first thread of two warps
  long long tk[6] = {0, 0, 0, 0, 0, 0}, tk_mark = clock64();
#define NS_TC5_TICK(i) do { const long long now_ = clock64(); tk[i] += now_ - tk_mark; tk_mark = now_; } while (0)
#else
#define NS_TC5_TICK(i) do {} while (0)
#endif
  // issue the round (one thread) and wait for its accumulators (everyone)
  auto run_round = [&](auto ri_tag) {
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;");
      round_mma(ri_tag);
    }
    NS_TC5_TICK(0);
    unsigned done = 0;
    for (int spin = 0; spin < (1 << 24) && !done; spin++)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(done)
                   : "r"(smem_u32(&s.mbar)), "r"(parity)
                   : "memory");
    if (!done) err = 1;  // a wedged tensor pipe must not hang the device: results are garbage, the host sees the flag
    parity ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;");
    NS_TC5_TICK(1);
  };
  // NC accumulators of this thread's quarter of the round's columns from column offset c0 of the quarter, scaled:
  // x = (acc + bias) / 256
  auto load_pre = [&](int r, int part_n, int c0, auto nc_tag, float *x) {
    constexpr int NC = decltype(nc_tag)::value;
    unsigned v[NC];
    tmem_ld<NC, (NC % 8 == 0 ? 8 : 4)>(lane_base + (unsigned)(kColD + hs * part_n + c0), v);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const float *b = s.bias + r * kBiasPerRound + hs * part_n + c0;
#pragma unroll
    for (int j = 0; j < NC; j++) x[j] = (__uint_as_float(v[j]) + b[j]) * (1.f / 256);
    NS_TC5_TICK(2);
  };
  auto end_round = [&]() {  // operands stored, accumulators read: the next round may issue
    NS_TC5_TICK(3);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;");
    NS_TC5_TICK(4);
    __syncthreads();
    NS_TC5_TICK(5);
  };

  if (p.n_frames > 0) fetch_features(0);
  for (int t = 0; t < p.n_frames; t++) {
    // features of this frame -> tensor memory; the next frame's are requested right away
    const bool sil = silw != 0u;
    tmem_st<12, 4>(lane_base + (unsigned)(fplane * kColLo + (kPosFeat >> 1) + 12 * fhalf), fw);
    if (t + 1 < p.n_frames) fetch_features(t + 1);
    end_round();
    float vad = 0.f;
    float x[12];
    // 0: input_dense -> dense
    run_round(IntC<0>{});
    load_pre(0, 8, 0, IntC<8>{}, x);
    {
      float y[6];
      activate_n<6>(tab, act_dense, x, y);
      store_act<6, 1>(lane_base, kPosDense + 6 * hs, y);
    }
    end_round();
    // 1: vad z | r
    float zv[6];
    run_round(IntC<1>{});
    load_pre(1, 12, 0, IntC<12>{}, x);
    {
      float rh[6];
#pragma unroll
      for (int j = 0; j < 6; j++) {
        zv[j] = sigmoid_approx(tab, x[j]);
        rh[j] = hv[j] * sigmoid_approx(tab, x[6 + j]);
      }
      store_act<6, 1>(lane_base, kPosVadR + 6 * hs, rh);
    }
    end_round();
    // 2: vad candidate -> vad state
    run_round(IntC<2>{});
    load_pre(2, 8, 0, IntC<8>{}, x);
    activate_n<6>(tab, act_vad, x, x);
#pragma unroll
    for (int j = 0; j < 6; j++) {
      const float hnew = zv[j] * hv[j] + (1.f - zv[j]) * x[j];
      if (!sil) hv[j] = hnew;
    }
    store_act<6, 1>(lane_base, kPosVadH + 6 * hs, hv);
    end_round();
    // 3: noise z | r -> z, r * h
    float zn[12];
    run_round(IntC<3>{});
    load_pre(3, 24, 0, IntC<12>{}, x);
#pragma unroll
    for (int j = 0; j < 12; j++) zn[j] = sigmoid_approx(tab, x[j]);
    load_pre(3, 24, 12, IntC<12>{}, x);
    {
      float rh[12];
#pragma unroll
      for (int j = 0; j < 12; j++) rh[j] = hn[j] * sigmoid_approx(tab, x[j]);
      store_act<12, 2>(lane_base, kPosNoiseR + 12 * hs, rh);
    }
    end_round();
    // 4: noise candidate -> noise state (+ vad_output in column 12 of quarter 0: the VAD state settled in round 2)
    run_round(IntC<4>{});
    load_pre(4, 16, 0, IntC<12>{}, x);
    activate_n<12>(tab, act_noise, x, x);
#pragma unroll
    for (int j = 0; j < 12; j++) {
      const float hnew = zn[j] * hn[j] + (1.f - zn[j]) * x[j];
      if (!sil) hn[j] = hnew;
    }
    store_act<12, 2>(lane_base, kPosNoiseH + 12 * hs, hn);
    if (hs == 0) {
      load_pre(4, 16, 12, IntC<4>{}, x);
      vad = activate(tab, act_vadout, x[0]);
    }
    end_round();
    // 5: denoise z
    float zd[24];
    run_round(IntC<5>{});
#pragma unroll
    for (int c = 0; c < 2; c++) {
      load_pre(5, 24, 12 * c, IntC<12>{}, x);
#pragma unroll
      for (int j = 0; j < 12; j++) zd[12 * c + j] = sigmoid_approx(tab, x[j]);
    }
    end_round();
    // 6: denoise r -> r * h
    run_round(IntC<6>{});
#pragma unroll
    for (int c = 0; c < 2; c++) {
      load_pre(6, 24, 12 * c, IntC<12>{}, x);
      float rh[12];
#pragma unroll
      for (int j = 0; j < 12; j++) rh[j] = hd[12 * c + j] * sigmoid_approx(tab, x[j]);
      store_act<12, 2>(lane_base, kPosDenR + 24 * hs + 12 * c, rh);
    }
    end_round();
    // 7: denoise candidate -> denoise state
    run_round(IntC<7>{});
#pragma unroll
    for (int c = 0; c < 2; c++) {
      load_pre(7, 24, 12 * c, IntC<12>{}, x);
      activate_n<12>(tab, act_den, x, x);
#pragma unroll
      for (int j = 0; j < 12; j++) {
        const float hnew = zd[12 * c + j] * hd[12 * c + j] + (1.f - zd[12 * c + j]) * x[j];
        if (!sil) hd[12 * c + j] = hnew;
      }
      store_act<12, 2>(lane_base, kPosDenH + 24 * hs + 12 * c, hd + 12 * c);
    }
    end_round();
    // 8: denoise_output -> band gains; g = max(g, 0.6 lastg)
    run_round(IntC<8>{});
    load_pre(8, 8, 0, IntC<8>{}, x);
    activate_n<6>(tab, act_out, x, x);
    if (live) {
      float *rec = p.rec + ((long long)stream * p.chunk_cap + t) * kRecFloats;
#pragma unroll
      for (int j = 0; j < 6; j++) {
        if (6 * hs + j < kBands) {
          float graw = 0.f, g = 0.f;
          if (!sil) {
            graw = x[j];
            g = fmaxf(graw, .6f * lastg[j]);
            lastg[j] = g;
          }
          rec[kRecGRaw + 6 * hs + j] = graw;
          rec[kRecG + 6 * hs + j] = g;
        }
      }
      if (hs == 0) {
        const float v = sil ? 0.f : vad;
        rec[kRecVad] = v;
        gate_step(gate, v, rec);
        if (p.vad) p.vad[(long long)stream * p.vad_stride + p.frame0 + t] = v;
      }
    }
    // the next frame's feature store and its end_round() order this round's accumulator reads before the next MMAs
  }
  if (live) {
    float *st = p.state + (long long)stream * kStateFloats;
#pragma unroll
    for (int j = 0; j < 6; j++) st[kStHVad + 6 * hs + j] = hv[j];
#pragma unroll
    for (int j = 0; j < 12; j++) st[kStHNoise + 12 * hs + j] = hn[j];
#pragma unroll
    for (int j = 0; j < 24; j++) st[kStHDen + 24 * hs + j] = hd[j];
#pragma unroll
    for (int j = 0; j < 6; j++)
      if (6 * hs + j < kBands) st[kStLastG + 6 * hs + j] = lastg[j];
    if (hs == 0) gate_save(gate, st);
    if (err && tid == 0) reinterpret_cast<int *>(st)[kStFrameCount] = -1;  // poison the informational frame counter
  }
#ifdef NS_TC5_CLOCKS
  if ((tid == 0 || tid == 480) && blockIdx.x == 0)
    printf("tc5 cycles per frame (thread %d): issue %lld | wait for MMAs %lld | tcgen05.ld + bias %lld | activations + tcgen05.st %lld | "
           "wait::st %lld | barrier %lld\n", tid, tk[0] / p.n_frames, tk[1] / p.n_frames, tk[2] / p.n_frames, tk[3] / p.n_frames,
           tk[4] / p.n_frames, tk[5] / p.n_frames);
#endif
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(kTmemCols));
}

#endif  // __CUDACC__

}  // namespace tc5
}  // namespace ns
