// crispy_ns.cu -- libcrispy_ns.so: the sm_100a kernels' entry points and the C ABI declared in
// include/crispy_ns.h.  No CPU fallback: every compute call needs a CUDA device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <exception>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/crispy_ns.h"
#include "ns_host.h"
#include "ns_pipe.cuh"
#include "ns_pitch7.cuh"
#include "ns_rnn_tc5.cuh"

// ------------------------------------------------------------------------------------------------
// kernels (bodies in ns_pipe.cuh)
// ------------------------------------------------------------------------------------------------
#ifndef NS_PITCH_RUN
#define NS_PITCH_RUN 8
#endif
constexpr int kPitchRun = NS_PITCH_RUN;  // frames of one stream per pitch CTA
// K1 generations: the first (ns_pipe.cuh pitch_body: all 147 x 240 coarse sums in the oracle's order) is the product;
// -DNS_PITCH_V7 builds the second (ns_pitch7.cuh: coarse search filtered on the tensor pipe), which is bit-exact too but
// measured slower on B200 (profiles/r2_pitch.md): legacy HMMA latency and shared-memory wavefronts eat what the
// 147 x 240 sums cost
#ifndef NS_PITCH_V7
#ifdef NS_PITCH_THREADS
constexpr int kPitchThreads = NS_PITCH_THREADS;
#else
constexpr int kPitchThreads = (37 * kPitchRun + 31) / 32 * 32 + 32;
#endif
using PitchShared = ns::PitchSmem<kPitchRun>;
#else
constexpr int kPitchThreads = ns::kP7Threads;
using PitchShared = ns::PitchSmem7<kPitchRun>;
#endif
//  // 37 lag-quads per frame in the coarse search + one helper warp
constexpr int kScanWarps = 4;
#ifndef NS_HP_EXCLUSIVE_MAX_STREAMS
#define NS_HP_EXCLUSIVE_MAX_STREAMS 768
#endif
#ifndef NS_RNN_TC5_MIN_STREAMS
#define NS_RNN_TC5_MIN_STREAMS (1 << 30)  // the tcgen05 recurrent core is opt-in ($CRISPY_NS_RNN=tc5) until measured
#endif

// K0 in its two forms (ns_pipe.cuh): one recursion warp, and parallel in time (one speculating warp + four exact warps).
// The second is the faster kernel (isolated 613 -> 424 us per 32,768 frames) and wins wherever K0 bounds the pipeline
// (small batches, where it also has its SMs to itself); beside the pitch CTAs of a full batch its eight warps cost the
// parallel kernels what its shorter run gives back, so the first form stays there (crispy_ns_batch::hp_par).
// F32: the biquad in f32 arithmetic alone (CRISPY_NS_BIQUAD_F32); the parallel form speculates the f64 expression only
template <bool F32>
__global__ void __launch_bounds__(ns::kHpThreads) ns_highpass_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ns::highpass_body<F32>(p, *reinterpret_cast<ns::HpSmem *>(smem_raw));
}
__global__ void __launch_bounds__(ns::kHpParThreads) ns_highpass_par_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ns::highpass_par_body(p, *reinterpret_cast<ns::HpParSmem *>(smem_raw));
}
// SP: the summation policy of the pitch path's inner products (CRISPY_NS_SUM_*; the second generation knows only 0)
template <int SP>
__global__ void __launch_bounds__(kPitchThreads) ns_pitch_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
#ifndef NS_PITCH_V7
  ns::pitch_body<kPitchRun, kPitchThreads, SP>(p, *reinterpret_cast<PitchShared *>(smem_raw));
#else
  static_assert(SP == 0, "ns_pitch7.cuh sums in the sequential order only");
  ns::pitch_body7<kPitchRun, kPitchThreads>(p, *reinterpret_cast<PitchShared *>(smem_raw));
#endif
}
#ifndef NS_PITCH_V7
constexpr int kPitchPolicies = 3;
#else
constexpr int kPitchPolicies = 1;
#endif
typedef void (*KernelFn)(ns::Params);
static KernelFn pitch_kernel(uint32_t numerics) {
#ifndef NS_PITCH_V7
  switch (numerics & CRISPY_NS_SUM_MASK) {
    case CRISPY_NS_SUM_DOT4: return ns_pitch_kernel<1>;
    case CRISPY_NS_SUM_DOT4_XCORR: return ns_pitch_kernel<2>;
    default: break;
  }
#endif
  return ns_pitch_kernel<0>;
}
static KernelFn highpass_kernel(uint32_t numerics) {
  return (numerics & CRISPY_NS_BIQUAD_F32) ? ns_highpass_kernel<true> : ns_highpass_kernel<false>;
}
__global__ void __launch_bounds__(32 * kScanWarps) ns_pitchscan_kernel(const __grid_constant__ ns::Params p) {
  ns::pitchscan_body(p, kScanWarps);
}
#ifndef NS_SPEC_MINB
#define NS_SPEC_MINB 8  // as NS_SYN_MINB: one resident wave of 8 CTAs per SM
#endif
#ifndef NS_SYN_MINB
#define NS_SYN_MINB 8  // measured on B200: 64 registers + 168 B of spill beat 4 resident CTAs at 119 registers
#endif
__global__ void __launch_bounds__(ns::kGroupThreads, NS_SPEC_MINB) ns_spectrum_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ns::spectrum_body(p, *reinterpret_cast<ns::SpecSmem *>(smem_raw));
}
__global__ void __launch_bounds__(32 * ns::kFeatWarps) ns_features_kernel(const __grid_constant__ ns::Params p) {
  __shared__ ns::FeatSmem sm;
  ns::features_body(p, sm);
}
__global__ void __launch_bounds__(ns::kMmaThreads, 1) ns_rnn_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ns::rnn_body(p, *reinterpret_cast<ns::RnnSmem *>(smem_raw));
}
// the same recurrent core on tcgen05 / tensor memory, 128 streams per CTA (ns_rnn_tc5.cuh)
__global__ void __launch_bounds__(ns::tc5::kThreads, 1) ns_rnn_tc5_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  ns::tc5::rnn_tc5_body(p, *reinterpret_cast<ns::tc5::Smem *>(smem_raw));
}
__global__ void __launch_bounds__(ns::kGroupThreads, NS_SYN_MINB) ns_synthesis_kernel(const __grid_constant__ ns::Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ns::synthesis_body(p, *reinterpret_cast<ns::SpecSmem *>(smem_raw));
}

// Per-stream state rows by index (subset calls, per-stream reset, save / load of single streams): one CTA per row,
// 16-byte accesses coalesced across the row's 11,136 bytes.  Row j of the launch moves src row (ids_on_src ? ids[j] :
// first + j) to dst row (ids_on_src ? first + j : ids[j]); src == null writes zeros.  synthesis_mem (kStSynth) is
// double buffered: dst's copy dst_cur receives src's copy src_cur, and dst's other copy src's other copy
// (keep_stale) or zeros -- the other copy is scratch the next chunk writes before any read.
constexpr int kRowIds = 960;  // ids per launch: the parameter block stays under 4 KB
struct RowArgs {
  float *dst;
  const float *src;
  int first, n, ids_on_src, src_cur, dst_cur, keep_stale;
  int ids[kRowIds];
};
constexpr int kRowVec = ns::kStateFloats / 4;
static_assert(ns::kStateFloats % 4 == 0 && ns::kStSynth % 4 == 0 && ns::kFrame % 4 == 0, "rows move as float4");
__global__ void __launch_bounds__(256) ns_state_rows_kernel(const __grid_constant__ RowArgs a) {
  const int j = blockIdx.x;
  const long long s = a.ids_on_src ? a.ids[j] : a.first + j, d = a.ids_on_src ? a.first + j : a.ids[j];
  const float4 *src = a.src ? reinterpret_cast<const float4 *>(a.src + s * ns::kStateFloats) : nullptr;
  float4 *dst = reinterpret_cast<float4 *>(a.dst + d * ns::kStateFloats);
  constexpr int syn0 = ns::kStSynth / 4, syn_len = ns::kFrame / 4;
  for (int q = threadIdx.x; q < kRowVec; q += blockDim.x) {
    int from = q;
    bool zero = src == nullptr;
    if (q >= syn0 && q < syn0 + 2 * syn_len) {
      const int copy = (q - syn0) / syn_len, off = (q - syn0) % syn_len;
      const int src_copy = copy == a.dst_cur ? a.src_cur : 1 - a.src_cur;
      from = syn0 + src_copy * syn_len + off;
      if (copy != a.dst_cur && !a.keep_stale) zero = true;
    }
    dst[q] = zero ? make_float4(0.f, 0.f, 0.f, 0.f) : src[from];
  }
}

// crispy_ns_batch_set_controls: thread j writes the four control words (ns_common.h kStCtl*) of state row ids[j]; the
// gate's carry (left, previous G) is left alone, so new controls take effect from the next frame on
constexpr int kCtlIds = 192;  // entries per launch: the parameter block stays under 4 KB
struct ControlArgs {
  float *state;
  int n;
  int ids[kCtlIds];
  uint32_t words[kCtlIds][4];
};
__global__ void __launch_bounds__(kCtlIds) ns_set_controls_kernel(const __grid_constant__ ControlArgs a) {
  const int j = threadIdx.x;
  if (j >= a.n) return;
  uint32_t *row = reinterpret_cast<uint32_t *>(a.state + (long long)a.ids[j] * ns::kStateFloats);
  static_assert(ns::kStCtlGateThr == ns::kStCtlMinGain + 1 && ns::kStCtlGateHold == ns::kStCtlMinGain + 2 &&
                    ns::kStCtlGateGain == ns::kStCtlMinGain + 3, "the four control words are contiguous");
  for (int w = 0; w < 4; w++) row[ns::kStCtlMinGain + w] = a.words[j][w];
}

// a4/f2: out[s][n] = in[s][idx[n]-1] + (in[s][idx[n]] - in[s][idx[n]-1]) * frac[n], no FMA
// contraction so the result is bit-identical to LinearResampler::process_sample (audio.rs:125-129).
__global__ void __launch_bounds__(256) ns_linear_resample_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                 const int32_t *__restrict__ idx, const float *__restrict__ frac,
                                                                 long long n_out, long long in_stride, long long out_stride,
                                                                 int vec_store) {
  // four consecutive outputs per thread and trip (their (index, fraction) entries are one 16-byte load each; the table
  // is shared by every stream and stays in L2), a CTA covers one contiguous tile of a row
  const int s = blockIdx.y;
  const float *src = in + (long long)s * in_stride;
  float *dst = out + (long long)s * out_stride;
  for (long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; n < n_out;
       n += (long long)gridDim.x * blockDim.x * 4) {
    if (n + 4 <= n_out) {
      const int4 i4 = __ldg(reinterpret_cast<const int4 *>(idx + n));
      const float4 f4v = __ldg(reinterpret_cast<const float4 *>(frac + n));
      const float l0 = src[i4.x - 1], c0 = src[i4.x], l1 = src[i4.y - 1], c1 = src[i4.y], l2 = src[i4.z - 1], c2 = src[i4.z],
                  l3 = src[i4.w - 1], c3 = src[i4.w];
      const float o0 = __fadd_rn(l0, __fmul_rn(__fsub_rn(c0, l0), f4v.x)), o1 = __fadd_rn(l1, __fmul_rn(__fsub_rn(c1, l1), f4v.y)),
                  o2 = __fadd_rn(l2, __fmul_rn(__fsub_rn(c2, l2), f4v.z)), o3 = __fadd_rn(l3, __fmul_rn(__fsub_rn(c3, l3), f4v.w));
      if (vec_store) {
        *reinterpret_cast<float4 *>(dst + n) = make_float4(o0, o1, o2, o3);
      } else {
        dst[n] = o0, dst[n + 1] = o1, dst[n + 2] = o2, dst[n + 3] = o3;
      }
    } else {
      for (long long m = n; m < n_out; m++) {
        const int i = idx[m];
        const float last = src[i - 1], cur = src[i];
        dst[m] = __fadd_rn(last, __fmul_rn(__fsub_rn(cur, last), frac[m]));
      }
    }
  }
}

// The capture callbacks' downmix (audio.rs:754-755, :816-818, :879-884): mono = sum over the frame's channels, in
// channel order, of the sample brought to unit scale, divided by the channel count; f32 adds, IEEE division.
template <typename T>
__device__ __forceinline__ float ns_unit_sample(T v);
template <>
__device__ __forceinline__ float ns_unit_sample<float>(float v) { return v; }
template <>
__device__ __forceinline__ float ns_unit_sample<int16_t>(int16_t v) { return __fmul_rn((float)v, 1.0f / 32768.0f); }  // a power of two: the same value as the division
template <>
__device__ __forceinline__ float ns_unit_sample<uint16_t>(uint16_t v) { return __fmul_rn(__fsub_rn((float)v, 32768.0f), 1.0f / 32768.0f); }
template <typename T>  // any channel count, any alignment: one frame per thread and trip
__global__ void __launch_bounds__(256) ns_downmix_kernel(const T *__restrict__ in, float *__restrict__ out, int n_channels,
                                                         long long n_frames, long long in_stride, long long out_stride) {
  const T *src = in + (long long)blockIdx.y * in_stride;
  float *dst = out + (long long)blockIdx.y * out_stride;
  const float div = (float)n_channels;
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_frames; n += (long long)gridDim.x * blockDim.x) {
    const T *f = src + n * n_channels;
    float sum = 0.f;
    for (int c = 0; c < n_channels; c++) sum = __fadd_rn(sum, ns_unit_sample<T>(f[c]));
    dst[n] = __fdiv_rn(sum, div);
  }
}
// Stereo, 16-byte aligned rows: a thread turns 32 bytes of interleaved input (two 16-byte loads: 4 f32 frames or 8
// PCM16 frames) into 16 or 32 bytes of output per trip, kDownmixTrips trips in flight per thread; a CTA covers one
// contiguous tile of a row, so every warp reads and writes whole 128-byte lines.  The kernel is bound by HBM.
constexpr int kDownmixTrips = 4;
template <typename T>
__global__ void __launch_bounds__(256) ns_downmix_stereo_kernel(const T *__restrict__ in, float *__restrict__ out, long long n_frames,
                                                                long long in_stride, long long out_stride) {
  constexpr int FR = 16 / (int)sizeof(T);  // frames per thread and trip: 4 (f32) or 8 (PCM16)
  const T *src = in + (long long)blockIdx.y * in_stride;
  float *dst = out + (long long)blockIdx.y * out_stride;
  const long long tile0 = (long long)blockIdx.x * (256 * FR * kDownmixTrips);
  uint4 raw[kDownmixTrips][2];
#pragma unroll
  for (int u = 0; u < kDownmixTrips; u++) {  // all loads first
    const long long n = tile0 + ((long long)u * 256 + threadIdx.x) * FR;
    if (n + FR <= n_frames) {
      const uint4 *q = reinterpret_cast<const uint4 *>(src + 2 * n);
      raw[u][0] = __ldg(q);
      raw[u][1] = __ldg(q + 1);
    }
  }
#pragma unroll
  for (int u = 0; u < kDownmixTrips; u++) {
    const long long n = tile0 + ((long long)u * 256 + threadIdx.x) * FR;
    if (n + FR <= n_frames) {
      const T *v = reinterpret_cast<const T *>(&raw[u][0]);
      float o[FR];
#pragma unroll
      for (int k = 0; k < FR; k++)
        o[k] = __fmul_rn(__fadd_rn(__fadd_rn(0.f, ns_unit_sample<T>(v[2 * k])), ns_unit_sample<T>(v[2 * k + 1])), .5f);  // / 2, exactly
#pragma unroll
      for (int k = 0; k < FR; k += 4) *reinterpret_cast<float4 *>(dst + n + k) = make_float4(o[k], o[k + 1], o[k + 2], o[k + 3]);
    } else {
      for (long long m = n; m < n_frames; m++)  // the row's last, partial vector
        dst[m] = __fmul_rn(__fadd_rn(__fadd_rn(0.f, ns_unit_sample<T>(src[2 * m])), ns_unit_sample<T>(src[2 * m + 1])), .5f);
    }
  }
}

// f2, app audio: resample_audio (recording.rs:13-39).  src_pos = i * ratio in f64, j = floor, frac = src_pos - j;
// out[i] = s[j] + (s[j+1] - s[j]) * (frac as f32) without FMA contraction, or s[j] on the last sample.
__global__ void __launch_bounds__(256) ns_resample_audio_kernel(const float *__restrict__ in, float *__restrict__ out, long long n_in,
                                                                long long n_out, long long in_stride, long long out_stride, double ratio,
                                                                int vec_store) {
  const int s = blockIdx.y;
  const float *src = in + (long long)s * in_stride;
  float *dst = out + (long long)s * out_stride;
  auto one = [&](long long n) -> float {
    const double pos = __dmul_rn((double)n, ratio);
    const long long j = (long long)floor(pos);
    const float frac = (float)(pos - (double)j);
    const float s1 = src[j];
    return (j + 1 < n_in) ? __fadd_rn(s1, __fmul_rn(__fsub_rn(src[j + 1], s1), frac)) : s1;
  };
  for (long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; n < n_out;
       n += (long long)gridDim.x * blockDim.x * 4) {
    if (n + 4 <= n_out && vec_store) {
      *reinterpret_cast<float4 *>(dst + n) = make_float4(one(n), one(n + 1), one(n + 2), one(n + 3));
    } else {
      for (long long m = n; m < n_out && m < n + 4; m++) dst[m] = one(m);
    }
  }
}

// f2 (north_star item 4): windowed-sinc polyphase resampler.  out[n] = sum_k h[(n*M)%L][k] *
// in[floor(n*M/L) - half + 1 + k].  A CTA covers T*Q consecutive outputs of one stream (T a multiple
// of L, so thread t keeps one phase for all of its Q outputs and holds the tap h[k][phase] in a
// register across them); the input span is staged once in shared memory, zero-filled outside
// [0, n_in).  One fmaf per tap in ascending k per output: bit-identical to the oracle's scalar loop.
template <int Q>
__global__ void __launch_bounds__(1024) ns_sinc_resample_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                const float *__restrict__ hT,  // [sinc_len][L]
                                                                long long n_total, long long in_first, long long in_end,
                                                                long long first_out, long long n_out, long long in_stride,
                                                                long long out_stride, int L, int M, int sinc_len,
                                                                int span) {
  // the recording has n_total input samples; in[0] is its sample in_first and samples [in_first, in_end) are present;
  // outputs first_out .. first_out + n_out (first_out a multiple of L) are written to out[0 .. n_out).  A partial last
  // tile stages a full tile's span: what lies beyond the caller's window feeds no stored output and is not read.
  extern __shared__ float xs[];
  const int T = blockDim.x, t = threadIdx.x;
  const long long n0 = first_out + (long long)blockIdx.x * T * Q;  // multiple of L
  const long long base0 = n0 / L * M - sinc_len / 2 + 1;           // recording index of xs[0]
  const float *src = in + (long long)blockIdx.y * in_stride - in_first;
  for (int i = t; i < span; i += T) {
    const long long g = base0 + i;
    xs[i] = (g >= in_first && g < in_end) ? __ldg(src + g) : 0.f;
  }
  __syncthreads();
  const int pos = t * M;  // t < 1024, M < 2^20
  const int phase = pos % L;
  const int rb = pos / L, step = T / L * M;
  float acc[Q];
#pragma unroll
  for (int q = 0; q < Q; q++) acc[q] = 0.f;
  const float *hp = hT + phase;
  const float *xp = xs + rb;
#pragma unroll 4
  for (int k = 0; k < sinc_len; k++) {
    const float h = __ldg(hp + (long long)k * L);
#pragma unroll
    for (int q = 0; q < Q; q++) acc[q] = fmaf(h, xp[q * step + k], acc[q]);
  }
  float *dst = out + (long long)blockIdx.y * out_stride;
#pragma unroll
  for (int q = 0; q < Q; q++) {
    const long long n = n0 + t + (long long)q * T - first_out;
    if (n < n_out) dst[n] = acc[q];
  }
}

// Second generation for upsampling ratios with 2/3 <= M/L < 1 (44.1 -> 48 kHz: 147/160).  The first kernel reads one
// input sample from shared memory per multiply-add, which caps it at a quarter of the FMA rate (it measures 20 %).
// Here a thread owns FOUR ADJACENT outputs u = 4t .. 4t + 3 of a period (and Q periods of them): adjacent outputs look at
// windows that start 0 or 1 sample apart, so sweeping over the INPUT index lets one staged sample feed all four --
// output r meets sample i with its tap k = i - d_r, d_r = window start of r minus that of output 0 (d_r is r or r - 1).
// The taps come from a table laid out in OUTPUT order, hs[k][u] = h[k][(u M) mod L], so the four taps of row k are one
// 16-byte load; row i - d_r is the row loaded d_r steps ago, kept in a four-deep register delay line, and the choice
// between "r steps ago" and "r - 1 steps ago" is one select per r and step (not per period).  Per step: Q 4-byte
// shared-memory loads + one 16-byte table load for 4 Q multiply-adds.  Every output still accumulates
// fmaf(h[k], x[start + k], acc) in ascending k: bit-identical to the first kernel and to the oracle's scalar loop.
template <int Q>
__global__ void __launch_bounds__(256) ns_sinc_resample4_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                const float *__restrict__ hs,  // [sinc_len][L], output order
                                                                long long n_total, long long in_first, long long in_end,
                                                                long long first_out, long long n_out, long long in_stride,
                                                                long long out_stride, int L, int M, int sinc_len, int span,
                                                                int vec_store) {
  extern __shared__ float xs[];
  const int T = blockDim.x, t = threadIdx.x;
  const long long tile = (long long)T * 4 * Q;
  const long long n0 = first_out + (long long)blockIdx.x * tile;  // multiple of L
  const long long base0 = n0 / L * M - sinc_len / 2 + 1;          // recording index of xs[0]
  const float *src = in + (long long)blockIdx.y * in_stride - in_first;
  for (int i = t; i < span; i += T) {
    const long long g = base0 + i;
    xs[i] = (g >= in_first && g < in_end) ? __ldg(src + g) : 0.f;
  }
  __syncthreads();
  const int pos0 = 4 * t * M;                 // 4 t < 1024, M < L <= 1024
  const int rb0 = pos0 / L;
  const bool f1 = (pos0 + M) / L - rb0 == 1, f2 = (pos0 + 2 * M) / L - rb0 == 2, f3 = (pos0 + 3 * M) / L - rb0 == 3;
  const int d1 = f1 ? 1 : 0, d2 = f2 ? 2 : 1, d3 = f3 ? 3 : 2;
  const int step = T * 4 / L * M;             // input samples between two periods of this thread
  const float4 *hrow = reinterpret_cast<const float4 *>(hs + (4 * t) % L);
  const int lrow = L / 4;
  float acc[4][Q];
#pragma unroll
  for (int r = 0; r < 4; r++)
#pragma unroll
    for (int q = 0; q < Q; q++) acc[r][q] = 0.f;
  const float *xp = xs + rb0;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 h0 = z4, h1 = z4, h2 = z4, h3 = z4;  // rows i, i - 1, i - 2, i - 3
  // prologue (i = 0, 1, 2: taps with negative index do not exist) and epilogue (i = sinc_len .. sinc_len + 2: taps past
  // the last do not exist) carry predicates; the main loop needs none
  auto step_fn = [&](int i, bool edge) {
    h3 = h2, h2 = h1, h1 = h0;
    h0 = (i < sinc_len) ? __ldg(hrow + (long long)i * lrow) : z4;
    const float t0 = h0.x, t1 = f1 ? h1.y : h0.y, t2 = f2 ? h2.z : h1.z, t3 = f3 ? h3.w : h2.w;
    const bool v0 = !edge || i < sinc_len, v1 = !edge || (unsigned)(i - d1) < (unsigned)sinc_len,
               v2 = !edge || (unsigned)(i - d2) < (unsigned)sinc_len, v3 = !edge || (unsigned)(i - d3) < (unsigned)sinc_len;
#pragma unroll
    for (int q = 0; q < Q; q++) {
      const float x = xp[q * step + i];
      if (v0) acc[0][q] = fmaf(t0, x, acc[0][q]);
      if (v1) acc[1][q] = fmaf(t1, x, acc[1][q]);
      if (v2) acc[2][q] = fmaf(t2, x, acc[2][q]);
      if (v3) acc[3][q] = fmaf(t3, x, acc[3][q]);
    }
  };
  step_fn(0, true);
  step_fn(1, true);
  step_fn(2, true);
#pragma unroll 4
  for (int i = 3; i < sinc_len; i++) step_fn(i, false);
  step_fn(sinc_len, true);
  step_fn(sinc_len + 1, true);
  step_fn(sinc_len + 2, true);
  float *dst = out + (long long)blockIdx.y * out_stride;
#pragma unroll
  for (int q = 0; q < Q; q++) {
    const long long n = n0 + (long long)q * T * 4 + 4 * t - first_out;
    if (vec_store && n + 4 <= n_out) {
      *reinterpret_cast<float4 *>(dst + n) = make_float4(acc[0][q], acc[1][q], acc[2][q], acc[3][q]);
    } else {
#pragma unroll
      for (int r = 0; r < 4; r++)
        if (n + r < n_out) dst[n + r] = acc[r][q];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string &msg) noexcept {
  try {
    g_err = msg;
  } catch (...) {  // the message itself could not be stored: the code still goes back
  }
  return code;
}
static int fail(int code, const char *msg) noexcept {
  try {
    g_err = msg;
  } catch (...) {
  }
  return code;
}
// Every extern "C" entry point runs its body through guard(): nothing thrown inside (std::bad_alloc from a
// std::vector / std::string / std::map, std::system_error from a std::thread) crosses the C boundary -- the
// reference builds with panic = "abort" (Cargo.toml:10-20) precisely so that nothing unwinds through FFI.
template <class F>
static int guard(const char *what, F &&body) noexcept {
  try {
    return body();
  } catch (const std::bad_alloc &) {
    return fail(CRISPY_NS_ENOMEM, what);
  } catch (const std::exception &e) {
    try {
      return fail(CRISPY_NS_EINVAL, std::string(what) + ": " + e.what());
    } catch (...) {
      return fail(CRISPY_NS_EINVAL, what);
    }
  } catch (...) {
    return fail(CRISPY_NS_EINVAL, what);
  }
}
#define NS_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(CRISPY_NS_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));            \
  } while (0)

struct crispy_ns_model {
  ns::Model m;
  uint32_t numerics = 0;  // crispy_ns_model_set_numerics; not part of the blob
};

constexpr int kSlots = 8;    // workspace slots: chunk c uses slot c % kSlots
constexpr int kNumKernels = 7;  // K0 highpass, K1 pitch, K2 pitchscan, K3 spectrum, K3b features, K4 rnn, K5 synthesis

struct crispy_ns_batch {
  int device = 0;
  int n_streams = 0;
  int n_sms = 148;
  int spec_ctas_per_sm = 4, syn_ctas_per_sm = 4;  // resident CTAs of the two persistent task-loop kernels
  int chunk_cap = 0;  // frames per chunk
  int syn_run_override = 0;  // $CRISPY_NS_SYN_RUN (tests: the result must not depend on it)
  int64_t launches = 0;
  int64_t frames_done = 0;
  int64_t chunks_done = 0;
  ns::Tables *d_tables = nullptr;
  ns::RnnHeader *d_hdr = nullptr;
  uint32_t *d_words = nullptr;
  float *d_bias = nullptr;
  // the tcgen05 recurrent core's weight blocks and biases (ns_rnn_tc5.cuh); rnn_tc5: which core K4 launches
  uint8_t *d_words_tc5 = nullptr;
  float *d_bias_tc5 = nullptr;
  bool rnn_tc5 = false;
  uint32_t numerics = 0;      // the model's crispy_ns_model_set_numerics at batch_create: K0's biquad form, K1's sum order
  bool hp_exclusive = false;  // K0 alone on its SMs (kHpExclusiveSmem)
  bool hp_par = false;        // K0 parallel in time (ns_highpass_par_kernel); $CRISPY_NS_HP_PAR overrides
  float *d_state = nullptr;
  // pipeline workspace + plumbing
  float *d_hp[kSlots] = {};
  uint32_t *d_tab[kSlots] = {};
  float *d_rec[kSlots] = {};
  ns::cf *d_spec[kSlots] = {};
  uint32_t *d_featq[kSlots] = {};
  cudaStream_t s_k[kNumKernels] = {};         // one internal stream per kernel of the pipeline
  cudaEvent_t e_start = nullptr;
  cudaEvent_t e_reset = nullptr;  // recorded by batch_reset_async; every internal stream waits for it once
  bool reset_pending = false;
  // per-stream operations (subset calls, reset / save / load of listed streams).  d_rows: compact state rows, allocated
  // at the first such operation.  Row copies run on the internal streams; e_rows marks the last one, and the next
  // call's first kernel waits for it (rows_pending).  per_stream_ops: the streams no longer share one first frame, so
  // a full call with CRISPY_NS_DROP_FIRST_FRAME is refused until the whole batch is reset or loaded.
  float *d_rows = nullptr;
  cudaEvent_t e_rows = nullptr;
  bool rows_pending = false;
  bool per_stream_ops = false;
  int hp_exclusive_env = -1, hp_par_env = -1;  // $CRISPY_NS_HP_EXCLUSIVE / $CRISPY_NS_HP_PAR at batch_create, -1 unset
  cudaEvent_t e_k[kSlots][kNumKernels] = {};  // "kernel k of the chunk in this slot has finished"
  // optional per-kernel timing (crispy_ns_batch_profile): CUDA events around every launch, each on
  // the stream the kernel is launched on
  bool prof_on = false;
  struct ProfRec {
    cudaEvent_t a, b;
    int kernel;
  };
  std::vector<ProfRec> prof;
  // host-pointer path
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t e_in[2] = {nullptr, nullptr}, e_run[2] = {nullptr, nullptr}, e_out[2] = {nullptr, nullptr},
              e_k0[2] = {nullptr, nullptr};
  void *d_in[2] = {nullptr, nullptr};
  void *d_out[2] = {nullptr, nullptr};
  float *d_vad[2] = {nullptr, nullptr};
  float *d_app[2] = {nullptr, nullptr};
  size_t cap_in = 0, cap_out = 0, cap_vad = 0, cap_app = 0;
};

struct crispy_ns_state {
  crispy_ns_batch *b = nullptr;
  float *h_pin = nullptr;  // 480 in + 480 out + 1 vad, pinned
  float *d_io = nullptr;   // same on device
  // the live path is launch bound (one frame through seven tiny kernels): each call replays a CUDA graph of
  // copy-in -> K0 .. K5 -> copy-out, one graph per workspace slot the chunk counter can select
  cudaStream_t s = nullptr;
  cudaGraphExec_t gexec[kSlots] = {};
};

// ------------------------------------------------------------------------------------------------
// launch: one call = a train of chunks; every chunk goes through the seven kernels, each kernel on
// its own internal stream.  Kernel k of chunk c waits for kernel k-1 of chunk c (event) and, by stream
// order, for kernel k of chunk c-1 (the serial-in-time kernels carry per-stream state from chunk to
// chunk).  With kSlots workspace slots the seven kernels work on up to seven different chunks at
// once, so the latency-bound serial kernels (K0, K2, K3b, K4) hide behind the parallel ones.
// ------------------------------------------------------------------------------------------------
static int default_chunk_cap(int n_streams) {
  const char *env = getenv("CRISPY_NS_CHUNK_FRAMES");
  if (env && atoi(env) > 0) return atoi(env) > 4096 ? 4096 : atoi(env);
  const long long per_frame = (long long)n_streams * (ns::kFrame * 4 + ns::kTabWords * 4 + ns::kRecFloats * 4 + 2 * ns::kSpecStride * 8);
  long long cap = (384ll << 20) / per_frame;  // ~384 MB of workspace per slot
  cap = (cap / kPitchRun) * kPitchRun;
  if (cap < kPitchRun) cap = kPitchRun;
  if (cap > 256) cap = 256;
  return (int)cap;
}

static size_t in_elem(uint32_t flags) { return (flags & CRISPY_NS_IN_I16) ? 2 : 4; }
static size_t out_elem(uint32_t flags) {
  if (flags & CRISPY_NS_MIX_STEREO_I16) return 4;
  return (flags & CRISPY_NS_OUT_I16) ? 2 : 4;
}

// Small batches are bound by the biquad (one lane per stream, 74 cycles per sample), and its recursion warp slows by half
// again when it shares an SM's issue slots with the parallel kernels.  Asking for the whole shared memory of an SM keeps
// every other CTA off the SMs the biquad runs on: it then runs at its isolated speed, at the price of streams / 32 SMs
// that the parallel kernels lose -- a gain up to ~800 streams per GPU, a loss above (profiles/r2_small_batches.md).
constexpr int kHpExclusiveSmem = 227 * 1024;
static cudaError_t configure_kernels(int dev) {
  static std::mutex mu;
  static std::map<int, bool> configured;
  std::lock_guard<std::mutex> lk(mu);
  if (configured[dev]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(ns_highpass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHpExclusiveSmem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_highpass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHpExclusiveSmem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_highpass_par_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHpExclusiveSmem);
  for (int sp = 0; sp < kPitchPolicies && e == cudaSuccess; sp++)
    e = cudaFuncSetAttribute(pitch_kernel((uint32_t)sp), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PitchShared));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_spectrum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ns::SpecSmem));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_synthesis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ns::SpecSmem));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_rnn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ns::RnnSmem));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ns_rnn_tc5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ns::tc5::Smem));
  if (e == cudaSuccess) configured[dev] = true;
  return e;
}

// K0's form for a call over n streams ($CRISPY_NS_HP_EXCLUSIVE / $CRISPY_NS_HP_PAR as read at batch_create win).  Both
// forms give the same bits, so a subset call may pick the form for its own size.  The parallel form speculates the f64
// expression only: under CRISPY_NS_BIQUAD_F32 the single recursion warp runs (its f32 chain is a few dependent f32
// operations a sample instead of the f64 chain's 74 cycles).
static void pick_hp_form(const crispy_ns_batch *b, int n, bool *exclusive, bool *par) {
  *exclusive = b->hp_exclusive_env >= 0 ? b->hp_exclusive_env != 0 : n <= NS_HP_EXCLUSIVE_MAX_STREAMS;
  *par = b->hp_par_env >= 0 ? b->hp_par_env != 0 : (NS_HP_PAR != 0 && *exclusive);
  if (b->numerics & CRISPY_NS_BIQUAD_F32) *par = false;
}

static cudaError_t prof_begin(crispy_ns_batch *b, int kernel, cudaStream_t s) {
  if (!b->prof_on) return cudaSuccess;
  crispy_ns_batch::ProfRec r;
  r.kernel = kernel;
  cudaError_t e = cudaEventCreate(&r.a);
  if (e == cudaSuccess) e = cudaEventCreate(&r.b);
  if (e == cudaSuccess) e = cudaEventRecord(r.a, s);
  if (e == cudaSuccess) b->prof.push_back(r);
  return e;
}
static cudaError_t prof_end(crispy_ns_batch *b, cudaStream_t s) {
  if (!b->prof_on) return cudaSuccess;
  return cudaEventRecord(b->prof.back().b, s);
}
static void prof_clear(crispy_ns_batch *b) {
  for (auto &r : b->prof) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  b->prof.clear();
}

// Optional stream plumbing of one run_device call (host-pointer path): instead of fencing the whole
// pipeline on the caller's stream at both ends, the first kernel waits for the input copy, the
// output-writing kernels wait for the buffer to be drained, and completion is published as events, so
// consecutive calls keep all seven kernels busy across the call boundary.
struct RunHooks {
  cudaEvent_t in_ready = nullptr;  // K0 waits for it (d_in filled)
  cudaEvent_t out_free = nullptr;  // K4 / K5 wait for it (d_vad / d_out / d_app reusable), may be null
  cudaEvent_t k0_done = nullptr;   // recorded after the call's last K0 (d_in may be overwritten)
  cudaEvent_t all_done = nullptr;  // recorded after the call's last K5
};

// one kernel of the chunk described by p (n streams x nf frames) on stream sk; K0 in the form hp_par / hp_exclusive
static void launch_kernel(crispy_ns_batch *b, int k, ns::Params &p, int n, int nf, int groups, cudaStream_t sk, bool hp_par,
                          bool hp_exclusive) {
  switch (k) {
    case 0:
      // measurement aid only: skip the biquad once N chunks have run (the slots then still hold realistic signal)
      if (getenv("CRISPY_NS_EXPERIMENT_SKIP_HP") && b->chunks_done >= atoll(getenv("CRISPY_NS_EXPERIMENT_SKIP_HP"))) break;
      if (hp_par)
        ns_highpass_par_kernel<<<(n + 31) / 32, ns::kHpParThreads, hp_exclusive ? (size_t)kHpExclusiveSmem : sizeof(ns::HpParSmem), sk>>>(p);
      else
        highpass_kernel(b->numerics)<<<(n + 31) / 32, ns::kHpThreads, hp_exclusive ? (size_t)kHpExclusiveSmem : sizeof(ns::HpSmem), sk>>>(p);
      break;
    case 1:
      pitch_kernel(b->numerics)<<<n * ((nf + kPitchRun - 1) / kPitchRun), kPitchThreads, sizeof(PitchShared), sk>>>(p);
      break;
    case 2:
      ns_pitchscan_kernel<<<(n + kScanWarps - 1) / kScanWarps, 32 * kScanWarps, 0, sk>>>(p);
      break;
    case 3: {
      long long ctas = (long long)n * nf;  // persistent task loop: exactly one resident wave
      if (ctas > (long long)b->n_sms * b->spec_ctas_per_sm) ctas = (long long)b->n_sms * b->spec_ctas_per_sm;
      ns_spectrum_kernel<<<(int)ctas, ns::kGroupThreads, sizeof(ns::SpecSmem), sk>>>(p);
      break;
    }
    case 4:
      ns_features_kernel<<<(groups * ns::kMmaStreams + ns::kFeatWarps - 1) / ns::kFeatWarps, 32 * ns::kFeatWarps, 0, sk>>>(p);
      break;
    case 5:
      if (getenv("CRISPY_NS_EXPERIMENT_SKIP_RNN")) break;  // measurement aid only: what the recurrent core costs the pipeline (results are garbage)
      if (b->rnn_tc5) {
        ns::Params q = p;
        q.rnn_words = reinterpret_cast<const uint32_t *>(b->d_words_tc5);
        q.rnn_bias = b->d_bias_tc5;
        ns_rnn_tc5_kernel<<<(n + ns::tc5::kStreams - 1) / ns::tc5::kStreams, ns::tc5::kThreads, sizeof(ns::tc5::Smem), sk>>>(q);
      } else {
        ns_rnn_kernel<<<groups, ns::kMmaThreads, sizeof(ns::RnnSmem), sk>>>(p);
      }
      break;
    default: {
      const int resident = b->n_sms * b->syn_ctas_per_sm;
      p.syn_run = ns::pick_syn_run(n, nf, resident);
      if (b->syn_run_override > 0) p.syn_run = b->syn_run_override < nf ? b->syn_run_override : nf;
      long long ctas = (long long)n * ((nf + p.syn_run - 1) / p.syn_run);
      if (ctas > resident) ctas = resident;
      ns_synthesis_kernel<<<(int)ctas, ns::kGroupThreads, sizeof(ns::SpecSmem), sk>>>(p);
      break;
    }
  }
}

static int run_device(crispy_ns_batch *b, const void *d_in, void *d_out, float *d_vad, const float *d_app,
                      float *d_taps, int n_frames, int64_t in_stride, int64_t out_stride,
                      int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume, cudaStream_t st,
                      const RunHooks *hooks = nullptr, int n_rows = 0) {
  // n_rows > 0: a subset call over the first n_rows compact rows of d_rows (rows_gather put them there); it leaves
  // frames_done alone
  if (!b || n_frames < 0) return fail(CRISPY_NS_EINVAL, "process_streams: bad argument");
  if (n_frames == 0) return CRISPY_NS_OK;  // an empty call touches nothing (its pointers may be null)
  if (!d_in || !d_out) return fail(CRISPY_NS_EINVAL, "process_streams: bad argument");
  if ((flags & CRISPY_NS_OUT_I16) && !(flags & CRISPY_NS_MIX_STEREO_I16) && volume != 1.0f)
    return fail(CRISPY_NS_EINVAL, "process_streams: CRISPY_NS_OUT_I16 is in 16-bit scale and takes no volume (use 1.0)");
  if ((flags & CRISPY_NS_DROP_FIRST_FRAME) && b->per_stream_ops)
    return fail(CRISPY_NS_EINVAL, "process_streams: CRISPY_NS_DROP_FIRST_FRAME after a per-stream operation: the streams no "
                                  "longer share a first frame (reset or load the whole batch first)");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(configure_kernels(b->device));
  ns::Params p;
  memset(&p, 0, sizeof(p));
  p.in = d_in;
  p.out = d_out;
  p.vad = d_vad;
  p.app = d_app;
  p.dbg = d_taps;
  p.state = n_rows > 0 ? b->d_rows : b->d_state;
  p.tables = b->d_tables;
  p.rnn_hdr = b->d_hdr;
  p.rnn_words = b->d_words;
  p.rnn_bias = b->d_bias;
  p.in_stride = in_stride;
  p.out_stride = out_stride;
  p.vad_stride = vad_stride;
  p.app_stride = app_stride;
  p.hp_stride = ns::kHist + (long long)b->chunk_cap * ns::kFrame;
  p.n_streams = n_rows > 0 ? n_rows : b->n_streams;
  p.n_frames_call = n_frames;
  p.chunk_cap = b->chunk_cap;
  p.out_frame_offset = ((flags & CRISPY_NS_DROP_FIRST_FRAME) && b->frames_done == 0) ? -1 : 0;
  p.flags = flags & 0xFFu;
  p.volume = volume;
  const int n = p.n_streams;
  const int groups = (n + ns::kMmaStreams - 1) / ns::kMmaStreams;
  bool hp_par = b->hp_par, hp_exclusive = b->hp_exclusive;
  if (n_rows > 0) pick_hp_form(b, n, &hp_exclusive, &hp_par);
  if (b->reset_pending) {  // an asynchronous reset of the per-stream state is in flight on some caller stream
    for (int k = 0; k < kNumKernels; k++) NS_CUDA(cudaStreamWaitEvent(b->s_k[k], b->e_reset, 0));
    b->reset_pending = false;
  }
  if (b->rows_pending) {  // a per-stream row operation is in flight on the internal streams
    NS_CUDA(cudaStreamWaitEvent(b->s_k[0], b->e_rows, 0));
    b->rows_pending = false;
  }
  if (hooks) {
    NS_CUDA(cudaStreamWaitEvent(b->s_k[0], hooks->in_ready, 0));
    if (hooks->out_free) {
      NS_CUDA(cudaStreamWaitEvent(b->s_k[kNumKernels - 2], hooks->out_free, 0));
      NS_CUDA(cudaStreamWaitEvent(b->s_k[kNumKernels - 1], hooks->out_free, 0));
    }
  } else {
    NS_CUDA(cudaEventRecord(b->e_start, st));
    NS_CUDA(cudaStreamWaitEvent(b->s_k[0], b->e_start, 0));
  }
  int last_slot = 0;
  for (int f0 = 0; f0 < n_frames; f0 += b->chunk_cap) {
    const int slot = (int)(b->chunks_done % kSlots);
    const int nf = (n_frames - f0) < b->chunk_cap ? (n_frames - f0) : b->chunk_cap;
    p.frame0 = f0;
    p.n_frames = nf;
    p.hp = b->d_hp[slot];
    p.tab = b->d_tab[slot];
    p.rec = b->d_rec[slot];
    p.spec = b->d_spec[slot];
    p.featq = b->d_featq[slot];
    p.synth_sel = (int)(b->chunks_done & 1);
    // the slot's previous chunk must have left the pipeline before K0 overwrites its workspace
    if (b->chunks_done >= kSlots) NS_CUDA(cudaStreamWaitEvent(b->s_k[0], b->e_k[slot][kNumKernels - 1], 0));
    for (int k = 0; k < kNumKernels; k++) {
      cudaStream_t sk = b->s_k[k];
      if (k > 0) NS_CUDA(cudaStreamWaitEvent(sk, b->e_k[slot][k - 1], 0));
      NS_CUDA(prof_begin(b, k, sk));
      launch_kernel(b, k, p, n, nf, groups, sk, hp_par, hp_exclusive);
      NS_CUDA(cudaGetLastError());
      NS_CUDA(prof_end(b, sk));
      NS_CUDA(cudaEventRecord(b->e_k[slot][k], sk));
    }
    b->launches += kNumKernels;
    b->chunks_done += 1;
    last_slot = slot;
  }
  if (hooks) {
    NS_CUDA(cudaEventRecord(hooks->k0_done, b->s_k[0]));
    NS_CUDA(cudaEventRecord(hooks->all_done, b->s_k[kNumKernels - 1]));
  } else {
    NS_CUDA(cudaStreamWaitEvent(st, b->e_k[last_slot][kNumKernels - 1], 0));
  }
  if (n_rows == 0) b->frames_done += n_frames;
  return CRISPY_NS_OK;
}

// ------------------------------------------------------------------------------------------------
// C ABI: the implementations live in namespace impl under the names include/crispy_ns.h declares; the extern "C"
// symbols themselves are the generated forwarding wrappers of crispy_ns_abi.inc (included at the end), which
// catch everything.
// ------------------------------------------------------------------------------------------------
namespace impl {

int frame_size(void) { return ns::kFrame; }
const char *last_error(void) { return g_err.c_str(); }
int device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}
int debug_floats(void) { return ns::kDbgFloats; }

int model_synthetic(uint64_t seed, crispy_ns_model **out) {
  if (!out) return fail(CRISPY_NS_EINVAL, "model_synthetic: out is null");
  crispy_ns_model *m = new (std::nothrow) crispy_ns_model();
  if (!m) return fail(CRISPY_NS_ENOMEM, "out of memory");
  ns::model_synthetic(m->m, seed);
  *out = m;
  return CRISPY_NS_OK;
}
int model_from_bytes(const void *blob, size_t len, crispy_ns_model **out) {
  if (!out) return fail(CRISPY_NS_EINVAL, "model_from_bytes: out is null");
  crispy_ns_model *m = new (std::nothrow) crispy_ns_model();
  if (!m) return fail(CRISPY_NS_ENOMEM, "out of memory");
  std::string err;
  if (!ns::model_from_bytes(m->m, blob, len, err)) {
    delete m;
    return fail(CRISPY_NS_EMODEL, err);
  }
  *out = m;
  return CRISPY_NS_OK;
}
int model_to_bytes(const crispy_ns_model *m, void *buf, size_t cap, size_t *needed) {
  if (!m) return fail(CRISPY_NS_EINVAL, "model_to_bytes: model is null");
  const std::vector<uint8_t> b = ns::model_to_bytes(m->m);
  if (needed) *needed = b.size();
  if (buf && cap >= b.size()) memcpy(buf, b.data(), b.size());
  return CRISPY_NS_OK;
}
void model_destroy(crispy_ns_model *m) { delete m; }
int model_set_numerics(crispy_ns_model *m, uint32_t numerics) {
  if (!m) return fail(CRISPY_NS_EINVAL, "model_set_numerics: model is null");
  if ((numerics & ~(uint32_t)(CRISPY_NS_SUM_MASK | CRISPY_NS_BIQUAD_F32)) || (numerics & CRISPY_NS_SUM_MASK) == CRISPY_NS_SUM_MASK)
    return fail(CRISPY_NS_EINVAL, "model_set_numerics: unknown bits, or sum order 3");
  m->numerics = numerics;
  return CRISPY_NS_OK;
}
uint32_t model_numerics(const crispy_ns_model *m) { return m ? m->numerics : 0u; }

static int default_model(ns::Model &m) {
  const char *path = getenv("CRISPY_NS_WEIGHTS");
  if (path && *path) {
    FILE *f = fopen(path, "rb");
    if (!f) return fail(CRISPY_NS_EIO, std::string("cannot open $CRISPY_NS_WEIGHTS: ") + path);
    std::vector<uint8_t> buf;
    uint8_t tmp[65536];
    size_t n;
    while ((n = fread(tmp, 1, sizeof(tmp), f)) > 0) buf.insert(buf.end(), tmp, tmp + n);
    fclose(f);
    std::string err;
    if (!ns::model_from_bytes(m, buf.data(), buf.size(), err)) return fail(CRISPY_NS_EMODEL, err);
    return CRISPY_NS_OK;
  }
  ns::model_synthetic(m, 0);
  return CRISPY_NS_OK;
}

void batch_destroy(crispy_ns_batch *b) {
  if (!b) return;
  cudaSetDevice(b->device);
  prof_clear(b);
  cudaFree(b->d_tables);
  cudaFree(b->d_hdr);
  cudaFree(b->d_words);
  cudaFree(b->d_bias);
  cudaFree(b->d_words_tc5);
  cudaFree(b->d_bias_tc5);
  cudaFree(b->d_state);
  cudaFree(b->d_rows);
  if (b->e_rows) cudaEventDestroy(b->e_rows);
  for (int i = 0; i < kSlots; i++) {
    cudaFree(b->d_hp[i]);
    cudaFree(b->d_tab[i]);
    cudaFree(b->d_rec[i]);
    cudaFree(b->d_spec[i]);
    cudaFree(b->d_featq[i]);
    for (int k = 0; k < kNumKernels; k++)
      if (b->e_k[i][k]) cudaEventDestroy(b->e_k[i][k]);
  }
  if (b->e_start) cudaEventDestroy(b->e_start);
  if (b->e_reset) cudaEventDestroy(b->e_reset);
  for (int k = 0; k < kNumKernels; k++)
    if (b->s_k[k] && (k == 0 || b->s_k[k] != b->s_k[0])) cudaStreamDestroy(b->s_k[k]);
  for (int i = 0; i < 2; i++) {
    cudaFree(b->d_in[i]);
    cudaFree(b->d_out[i]);
    cudaFree(b->d_vad[i]);
    cudaFree(b->d_app[i]);
    if (b->e_in[i]) cudaEventDestroy(b->e_in[i]);
    if (b->e_run[i]) cudaEventDestroy(b->e_run[i]);
    if (b->e_out[i]) cudaEventDestroy(b->e_out[i]);
    if (b->e_k0[i]) cudaEventDestroy(b->e_k0[i]);
  }
  if (b->s_in) cudaStreamDestroy(b->s_in);
  if (b->s_out) cudaStreamDestroy(b->s_out);
  delete b;
}

int batch_create(const crispy_ns_model *model, int device, int n_streams, crispy_ns_batch **out) {
  if (!out || n_streams < 1) return fail(CRISPY_NS_EINVAL, "batch_create: bad argument");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  const uint32_t numerics = model_numerics(model);
#ifdef NS_PITCH_V7
  if (numerics & CRISPY_NS_SUM_MASK)
    return fail(CRISPY_NS_EINVAL, "batch_create: this build's pitch kernel (NS_PITCH_V7) sums in the sequential order only");
#endif
  ns::Model local;
  const ns::Model *m = nullptr;
  if (model) {
    m = &model->m;
  } else {
    const int rc = default_model(local);
    if (rc != CRISPY_NS_OK) return rc;
    m = &local;
  }
  NS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  NS_CUDA(cudaGetDeviceProperties(&prop, device));
  crispy_ns_batch *b = new (std::nothrow) crispy_ns_batch();
  if (!b) return fail(CRISPY_NS_ENOMEM, "out of memory");
  b->device = device;
  b->n_streams = n_streams;
  b->numerics = numerics;
  b->n_sms = prop.multiProcessorCount;
  b->chunk_cap = default_chunk_cap(n_streams);
  if (const char *e = getenv("CRISPY_NS_SYN_RUN")) b->syn_run_override = atoi(e);
  if ((long long)n_streams * b->chunk_cap >= (1ll << 31)) {  // the task-loop kernels index (stream, frame) in 32 bits
    delete b;
    return fail(CRISPY_NS_EINVAL, "batch_create: n_streams x chunk frames must stay below 2^31");
  }
  if (cudaError_t ce = configure_kernels(device); ce != cudaSuccess) {
    delete b;
    return fail(CRISPY_NS_ECUDA, std::string("batch_create: ") + cudaGetErrorString(ce));
  }
  {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ns_spectrum_kernel, ns::kGroupThreads, sizeof(ns::SpecSmem)) == cudaSuccess && occ > 0)
      b->spec_ctas_per_sm = occ;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ns_synthesis_kernel, ns::kGroupThreads, sizeof(ns::SpecSmem)) == cudaSuccess && occ > 0)
      b->syn_ctas_per_sm = occ;
    if (getenv("CRISPY_NS_SPEC_CTAS") && atoi(getenv("CRISPY_NS_SPEC_CTAS")) > 0) b->spec_ctas_per_sm = atoi(getenv("CRISPY_NS_SPEC_CTAS"));
    if (getenv("CRISPY_NS_SYN_CTAS") && atoi(getenv("CRISPY_NS_SYN_CTAS")) > 0) b->syn_ctas_per_sm = atoi(getenv("CRISPY_NS_SYN_CTAS"));
  }
  ns::PackedRnn pk;
  ns::pack_rnn(*m, pk);
  static ns::Tables tab;
  static std::once_flag once;
  std::call_once(once, [] { ns::make_tables(tab); });
  cudaError_t e = cudaSuccess;
  auto up = [&](void **dst, const void *src, size_t bytes) {
    if (e != cudaSuccess) return;
    e = cudaMalloc(dst, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
  };
  up((void **)&b->d_tables, &tab, sizeof(tab));
  up((void **)&b->d_hdr, &pk.hdr, sizeof(pk.hdr));
  up((void **)&b->d_words, pk.words.data(), pk.words.size() * sizeof(uint32_t));
  up((void **)&b->d_bias, pk.bias.data(), pk.bias.size() * sizeof(float));
  {
    // K4 variant: $CRISPY_NS_RNN = "tc5" (tcgen05 / tensor memory, 128 streams per CTA) or "mma" (warp-level mma.sync,
    // 16 streams per CTA).  Default: mma.  tc5 holds 8 SMs per 1,024 streams instead of 64, which the parallel kernels
    // get back, but its step is longer (thirteen rounds per frame) and the pipeline measured no faster with it
    // (profiles/r2_k4_tcgen05.md), so it stays opt-in (NS_RNN_TC5_MIN_STREAMS).
    // K0 alone on its SMs: $CRISPY_NS_HP_EXCLUSIVE = 1 / 0, default by batch size
    const char *hx = getenv("CRISPY_NS_HP_EXCLUSIVE");
    const char *hpp = getenv("CRISPY_NS_HP_PAR");
    b->hp_exclusive_env = hx ? atoi(hx) != 0 : -1;
    b->hp_par_env = hpp ? atoi(hpp) != 0 : -1;
    pick_hp_form(b, n_streams, &b->hp_exclusive, &b->hp_par);
    const char *sel = getenv("CRISPY_NS_RNN");
    b->rnn_tc5 = sel ? (strcmp(sel, "tc5") == 0) : (n_streams >= NS_RNN_TC5_MIN_STREAMS);
    std::vector<uint8_t> w5;
    std::vector<float> b5;
    ns::pack_rnn_tc5(*m, w5, b5);
    up((void **)&b->d_words_tc5, w5.data(), w5.size());
    up((void **)&b->d_bias_tc5, b5.data(), b5.size() * sizeof(float));
  }
  if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_state, (size_t)n_streams * ns::kStateFloats * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(b->d_state, 0, (size_t)n_streams * ns::kStateFloats * sizeof(float));
  for (int i = 0; i < kSlots && e == cudaSuccess; i++) {
    const size_t nf = (size_t)n_streams * b->chunk_cap;
    e = cudaMalloc((void **)&b->d_hp[i], (size_t)n_streams * (ns::kHist + (size_t)b->chunk_cap * ns::kFrame) * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_tab[i], nf * ns::kTabWords * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_rec[i], nf * ns::kRecFloats * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_spec[i], nf * 2 * ns::kSpecStride * sizeof(ns::cf));
    if (e == cudaSuccess)
      e = cudaMalloc((void **)&b->d_featq[i], (size_t)((n_streams + ns::kMmaStreams - 1) / ns::kMmaStreams) * b->chunk_cap *
                                                  ns::kFeatBlockWords * sizeof(uint32_t));
    for (int k = 0; k < kNumKernels && e == cudaSuccess; k++) e = cudaEventCreateWithFlags(&b->e_k[i][k], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->e_start, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->e_reset, cudaEventDisableTiming);
  {  // the serial-in-time kernels (few warps, latency bound) get the higher block-scheduling priority
    int prio_lo = 0, prio_hi = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    static const bool serial[kNumKernels] = {true, false, true, false, true, true, false};
    // $CRISPY_NS_SERIAL=1 (measurement aid): every kernel on one stream, so per-kernel event times are
    // isolated durations comparable with an ncu launch list
    const bool one_stream = getenv("CRISPY_NS_SERIAL") && atoi(getenv("CRISPY_NS_SERIAL")) > 0;
    for (int k = 0; k < kNumKernels && e == cudaSuccess; k++) {
      if (one_stream && k > 0)
        b->s_k[k] = b->s_k[0];
      else
        e = cudaStreamCreateWithPriority(&b->s_k[k], cudaStreamNonBlocking, serial[k] ? prio_hi : prio_lo);
    }
  }
  if (e != cudaSuccess) {
    batch_destroy(b);
    return fail(CRISPY_NS_ECUDA, std::string("batch_create: ") + cudaGetErrorString(e));
  }
  *out = b;
  return CRISPY_NS_OK;
}

int batch_reset(crispy_ns_batch *b) {
  if (!b) return fail(CRISPY_NS_EINVAL, "batch_reset: null handle");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaDeviceSynchronize());
  NS_CUDA(cudaMemset(b->d_state, 0, (size_t)b->n_streams * ns::kStateFloats * sizeof(float)));
  b->frames_done = 0;
  b->per_stream_ops = false;
  return CRISPY_NS_OK;
}
int batch_reset_async(crispy_ns_batch *b, void *cuda_stream) {
  if (!b) return fail(CRISPY_NS_EINVAL, "batch_reset_async: null handle");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaMemsetAsync(b->d_state, 0, (size_t)b->n_streams * ns::kStateFloats * sizeof(float), (cudaStream_t)cuda_stream));
  NS_CUDA(cudaEventRecord(b->e_reset, (cudaStream_t)cuda_stream));
  b->reset_pending = true;
  b->frames_done = 0;
  b->per_stream_ops = false;
  return CRISPY_NS_OK;
}
int batch_n_streams(const crispy_ns_batch *b) { return b ? b->n_streams : 0; }

int process_streams(crispy_ns_batch *b, const void *d_in, void *d_out, float *d_vad,
                              const float *d_app, int n_frames, int64_t in_stride, int64_t out_stride,
                              int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume,
                              void *cuda_stream) {
  return run_device(b, d_in, d_out, d_vad, d_app, nullptr, n_frames, in_stride, out_stride, vad_stride,
                    app_stride, flags, volume, (cudaStream_t)cuda_stream);
}

int process_streams_debug(crispy_ns_batch *b, const void *d_in, void *d_out, float *d_vad,
                                    float *d_taps, int n_frames, int64_t in_stride, int64_t out_stride,
                                    uint32_t flags, float volume, void *cuda_stream) {
  return run_device(b, d_in, d_out, d_vad, nullptr, d_taps, n_frames, in_stride, out_stride, n_frames, 0,
                    flags, volume, (cudaStream_t)cuda_stream);
}

// the host-pointer path over all streams, or (n_rows > 0) over the compact rows a subset call gathered
static int run_host(crispy_ns_batch *b, const void *h_in, void *h_out, float *h_vad, const float *h_app, int n_frames,
                    int64_t in_stride, int64_t out_stride, int64_t vad_stride, int64_t app_stride, uint32_t flags,
                    float volume, int n_rows) {
  if (!b || n_frames < 0) return fail(CRISPY_NS_EINVAL, "process_streams_host: bad argument");
  if (n_frames == 0) return CRISPY_NS_OK;  // an empty call touches nothing (its pointers may be null)
  if (!h_in || !h_out) return fail(CRISPY_NS_EINVAL, "process_streams_host: bad argument");
  if ((flags & CRISPY_NS_DROP_FIRST_FRAME) && b->per_stream_ops)
    return fail(CRISPY_NS_EINVAL, "process_streams_host: CRISPY_NS_DROP_FIRST_FRAME after a per-stream operation: the "
                                  "streams no longer share a first frame (reset or load the whole batch first)");
  NS_CUDA(cudaSetDevice(b->device));
  if (!b->s_in) {
    NS_CUDA(cudaStreamCreateWithFlags(&b->s_in, cudaStreamNonBlocking));
    NS_CUDA(cudaStreamCreateWithFlags(&b->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      NS_CUDA(cudaEventCreateWithFlags(&b->e_in[i], cudaEventDisableTiming));
      NS_CUDA(cudaEventCreateWithFlags(&b->e_run[i], cudaEventDisableTiming));
      NS_CUDA(cudaEventCreateWithFlags(&b->e_out[i], cudaEventDisableTiming));
      NS_CUDA(cudaEventCreateWithFlags(&b->e_k0[i], cudaEventDisableTiming));
    }
  }
  const size_t ie = in_elem(flags), oe = out_elem(flags);
  const int n = n_rows > 0 ? n_rows : b->n_streams;
  // host chunk length in frames: a whole number of engine chunks, ~128 MiB of input per buffer
  long long ch = (128ll << 20) / ((long long)n * ns::kFrame * (long long)ie) / b->chunk_cap * b->chunk_cap;
  if (ch < b->chunk_cap) ch = b->chunk_cap;
  if (ch > n_frames) ch = n_frames;
  const char *env = getenv("CRISPY_NS_HOST_CHUNK_FRAMES");
  if (env && atoi(env) > 0) ch = atoi(env) < n_frames ? atoi(env) : n_frames;
  const size_t in_bytes = (size_t)n * ch * ns::kFrame * ie, out_bytes = (size_t)n * ch * ns::kFrame * oe;
  const bool use_app = (flags & CRISPY_NS_MIX_STEREO_I16) && h_app;
  // (re)allocate double buffers
  if (b->cap_in < in_bytes) {
    for (int i = 0; i < 2; i++) {
      if (b->d_in[i]) cudaFree(b->d_in[i]);
      b->d_in[i] = nullptr;
    }
    NS_CUDA(cudaMalloc(&b->d_in[0], in_bytes));
    NS_CUDA(cudaMalloc(&b->d_in[1], in_bytes));
    b->cap_in = in_bytes;
  }
  if (b->cap_out < out_bytes) {
    for (int i = 0; i < 2; i++) {
      if (b->d_out[i]) cudaFree(b->d_out[i]);
      b->d_out[i] = nullptr;
    }
    NS_CUDA(cudaMalloc(&b->d_out[0], out_bytes));
    NS_CUDA(cudaMalloc(&b->d_out[1], out_bytes));
    b->cap_out = out_bytes;
  }
  const size_t vad_bytes = (size_t)n * ch * sizeof(float);
  if (h_vad && b->cap_vad < vad_bytes) {
    for (int i = 0; i < 2; i++) {
      if (b->d_vad[i]) cudaFree(b->d_vad[i]);
      b->d_vad[i] = nullptr;
    }
    NS_CUDA(cudaMalloc((void **)&b->d_vad[0], vad_bytes));
    NS_CUDA(cudaMalloc((void **)&b->d_vad[1], vad_bytes));
    b->cap_vad = vad_bytes;
  }
  const size_t app_bytes = (size_t)n * ch * ns::kFrame * sizeof(float);
  if (use_app && b->cap_app < app_bytes) {
    for (int i = 0; i < 2; i++) {
      if (b->d_app[i]) cudaFree(b->d_app[i]);
      b->d_app[i] = nullptr;
    }
    NS_CUDA(cudaMalloc((void **)&b->d_app[0], app_bytes));
    NS_CUDA(cudaMalloc((void **)&b->d_app[1], app_bytes));
    b->cap_app = app_bytes;
  }
  const bool drop = (flags & CRISPY_NS_DROP_FIRST_FRAME) && b->frames_done == 0;
  int c = 0;
  for (long long f0 = 0; f0 < n_frames; f0 += ch, c++) {
    const int k = c & 1;
    const long long nf = (f0 + ch <= n_frames) ? ch : (n_frames - f0);
    // the in buffer k was last read by the biquad of host chunk c-2; the out buffer k was last
    // drained by copy c-2 (the output-writing kernels wait for that through the hooks)
    if (c >= 2) {
      NS_CUDA(cudaStreamWaitEvent(b->s_in, b->e_k0[k], 0));
      if (use_app) NS_CUDA(cudaStreamWaitEvent(b->s_in, b->e_run[k], 0));  // K5 of host chunk c-2 read d_app[k]
    }
    const long long row = nf * ns::kFrame;
    NS_CUDA(cudaMemcpy2DAsync(b->d_in[k], (size_t)row * ie, (const char *)h_in + (size_t)f0 * ns::kFrame * ie,
                              (size_t)in_stride * ie, (size_t)row * ie, n, cudaMemcpyHostToDevice, b->s_in));
    // frames the chunk emits and where they land in the caller's output
    const int off = (drop && f0 == 0) ? -1 : 0;
    const long long nf_out = nf + off;
    const long long out_f0 = f0 + ((drop && f0 > 0) ? -1 : 0);
    if (use_app && nf_out > 0)
      NS_CUDA(cudaMemcpy2DAsync(b->d_app[k], (size_t)row * 4, (const char *)h_app + (size_t)out_f0 * ns::kFrame * 4,
                                (size_t)app_stride * 4, (size_t)nf_out * ns::kFrame * 4, n,
                                cudaMemcpyHostToDevice, b->s_in));
    NS_CUDA(cudaEventRecord(b->e_in[k], b->s_in));
    RunHooks hooks;
    hooks.in_ready = b->e_in[k];
    hooks.out_free = (c >= 2) ? b->e_out[k] : nullptr;
    hooks.k0_done = b->e_k0[k];
    hooks.all_done = b->e_run[k];
    const int rc = run_device(b, b->d_in[k], b->d_out[k], h_vad ? b->d_vad[k] : nullptr,
                              use_app ? b->d_app[k] : nullptr, nullptr, (int)nf, row, row, nf, row, flags,
                              volume, nullptr, &hooks, n_rows);
    if (rc != CRISPY_NS_OK) return rc;
    NS_CUDA(cudaStreamWaitEvent(b->s_out, b->e_run[k], 0));
    if (nf_out > 0)
      NS_CUDA(cudaMemcpy2DAsync((char *)h_out + (size_t)out_f0 * ns::kFrame * oe, (size_t)out_stride * oe,
                                b->d_out[k], (size_t)row * oe, (size_t)nf_out * ns::kFrame * oe, n,
                                cudaMemcpyDeviceToHost, b->s_out));
    if (h_vad)
      NS_CUDA(cudaMemcpy2DAsync(h_vad + f0, (size_t)vad_stride * 4, b->d_vad[k], (size_t)nf * 4, (size_t)nf * 4, n,
                                cudaMemcpyDeviceToHost, b->s_out));
    NS_CUDA(cudaEventRecord(b->e_out[k], b->s_out));
  }
  NS_CUDA(cudaStreamSynchronize(b->s_out));
  NS_CUDA(cudaStreamSynchronize(b->s_in));
  return CRISPY_NS_OK;
}

int process_streams_host(crispy_ns_batch *b, const void *h_in, void *h_out, float *h_vad,
                                   const float *h_app, int n_frames, int64_t in_stride,
                                   int64_t out_stride, int64_t vad_stride, int64_t app_stride,
                                   uint32_t flags, float volume) {
  return run_host(b, h_in, h_out, h_vad, h_app, n_frames, in_stride, out_stride, vad_stride, app_stride, flags, volume, 0);
}

size_t batch_state_size(const crispy_ns_batch *b) {
  return b ? (size_t)b->n_streams * ns::kStateFloats * sizeof(float) + 16 : 0;
}
int batch_save_state(crispy_ns_batch *b, void *buf, size_t len) {
  if (!b || !buf || len < batch_state_size(b)) return fail(CRISPY_NS_EINVAL, "save_state: bad argument");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaDeviceSynchronize());
  int64_t hdr[2] = {b->n_streams | (b->chunks_done & 1) << 40, b->frames_done};
  memcpy(buf, hdr, 16);
  NS_CUDA(cudaMemcpy((char *)buf + 16, b->d_state, len - 16 < batch_state_size(b) - 16 ? len - 16 : batch_state_size(b) - 16,
                     cudaMemcpyDeviceToHost));
  return CRISPY_NS_OK;
}
int batch_load_state(crispy_ns_batch *b, const void *buf, size_t len) {
  if (!b || !buf || len < batch_state_size(b)) return fail(CRISPY_NS_EINVAL, "load_state: bad argument");
  int64_t hdr[2];
  memcpy(hdr, buf, 16);
  const int64_t sel = (hdr[0] >> 40) & 1;
  hdr[0] &= ((int64_t)1 << 40) - 1;
  if (hdr[0] != b->n_streams) return fail(CRISPY_NS_EINVAL, "load_state: stream count mismatch");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaDeviceSynchronize());
  NS_CUDA(cudaMemcpy(b->d_state, (const char *)buf + 16, batch_state_size(b) - 16, cudaMemcpyHostToDevice));
  b->frames_done = hdr[1];
  b->per_stream_ops = false;
  if ((b->chunks_done & 1) != sel) b->chunks_done += 1;  // synthesis_mem double buffer parity (ns_common.h kStSynth)
  return CRISPY_NS_OK;
}

// ---- per-stream operations ---------------------------------------------------------------------------
// Subset calls gather the listed state rows into d_rows, run the unchanged pipeline over them and scatter them back.
// Ordering: every row copy sits on an internal stream behind the last K5 already enqueued (s_k[6] carries every K5, and
// each chunk's K5 follows its K0 .. K4), and e_rows, recorded after it, is what the next call's K0 waits for.
// synthesis_mem parity: every stream's current copy is copy (chunks_done & 1).  A subset call of k chunks leaves its
// rows' current copy at (P + k) & 1; an odd k advances chunks_done once more (one workspace slot skipped, as
// batch_load_state does) and the scatter puts that copy back at P, so the invariant holds for every stream.
// A stream record is a 16-byte header and the state row with the current copy first and zeros in the other.  The
// header's last word is the batch's numerics: a state evolved under one arithmetic does not continue under another.
static const char kStreamMagic[8] = {'C', 'R', 'N', 'S', 'S', 'T', 'R', '1'};
constexpr size_t kStreamHeader = 16, kRowBytes = (size_t)ns::kStateFloats * sizeof(float);

static int check_ids(const crispy_ns_batch *b, const int *ids, int n, const char *what) {
  if (!b) return fail(CRISPY_NS_EINVAL, std::string(what) + ": null handle");
  if (n < 0 || n > b->n_streams || (n > 0 && !ids))
    return fail(CRISPY_NS_EINVAL, std::string(what) + ": the stream count must be in [0, n_streams] with a stream list");
  std::vector<char> seen((size_t)b->n_streams, 0);
  for (int i = 0; i < n; i++) {
    if (ids[i] < 0 || ids[i] >= b->n_streams) return fail(CRISPY_NS_EINVAL, std::string(what) + ": stream id out of range");
    if (seen[(size_t)ids[i]]) return fail(CRISPY_NS_EINVAL, std::string(what) + ": stream listed twice");
    seen[(size_t)ids[i]] = 1;
  }
  return CRISPY_NS_OK;
}

// e_rows exists, and the internal streams are ordered after an asynchronous whole-batch reset
static int rows_order(crispy_ns_batch *b) {
  NS_CUDA(cudaSetDevice(b->device));
  if (!b->e_rows) NS_CUDA(cudaEventCreateWithFlags(&b->e_rows, cudaEventDisableTiming));
  if (b->reset_pending) {
    for (int k = 0; k < kNumKernels; k++) NS_CUDA(cudaStreamWaitEvent(b->s_k[k], b->e_reset, 0));
    b->reset_pending = false;
  }
  return CRISPY_NS_OK;
}

// as rows_order, and d_rows exists
static int rows_prepare(crispy_ns_batch *b) {
  if (int rc = rows_order(b)) return rc;
  if (!b->d_rows) NS_CUDA(cudaMalloc((void **)&b->d_rows, (size_t)b->n_streams * kRowBytes));
  return CRISPY_NS_OK;
}

static int rows_launch(cudaStream_t s, float *dst, const float *src, const int *ids, int n,
                       bool ids_on_src, int src_cur, int dst_cur, bool keep_stale) {
  RowArgs a;
  a.dst = dst;
  a.src = src;
  a.ids_on_src = ids_on_src;
  a.src_cur = src_cur;
  a.dst_cur = dst_cur;
  a.keep_stale = keep_stale;
  for (int first = 0; first < n; first += kRowIds) {
    a.first = first;
    a.n = n - first < kRowIds ? n - first : kRowIds;
    memcpy(a.ids, ids + first, (size_t)a.n * sizeof(int));
    ns_state_rows_kernel<<<a.n, 256, 0, s>>>(a);
    NS_CUDA(cudaGetLastError());
  }
  return CRISPY_NS_OK;
}

// row operation on s_k[6] done: the next call waits for it
static int rows_publish(crispy_ns_batch *b) {
  NS_CUDA(cudaEventRecord(b->e_rows, b->s_k[kNumKernels - 1]));
  b->rows_pending = true;
  return CRISPY_NS_OK;
}

static int subset_check(crispy_ns_batch *b, const int *ids, int m, const void *in, const void *out, int n_frames,
                        uint32_t flags, float volume, const char *what) {
  if (int rc = check_ids(b, ids, m, what)) return rc;
  if (n_frames < 0) return fail(CRISPY_NS_EINVAL, std::string(what) + ": bad argument");
  if (flags & CRISPY_NS_DROP_FIRST_FRAME)
    return fail(CRISPY_NS_EINVAL, std::string(what) + ": CRISPY_NS_DROP_FIRST_FRAME is not taken on subset calls");
  if (m == 0 || n_frames == 0) return CRISPY_NS_OK;
  if (!in || !out) return fail(CRISPY_NS_EINVAL, std::string(what) + ": bad argument");
  if ((flags & CRISPY_NS_OUT_I16) && !(flags & CRISPY_NS_MIX_STEREO_I16) && volume != 1.0f)
    return fail(CRISPY_NS_EINVAL, std::string(what) + ": CRISPY_NS_OUT_I16 is in 16-bit scale and takes no volume (use 1.0)");
  return CRISPY_NS_OK;
}

// gather on s_k[0], behind everything enqueued so far (the previous call's scatter included)
static int subset_begin(crispy_ns_batch *b, const int *ids, int m) {
  if (int rc = rows_prepare(b)) return rc;
  NS_CUDA(cudaEventRecord(b->e_rows, b->s_k[kNumKernels - 1]));
  NS_CUDA(cudaStreamWaitEvent(b->s_k[0], b->e_rows, 0));
  b->rows_pending = false;
  return rows_launch(b->s_k[0], b->d_rows, b->d_state, ids, m, true, 0, 0, true);
}

// scatter on s_k[6] after the call's last K5, restoring the parity invariant
static int subset_end(crispy_ns_batch *b, const int *ids, int m, int64_t chunks_before) {
  const int64_t k = b->chunks_done - chunks_before;
  if (k & 1) b->chunks_done += 1;
  b->per_stream_ops = true;
  if (int rc = rows_launch(b->s_k[kNumKernels - 1], b->d_state, b->d_rows, ids, m, false, (int)((chunks_before + k) & 1),
                           (int)(chunks_before & 1), true))
    return rc;
  return rows_publish(b);
}

int process_streams_subset(crispy_ns_batch *b, const int *streams, int n_active, const void *d_in, void *d_out,
                           float *d_vad, const float *d_app, int n_frames, int64_t in_stride, int64_t out_stride,
                           int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume, void *cuda_stream) {
  if (int rc = subset_check(b, streams, n_active, d_in, d_out, n_frames, flags, volume, "process_streams_subset")) return rc;
  if (n_active == 0 || n_frames == 0) return CRISPY_NS_OK;
  const int64_t c0 = b->chunks_done;
  if (int rc = subset_begin(b, streams, n_active)) return rc;
  if (int rc = run_device(b, d_in, d_out, d_vad, d_app, nullptr, n_frames, in_stride, out_stride, vad_stride, app_stride,
                          flags, volume, (cudaStream_t)cuda_stream, nullptr, n_active))
    return rc;
  if (int rc = subset_end(b, streams, n_active, c0)) return rc;
  NS_CUDA(cudaStreamWaitEvent((cudaStream_t)cuda_stream, b->e_rows, 0));
  return CRISPY_NS_OK;
}

int process_streams_subset_host(crispy_ns_batch *b, const int *streams, int n_active, const void *h_in, void *h_out,
                                float *h_vad, const float *h_app, int n_frames, int64_t in_stride, int64_t out_stride,
                                int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume) {
  if (int rc = subset_check(b, streams, n_active, h_in, h_out, n_frames, flags, volume, "process_streams_subset_host"))
    return rc;
  if (n_active == 0 || n_frames == 0) return CRISPY_NS_OK;
  const int64_t c0 = b->chunks_done;
  if (int rc = subset_begin(b, streams, n_active)) return rc;
  if (int rc = run_host(b, h_in, h_out, h_vad, h_app, n_frames, in_stride, out_stride, vad_stride, app_stride, flags,
                        volume, n_active))
    return rc;
  if (int rc = subset_end(b, streams, n_active, c0)) return rc;
  NS_CUDA(cudaStreamSynchronize(b->s_k[kNumKernels - 1]));
  return CRISPY_NS_OK;
}

int batch_reset_streams(crispy_ns_batch *b, const int *streams, int n, void *cuda_stream) {
  if (int rc = check_ids(b, streams, n, "batch_reset_streams")) return rc;
  if (n == 0) return CRISPY_NS_OK;
  if (int rc = rows_prepare(b)) return rc;
  cudaStream_t s6 = b->s_k[kNumKernels - 1];
  NS_CUDA(cudaEventRecord(b->e_start, (cudaStream_t)cuda_stream));  // behind the caller's work, too
  NS_CUDA(cudaStreamWaitEvent(s6, b->e_start, 0));
  if (int rc = rows_launch(s6, b->d_state, nullptr, streams, n, false, 0, 0, false)) return rc;
  b->per_stream_ops = true;
  if (int rc = rows_publish(b)) return rc;
  NS_CUDA(cudaStreamWaitEvent((cudaStream_t)cuda_stream, b->e_rows, 0));
  return CRISPY_NS_OK;
}

size_t stream_state_size(void) { return kStreamHeader + kRowBytes; }

int batch_save_streams(crispy_ns_batch *b, const int *streams, int n, void *buf, size_t len) {
  if (int rc = check_ids(b, streams, n, "batch_save_streams")) return rc;
  if ((n > 0 && !buf) || len < (size_t)n * stream_state_size())
    return fail(CRISPY_NS_EINVAL, "batch_save_streams: the buffer must hold n * crispy_ns_stream_state_size() bytes");
  if (n == 0) return CRISPY_NS_OK;
  if (int rc = rows_prepare(b)) return rc;
  cudaStream_t s6 = b->s_k[kNumKernels - 1];
  if (int rc = rows_launch(s6, b->d_rows, b->d_state, streams, n, true, (int)(b->chunks_done & 1), 0, false)) return rc;
  NS_CUDA(cudaMemcpy2DAsync((char *)buf + kStreamHeader, stream_state_size(), b->d_rows, kRowBytes, kRowBytes, (size_t)n,
                            cudaMemcpyDeviceToHost, s6));
  if (int rc = rows_publish(b)) return rc;
  NS_CUDA(cudaStreamSynchronize(s6));
  for (int i = 0; i < n; i++) {
    uint8_t *h = (uint8_t *)buf + (size_t)i * stream_state_size();
    const uint32_t words[2] = {(uint32_t)ns::kStateFloats, b->numerics};
    memcpy(h, kStreamMagic, 8);
    memcpy(h + 8, words, 8);
  }
  return CRISPY_NS_OK;
}

int batch_load_streams(crispy_ns_batch *b, const int *streams, int n, const void *buf, size_t len) {
  if (int rc = check_ids(b, streams, n, "batch_load_streams")) return rc;
  if ((n > 0 && !buf) || len != (size_t)n * stream_state_size())
    return fail(CRISPY_NS_EINVAL, "batch_load_streams: the buffer must be n records of crispy_ns_stream_state_size() bytes");
  for (int i = 0; i < n; i++) {
    const uint8_t *h = (const uint8_t *)buf + (size_t)i * stream_state_size();
    uint32_t words[2];
    memcpy(words, h + 8, 8);
    if (memcmp(h, kStreamMagic, 8) != 0 || words[0] != (uint32_t)ns::kStateFloats)
      return fail(CRISPY_NS_EINVAL, "batch_load_streams: not a stream record of this build");
    if (words[1] != b->numerics)
      return fail(CRISPY_NS_EINVAL, "batch_load_streams: the record was saved under other numerics than the batch's");
  }
  if (n == 0) return CRISPY_NS_OK;
  if (int rc = rows_prepare(b)) return rc;
  cudaStream_t s6 = b->s_k[kNumKernels - 1];
  NS_CUDA(cudaMemcpy2DAsync(b->d_rows, kRowBytes, (const char *)buf + kStreamHeader, stream_state_size(), kRowBytes, (size_t)n,
                            cudaMemcpyHostToDevice, s6));
  if (int rc = rows_launch(s6, b->d_state, b->d_rows, streams, n, false, 0, (int)(b->chunks_done & 1), false)) return rc;
  b->per_stream_ops = true;
  if (int rc = rows_publish(b)) return rc;
  NS_CUDA(cudaStreamSynchronize(s6));  // buf may be reused as soon as the call returns
  return CRISPY_NS_OK;
}
// ---- per-stream suppression controls: four words of the state row (ns_common.h kStCtl*), so subset calls, stream
// records, whole-batch states and the single-frame graphs carry them, and every reset turns them off
static bool unit_interval(float x) { return x >= 0.f && x <= 1.f; }  // false for NaN
static int check_controls(const crispy_ns_controls *c, int n, const char *what) {
  if (n > 0 && !c) return fail(CRISPY_NS_EINVAL, std::string(what) + ": controls is null");
  for (int i = 0; i < n; i++)
    if (!unit_interval(c[i].min_gain) || !unit_interval(c[i].gate_threshold) || !unit_interval(c[i].gate_gain) ||
        c[i].gate_hold < 0 || c[i].gate_hold > (1 << 20))
      return fail(CRISPY_NS_EINVAL, std::string(what) + ": a control is out of range or NaN");
  return CRISPY_NS_OK;
}

int batch_set_controls(crispy_ns_batch *b, const int *streams, int n, const void *controls_v, void *cuda_stream) {
  const crispy_ns_controls *controls = static_cast<const crispy_ns_controls *>(controls_v);
  if (int rc = check_ids(b, streams, n, "batch_set_controls")) return rc;
  if (int rc = check_controls(controls, n, "batch_set_controls")) return rc;
  if (n == 0) return CRISPY_NS_OK;
  if (int rc = rows_order(b)) return rc;
  cudaStream_t s6 = b->s_k[kNumKernels - 1];
  NS_CUDA(cudaEventRecord(b->e_start, (cudaStream_t)cuda_stream));  // behind the caller's work, as reset_streams
  NS_CUDA(cudaStreamWaitEvent(s6, b->e_start, 0));
  ControlArgs a;
  a.state = b->d_state;
  for (int first = 0; first < n; first += kCtlIds) {
    a.n = n - first < kCtlIds ? n - first : kCtlIds;
    for (int j = 0; j < a.n; j++) {
      const crispy_ns_controls &c = controls[first + j];
      a.ids[j] = streams[first + j];
      memcpy(&a.words[j][0], &c.min_gain, 4);
      memcpy(&a.words[j][1], &c.gate_threshold, 4);
      memcpy(&a.words[j][2], &c.gate_hold, 4);
      memcpy(&a.words[j][3], &c.gate_gain, 4);
    }
    ns_set_controls_kernel<<<1, kCtlIds, 0, s6>>>(a);
    NS_CUDA(cudaGetLastError());
  }
  if (int rc = rows_publish(b)) return rc;
  NS_CUDA(cudaStreamWaitEvent((cudaStream_t)cuda_stream, b->e_rows, 0));
  return CRISPY_NS_OK;
}

int batch_get_controls(crispy_ns_batch *b, const int *streams, int n, void *out_v) {
  crispy_ns_controls *out = static_cast<crispy_ns_controls *>(out_v);
  if (int rc = check_ids(b, streams, n, "batch_get_controls")) return rc;
  if (n > 0 && !out) return fail(CRISPY_NS_EINVAL, "batch_get_controls: out is null");
  if (n == 0) return CRISPY_NS_OK;
  if (int rc = rows_order(b)) return rc;
  cudaStream_t s6 = b->s_k[kNumKernels - 1];  // behind every set_controls, reset and load already enqueued
  std::vector<uint32_t> w((size_t)b->n_streams * 4);
  NS_CUDA(cudaMemcpy2DAsync(w.data(), 16, b->d_state + ns::kStCtlMinGain, kRowBytes, 16, (size_t)b->n_streams,
                            cudaMemcpyDeviceToHost, s6));
  NS_CUDA(cudaStreamSynchronize(s6));
  for (int i = 0; i < n; i++) {
    const uint32_t *r = &w[(size_t)streams[i] * 4];
    memcpy(&out[i].min_gain, &r[0], 4);
    memcpy(&out[i].gate_threshold, &r[1], 4);
    memcpy(&out[i].gate_hold, &r[2], 4);
    memcpy(&out[i].gate_gain, &r[3], 4);
  }
  return CRISPY_NS_OK;
}

int batch_info(const crispy_ns_batch *b, int *streams_per_cta, int *n_ctas, int64_t *launches,
                         int64_t *frames_done) {  // (rnn_streams_per_cta, chunk_frames, ...)
  if (!b) return fail(CRISPY_NS_EINVAL, "batch_info: null handle");
  if (streams_per_cta) *streams_per_cta = b->rnn_tc5 ? ns::tc5::kStreams : ns::kMmaStreams;
  if (n_ctas) *n_ctas = b->chunk_cap;
  if (launches) *launches = b->launches;
  if (frames_done) *frames_done = b->frames_done;
  return CRISPY_NS_OK;
}

int kernel_count(void) { return kNumKernels; }
const char *kernel_name(int k) {
  static const char *names[kNumKernels] = {"ns_highpass_kernel", "ns_pitch_kernel",    "ns_pitchscan_kernel", "ns_spectrum_kernel",
                                           "ns_features_kernel", "ns_rnn_kernel",      "ns_synthesis_kernel"};
  return (k >= 0 && k < kNumKernels) ? names[k] : "";
}
int batch_profile(crispy_ns_batch *b, int enable) {
  if (!b) return fail(CRISPY_NS_EINVAL, "batch_profile: null handle");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaDeviceSynchronize());
  prof_clear(b);
  b->prof_on = enable != 0;
  return CRISPY_NS_OK;
}
int batch_profile_read(crispy_ns_batch *b, double *ms_total, int64_t *n_launches, int n_kernels) {
  if (!b || !ms_total || !n_launches || n_kernels < kNumKernels) return fail(CRISPY_NS_EINVAL, "batch_profile_read: bad argument");
  NS_CUDA(cudaSetDevice(b->device));
  NS_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < n_kernels; k++) {
    ms_total[k] = 0.0;
    n_launches[k] = 0;
  }
  for (auto &r : b->prof) {
    float ms = 0.f;
    NS_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    ms_total[r.kernel] += ms;
    n_launches[r.kernel] += 1;
  }
  prof_clear(b);
  return CRISPY_NS_OK;
}

int host_alloc(void **ptr, size_t bytes) {
  if (!ptr) return fail(CRISPY_NS_EINVAL, "host_alloc: null");
  NS_CUDA(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
  return CRISPY_NS_OK;
}
void host_free(void *ptr) {
  if (ptr) cudaFreeHost(ptr);
}

// ---- single stream: DenoiseState ------------------------------------------------------------------
void destroy(crispy_ns_state *st) {
  if (!st) return;
  if (st->b) cudaSetDevice(st->b->device);
  for (int i = 0; i < kSlots; i++)
    if (st->gexec[i]) cudaGraphExecDestroy(st->gexec[i]);
  if (st->s) cudaStreamDestroy(st->s);
  if (st->h_pin) cudaFreeHost(st->h_pin);
  if (st->d_io) cudaFree(st->d_io);
  batch_destroy(st->b);
  delete st;
}
int create(const crispy_ns_model *model, int device, crispy_ns_state **out) {
  if (!out) return fail(CRISPY_NS_EINVAL, "create: out is null");
  crispy_ns_state *st = new (std::nothrow) crispy_ns_state();
  if (!st) return fail(CRISPY_NS_ENOMEM, "out of memory");
  int rc = batch_create(model, device, 1, &st->b);
  if (rc != CRISPY_NS_OK) {
    delete st;
    return rc;
  }
  cudaError_t e = cudaHostAlloc((void **)&st->h_pin, 964 * sizeof(float), cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaMalloc((void **)&st->d_io, 964 * sizeof(float));
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st->s, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    destroy(st);
    return fail(CRISPY_NS_ECUDA, std::string("create: ") + cudaGetErrorString(e));
  }
  *out = st;
  return CRISPY_NS_OK;
}
// one frame of the state's single stream as a captured graph on st->s (built on the first use of each slot)
static int frame_graph(crispy_ns_state *st, int slot) {
  crispy_ns_batch *b = st->b;
  ns::Params p;
  memset(&p, 0, sizeof(p));
  p.in = st->d_io;
  p.out = st->d_io + 480;
  p.vad = st->d_io + 960;
  p.state = b->d_state;
  p.tables = b->d_tables;
  p.rnn_hdr = b->d_hdr;
  p.rnn_words = b->d_words;
  p.rnn_bias = b->d_bias;
  p.in_stride = 480;
  p.out_stride = 480;
  p.vad_stride = 1;
  p.hp_stride = ns::kHist + (long long)b->chunk_cap * ns::kFrame;
  p.n_streams = 1;
  p.n_frames_call = 1;
  p.n_frames = 1;
  p.chunk_cap = b->chunk_cap;
  p.volume = 1.0f;
  p.hp = b->d_hp[slot];
  p.tab = b->d_tab[slot];
  p.rec = b->d_rec[slot];
  p.spec = b->d_spec[slot];
  p.featq = b->d_featq[slot];
  p.synth_sel = slot & 1;  // == chunk counter & 1: kSlots is even
  static_assert(kSlots % 2 == 0, "the synthesis_mem parity follows the slot");
  NS_CUDA(cudaStreamBeginCapture(st->s, cudaStreamCaptureModeThreadLocal));
  cudaMemcpyAsync(st->d_io, st->h_pin, ns::kFrame * sizeof(float), cudaMemcpyHostToDevice, st->s);
  for (int k = 0; k < kNumKernels; k++) launch_kernel(b, k, p, 1, 1, 1, st->s, b->hp_par, b->hp_exclusive);
  cudaMemcpyAsync(st->h_pin + 480, st->d_io + 480, 481 * sizeof(float), cudaMemcpyDeviceToHost, st->s);
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(st->s, &graph);
  if (e != cudaSuccess || !graph) {
    cudaGetLastError();
    return fail(CRISPY_NS_ECUDA, std::string("process_frame: graph capture: ") + cudaGetErrorString(e));
  }
  const cudaError_t ei = cudaGraphInstantiate(&st->gexec[slot], graph, 0);
  cudaGraphDestroy(graph);
  if (ei != cudaSuccess) return fail(CRISPY_NS_ECUDA, std::string("process_frame: graph instantiate: ") + cudaGetErrorString(ei));
  return CRISPY_NS_OK;
}

int process_frame(crispy_ns_state *st, float *out480, const float *in480, float *vad) {
  if (!st || !out480 || !in480) return fail(CRISPY_NS_EINVAL, "process_frame: bad argument");
  crispy_ns_batch *b = st->b;
  NS_CUDA(cudaSetDevice(b->device));
  memcpy(st->h_pin, in480, ns::kFrame * sizeof(float));
  if (b->prof_on || b->reset_pending || getenv("CRISPY_NS_NO_GRAPH")) {  // plain launches (measurement / async reset)
    NS_CUDA(cudaMemcpyAsync(st->d_io, st->h_pin, ns::kFrame * sizeof(float), cudaMemcpyHostToDevice, 0));
    const int rc = run_device(b, st->d_io, st->d_io + 480, st->d_io + 960, nullptr, nullptr, 1, 480, 480, 1, 0, 0, 1.0f, 0);
    if (rc != CRISPY_NS_OK) return rc;
    NS_CUDA(cudaMemcpyAsync(st->h_pin + 480, st->d_io + 480, 481 * sizeof(float), cudaMemcpyDeviceToHost, 0));
    NS_CUDA(cudaStreamSynchronize(0));
  } else {
    const int slot = (int)(b->chunks_done % kSlots);
    if (!st->gexec[slot]) {
      NS_CUDA(configure_kernels(b->device));
      const int rc = frame_graph(st, slot);
      if (rc != CRISPY_NS_OK) return rc;
    }
    NS_CUDA(cudaGraphLaunch(st->gexec[slot], st->s));
    NS_CUDA(cudaStreamSynchronize(st->s));
    b->launches += kNumKernels;
    b->chunks_done += 1;
    b->frames_done += 1;
  }
  memcpy(out480, st->h_pin + 480, ns::kFrame * sizeof(float));
  if (vad) *vad = st->h_pin[960];
  return CRISPY_NS_OK;
}
int reset(crispy_ns_state *st) {
  if (!st) return fail(CRISPY_NS_EINVAL, "reset: null handle");
  return batch_reset(st->b);
}
// the graphs read the controls from the state row, so they need no new capture
int set_controls(crispy_ns_state *st, const void *c) {
  if (!st) return fail(CRISPY_NS_EINVAL, "set_controls: null handle");
  const int id = 0;
  if (int rc = batch_set_controls(st->b, &id, 1, c, st->s)) return rc;
  NS_CUDA(cudaStreamSynchronize(st->s));
  return CRISPY_NS_OK;
}
int get_controls(crispy_ns_state *st, void *out) {
  if (!st) return fail(CRISPY_NS_EINVAL, "get_controls: null handle");
  const int id = 0;
  return batch_get_controls(st->b, &id, 1, out);
}

// ---- a4 / f2: LinearResampler -------------------------------------------------------------------
struct ResampleTable {
  std::vector<int32_t> idx;
  std::vector<float> frac;
};
// Replays LinearResampler::process_sample's position arithmetic (audio.rs:108-133) for n_in input
// samples and records, for each emitted sample, the index of the "current" input and t.
static void build_resample_table(float input_rate, float output_rate, int64_t n_in, ResampleTable &t) {
  t.idx.clear();
  t.frac.clear();
  double input_pos = 0.0, next_output_pos = 0.0;
  const double step = (double)(input_rate / output_rate);
  for (int64_t i = 1; i < n_in; i++) {  // sample 0 only primes the state
    input_pos += 1.0;
    while (next_output_pos <= input_pos) {
      float f = (float)(next_output_pos - (input_pos - 1.0));
      f = f < 0.f ? 0.f : (f > 1.f ? 1.f : f);
      t.idx.push_back((int32_t)i);
      t.frac.push_back(f);
      next_output_pos += step;
    }
  }
}
namespace {
struct LinKey {
  int device;
  uint32_t in_rate_bits, out_rate_bits;
  int64_t n_in;
  bool operator<(const LinKey &o) const {
    return std::tie(device, in_rate_bits, out_rate_bits, n_in) < std::tie(o.device, o.in_rate_bits, o.out_rate_bits, o.n_in);
  }
};
struct LinEntry {
  int32_t *d_idx = nullptr;
  float *d_frac = nullptr;
  int64_t n_out = 0;
};
std::mutex g_lin_mu;
std::map<LinKey, LinEntry> g_lin_tables;  // device copies of the (index, fraction) tables
}  // namespace
int64_t linear_resample_count(float input_rate, float output_rate, int64_t n_in) {
  if (n_in <= 0) return 0;
  const float d = input_rate - output_rate;
  if ((d < 0 ? -d : d) < 1.0f) return n_in;
  // the count comes out of the same f64 replay as the table; remembered per (rates, n_in) so that asking for it
  // before every call does not replay a whole recording's positions on the host each time
  static std::mutex mu;
  static std::map<std::tuple<uint32_t, uint32_t, int64_t>, int64_t> counts;
  uint32_t ri, ro;
  memcpy(&ri, &input_rate, 4);
  memcpy(&ro, &output_rate, 4);
  const auto key = std::make_tuple(ri, ro, n_in);
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = counts.find(key);
    if (it != counts.end()) return it->second;
  }
  ResampleTable t;
  build_resample_table(input_rate, output_rate, n_in, t);
  const int64_t n = (int64_t)t.idx.size();
  std::lock_guard<std::mutex> lk(mu);
  if (counts.size() >= 256) counts.clear();
  counts[key] = n;
  return n;
}
int linear_resample(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in,
                              int64_t in_stride, int64_t out_stride, float input_rate,
                              float output_rate, void *cuda_stream) {
  if (!d_in || !d_out || n_streams < 1 || n_in < 0) return fail(CRISPY_NS_EINVAL, "linear_resample: bad argument");
  if (n_in >= (1ll << 31)) return fail(CRISPY_NS_EINVAL, "linear_resample: n_in too large for one call");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  NS_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const float d = input_rate - output_rate;
  if ((d < 0 ? -d : d) < 1.0f) {  // audio.rs:109-112 passthrough
    NS_CUDA(cudaMemcpy2DAsync(d_out, (size_t)out_stride * 4, d_in, (size_t)in_stride * 4, (size_t)n_in * 4,
                              n_streams, cudaMemcpyDeviceToDevice, st));
    return CRISPY_NS_OK;
  }
  // The (index, fraction) table depends only on (rates, n_in): it is built and uploaded once per device and kept
  // (like the sinc taps), so the call itself is asynchronous on `st` and capturable in a CUDA graph.
  int32_t *d_idx = nullptr;
  float *d_frac = nullptr;
  int64_t n_out = 0;
  {
    std::lock_guard<std::mutex> lk(g_lin_mu);
    uint32_t ri, ro;
    memcpy(&ri, &input_rate, 4);
    memcpy(&ro, &output_rate, 4);
    const LinKey key{device, ri, ro, n_in};
    auto it = g_lin_tables.find(key);
    if (it == g_lin_tables.end()) {
      if (g_lin_tables.size() >= 32) {  // bounded cache: drop everything once no stream can still be reading it
        NS_CUDA(cudaDeviceSynchronize());
        for (auto &kv : g_lin_tables) {
          cudaSetDevice(kv.first.device);
          cudaFree(kv.second.d_idx);
          cudaFree(kv.second.d_frac);
        }
        g_lin_tables.clear();
        NS_CUDA(cudaSetDevice(device));
      }
      ResampleTable t;
      build_resample_table(input_rate, output_rate, n_in, t);
      LinEntry e;
      e.n_out = (int64_t)t.idx.size();
      if (e.n_out > 0) {
        NS_CUDA(cudaMalloc((void **)&e.d_idx, (size_t)e.n_out * 4));
        if (cudaError_t ce = cudaMalloc((void **)&e.d_frac, (size_t)e.n_out * 4); ce != cudaSuccess) {
          cudaFree(e.d_idx);
          return fail(CRISPY_NS_ECUDA, std::string("linear_resample: ") + cudaGetErrorString(ce));
        }
        // synchronous copies from the pageable host table: done before it goes out of scope
        NS_CUDA(cudaMemcpy(e.d_idx, t.idx.data(), (size_t)e.n_out * 4, cudaMemcpyHostToDevice));
        NS_CUDA(cudaMemcpy(e.d_frac, t.frac.data(), (size_t)e.n_out * 4, cudaMemcpyHostToDevice));
      }
      it = g_lin_tables.emplace(key, e).first;
    }
    d_idx = it->second.d_idx;
    d_frac = it->second.d_frac;
    n_out = it->second.n_out;
  }
  if (n_out == 0) return CRISPY_NS_OK;
  int gx = (int)((n_out + 4095) / 4096);  // 256 threads x 4 outputs x 4 trips per CTA
  if (gx < 1) gx = 1;
  dim3 grid(gx, n_streams);
  const int vec_store = ((uintptr_t)d_out % 16) == 0 && (out_stride % 4) == 0;
  ns_linear_resample_kernel<<<grid, 256, 0, st>>>(d_in, d_out, d_idx, d_frac, n_out, in_stride, out_stride, vec_store);
  NS_CUDA(cudaGetLastError());
  return CRISPY_NS_OK;
}

// ---- the capture callbacks' downmix to mono (audio.rs:754-755, :816-818, :879-884) ---------------------
template <typename T>
static int downmix_launch(const void *d_in, int n_channels, float *d_out, int n_streams, int64_t n_frames, int64_t in_stride,
                          int64_t out_stride, cudaStream_t st) {
  const T *in = static_cast<const T *>(d_in);
  const bool vec_ok = n_channels == 2 && ((uintptr_t)d_in % 16) == 0 && ((uintptr_t)d_out % 16) == 0 &&
                      ((in_stride * (int64_t)sizeof(T)) % 16) == 0 && (out_stride % 4) == 0;
  if (vec_ok) {
    constexpr int64_t tile = 256 * (16 / (int64_t)sizeof(T)) * kDownmixTrips;
    const int64_t gx = (n_frames + tile - 1) / tile;
    if (gx > 0x7fffffffll) return CRISPY_NS_EINVAL;
    ns_downmix_stereo_kernel<T><<<dim3((unsigned)gx, n_streams), 256, 0, st>>>(in, d_out, n_frames, in_stride, out_stride);
  } else {
    int gx = (int)((n_frames + 255) / 256);
    if (gx > 148 * 16) gx = 148 * 16;
    ns_downmix_kernel<T><<<dim3(gx, n_streams), 256, 0, st>>>(in, d_out, n_channels, n_frames, in_stride, out_stride);
  }
  return cudaGetLastError() == cudaSuccess ? CRISPY_NS_OK : CRISPY_NS_ECUDA;
}
int downmix_mono(int device, const void *d_in, int sample_format, int n_channels, float *d_out, int n_streams,
                 int64_t n_frames, int64_t in_stride, int64_t out_stride, void *cuda_stream) {
  if (n_streams < 1 || n_frames < 0 || n_channels < 1 || n_channels > 64 || sample_format < 0 || sample_format > 2)
    return fail(CRISPY_NS_EINVAL, "downmix_mono: bad argument");
  if (n_frames == 0) return CRISPY_NS_OK;
  if (!d_in || !d_out || n_streams > 65535) return fail(CRISPY_NS_EINVAL, "downmix_mono: bad argument");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  NS_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  int rc;
  if (sample_format == CRISPY_NS_FMT_F32)
    rc = downmix_launch<float>(d_in, n_channels, d_out, n_streams, n_frames, in_stride, out_stride, st);
  else if (sample_format == CRISPY_NS_FMT_I16)
    rc = downmix_launch<int16_t>(d_in, n_channels, d_out, n_streams, n_frames, in_stride, out_stride, st);
  else
    rc = downmix_launch<uint16_t>(d_in, n_channels, d_out, n_streams, n_frames, in_stride, out_stride, st);
  if (rc != CRISPY_NS_OK) return fail(CRISPY_NS_ECUDA, "downmix_mono: kernel launch failed");
  return CRISPY_NS_OK;
}

// ---- f2, app audio: resample_audio (recording.rs:13-39) ---------------------------------------------
int64_t resample_audio_count(int64_t n_in, int from_rate, int to_rate) {
  if (n_in <= 0 || from_rate < 1 || to_rate < 1) return 0;
  if (from_rate == to_rate) return n_in;  // recording.rs:14-16
  const double ratio = (double)from_rate / (double)to_rate;
  int64_t n_out = (int64_t)ceil((double)n_in / ratio);  // recording.rs:19
  // recording.rs:27-35 pushes nothing once floor(i * ratio) reaches the end of the input: trailing outputs only
  while (n_out > 0 && (int64_t)floor((double)(n_out - 1) * ratio) >= n_in) n_out--;
  return n_out;
}
int resample_audio(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in, int64_t in_stride,
                   int64_t out_stride, int from_rate, int to_rate, void *cuda_stream) {
  if (!d_in || !d_out || n_streams < 1 || n_in < 0 || from_rate < 1 || to_rate < 1)
    return fail(CRISPY_NS_EINVAL, "resample_audio: bad argument");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  if (n_streams > 65535) return fail(CRISPY_NS_EINVAL, "resample_audio: too many streams for one call");
  NS_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (n_in == 0) return CRISPY_NS_OK;
  if (from_rate == to_rate) {
    NS_CUDA(cudaMemcpy2DAsync(d_out, (size_t)out_stride * 4, d_in, (size_t)in_stride * 4, (size_t)n_in * 4, n_streams,
                              cudaMemcpyDeviceToDevice, st));
    return CRISPY_NS_OK;
  }
  const int64_t n_out = resample_audio_count(n_in, from_rate, to_rate);
  if (n_out == 0) return CRISPY_NS_OK;
  int gx = (int)((n_out + 4095) / 4096);  // 256 threads x 4 outputs x 4 trips per CTA
  const int vec_store = ((uintptr_t)d_out % 16) == 0 && (out_stride % 4) == 0;
  ns_resample_audio_kernel<<<dim3(gx, n_streams), 256, 0, st>>>(d_in, d_out, n_in, n_out, in_stride, out_stride,
                                                                (double)from_rate / (double)to_rate, vec_store);
  NS_CUDA(cudaGetLastError());
  return CRISPY_NS_OK;
}

// ---- f2 (north_star item 4): windowed-sinc polyphase resampler -------------------------------------
// rubato 0.16.2 (Cargo.lock:4166) synchronous sinc design -- make_sincs with the BlackmanHarris2
// window, sinc_len taps, f_cutoff relative to Nyquist (scaled by the ratio when downsampling) --
// with the oversampling factor equal to L of the reduced ratio L/M, so every output lands on a
// tabulated phase.  Delay-compensated; zeros outside the input.
namespace {
struct SincKey {
  int device, L, M, sinc_len;
  float f_cutoff;
  bool operator<(const SincKey &o) const {
    return std::tie(device, L, M, sinc_len, f_cutoff) < std::tie(o.device, o.L, o.M, o.sinc_len, o.f_cutoff);
  }
};
std::mutex g_sinc_mu;
std::map<SincKey, float *> g_sinc_tables;  // device copies, [sinc_len][L]; live until process exit
std::map<SincKey, float *> g_sinc_tables_out_order;  // the same taps with the columns in output order (ns_sinc_resample4_kernel)

int reduce_ratio(int input_rate, int output_rate, int *L, int *M) {
  if (input_rate < 1 || output_rate < 1) return 0;
  int a = input_rate, b = output_rate;
  while (b) {
    const int t = a % b;
    a = b;
    b = t;
  }
  *L = output_rate / a;
  *M = input_rate / a;
  return *L <= 1024;
}
// taps[k*L + p]: the filter sampled (k - half + 1) - p/L input samples from the interpolation point
void sinc_taps_transposed(int L, int M, int sinc_len, float f_cutoff, std::vector<float> &taps) {
  const double kPi = 3.14159265358979323846;
  double fc = (double)f_cutoff;
  if (L < M) fc = fc * (double)L / (double)M;
  const long tot = (long)sinc_len * L;
  std::vector<double> y((size_t)tot);
  double sum = 0.0;
  for (long x = 0; x < tot; x++) {
    const double t = ((double)x - (double)(tot / 2)) * fc / (double)L;
    const double s = t == 0.0 ? 1.0 : sin(kPi * t) / (kPi * t);
    const double a = 2.0 * kPi * (double)x / (double)tot;
    const double w = 0.35875 - 0.48829 * cos(a) + 0.14128 * cos(2.0 * a) - 0.01168 * cos(3.0 * a);
    y[(size_t)x] = w * w * s;
    sum += y[(size_t)x];
  }
  sum /= (double)L;
  taps.assign((size_t)tot, 0.f);
  for (int k = 0; k < sinc_len; k++)
    for (int p = 0; p < L; p++) {
      const long x = (long)L * (k + 1) - p;
      if (x < tot) taps[(size_t)k * L + p] = (float)(y[(size_t)x] / sum);
    }
}
}  // namespace

int64_t sinc_resample_count(int input_rate, int output_rate, int64_t n_in) {
  int L, M;
  if (n_in <= 0 || !reduce_ratio(input_rate, output_rate, &L, &M)) return 0;
  return (int64_t)(((unsigned long long)n_in * (unsigned)L + (unsigned)M - 1) / (unsigned)M);
}
int sinc_resample_needed(int input_rate, int output_rate, int sinc_len, int64_t n_total, int64_t first_out,
                                   int64_t n_out, int64_t *in_first, int64_t *n_in) {
  int L, M;
  if (sinc_len == 0) sinc_len = 256;
  if (!reduce_ratio(input_rate, output_rate, &L, &M) || n_total < 0 || first_out < 0 || n_out < 0 || sinc_len < 2 || (sinc_len & 1))
    return fail(CRISPY_NS_EINVAL, "sinc_resample_needed: bad argument");
  if (n_out == 0) {
    if (in_first) *in_first = 0;
    if (n_in) *n_in = 0;
    return CRISPY_NS_OK;
  }
  const long long half = sinc_len / 2;
  long long lo = (long long)((unsigned long long)first_out * (unsigned)M / (unsigned)L) - half + 1;
  long long hi = (long long)((unsigned long long)(first_out + n_out - 1) * (unsigned)M / (unsigned)L) + half + 1;  // exclusive
  if (lo < 0) lo = 0;
  if (hi > n_total) hi = n_total;
  if (hi < lo) hi = lo;
  if (in_first) *in_first = lo;
  if (n_in) *n_in = hi - lo;
  return CRISPY_NS_OK;
}

int sinc_resample_chunk(int device, const float *d_in, int64_t in_first, int64_t n_in, int64_t n_total,
                                  float *d_out, int64_t first_out, int64_t n_out, int n_streams, int64_t in_stride,
                                  int64_t out_stride, int input_rate, int output_rate, int sinc_len, float f_cutoff,
                                  void *cuda_stream) {
  if (!d_in || !d_out || n_streams < 1 || n_in < 0 || n_total < 0 || in_first < 0 || first_out < 0 || n_out < 0)
    return fail(CRISPY_NS_EINVAL, "sinc_resample: bad argument");
  if (sinc_len == 0) sinc_len = 256;
  if (f_cutoff == 0.f) f_cutoff = 0.95f;
  if (sinc_len < 2 || sinc_len > 2048 || (sinc_len & 1) || !(f_cutoff > 0.f) || f_cutoff > 1.f)
    return fail(CRISPY_NS_EINVAL, "sinc_resample: sinc_len must be even in [2, 2048], f_cutoff in (0, 1]");
  int L, M;
  if (!reduce_ratio(input_rate, output_rate, &L, &M))
    return fail(CRISPY_NS_EINVAL, "sinc_resample: output_rate/input_rate must reduce to L/M with L <= 1024");
  if (M >= (1 << 20)) return fail(CRISPY_NS_EINVAL, "sinc_resample: ratio too extreme");
  if (first_out % L) return fail(CRISPY_NS_EINVAL, "sinc_resample: first_out must be a multiple of L (a whole number of periods)");
  if (first_out + n_out > sinc_resample_count(input_rate, output_rate, n_total))
    return fail(CRISPY_NS_EINVAL, "sinc_resample: outputs beyond the end of the recording");
  {
    int64_t need_first = 0, need_n = 0;
    sinc_resample_needed(input_rate, output_rate, sinc_len, n_total, first_out, n_out, &need_first, &need_n);
    if (need_n > 0 && (need_first < in_first || need_first + need_n > in_first + n_in))
      return fail(CRISPY_NS_EINVAL, "sinc_resample: the input window does not cover the taps of the requested outputs "
                                    "(crispy_ns_sinc_resample_needed gives the range)");
  }
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  NS_CUDA(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (n_out == 0) return CRISPY_NS_OK;
  float *d_taps = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_sinc_mu);
    const SincKey key{device, L, M, sinc_len, f_cutoff};
    auto it = g_sinc_tables.find(key);
    if (it == g_sinc_tables.end()) {
      std::vector<float> taps;
      sinc_taps_transposed(L, M, sinc_len, f_cutoff, taps);
      NS_CUDA(cudaMalloc((void **)&d_taps, taps.size() * sizeof(float)));
      NS_CUDA(cudaMemcpy(d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
      g_sinc_tables[key] = d_taps;
    } else {
      d_taps = it->second;
    }
  }
  // samples of the recording the kernel may read: the caller's window, clipped to the recording
  const long long in_end_all = (in_first + n_in < n_total) ? in_first + n_in : n_total;
  if (n_streams > 65535) return fail(CRISPY_NS_EINVAL, "sinc_resample: too large for one call");
  // second-generation kernel: four adjacent outputs per thread (2/3 <= M/L < 1, L a multiple of 4)
  if (M < L && 3 * (long long)M >= 2 * (long long)L && L % 4 == 0 && !getenv("CRISPY_NS_SINC_V1")) {
    const int unit = L / 4;                       // T * 4 must be a multiple of L
    int T = unit * ((160 + unit - 1) / unit);
    if (T <= 256) {
      constexpr int Q = 8;
      const long long tile = (long long)T * 4 * Q;
      const long long span = tile / L * M + sinc_len + 4;
      const size_t smem = (size_t)span * sizeof(float);
      const long long tiles = (n_out + tile - 1) / tile;
      if (smem <= 96 * 1024 && tiles <= 0x7fffffffll) {
        float *d_taps4 = nullptr;
        {
          std::lock_guard<std::mutex> lk(g_sinc_mu);
          const SincKey key{device, L, M, sinc_len, f_cutoff};
          auto it = g_sinc_tables_out_order.find(key);
          if (it == g_sinc_tables_out_order.end()) {
            std::vector<float> taps, taps4;
            sinc_taps_transposed(L, M, sinc_len, f_cutoff, taps);
            taps4.resize(taps.size());
            for (int k = 0; k < sinc_len; k++)
              for (int u = 0; u < L; u++) taps4[(size_t)k * L + u] = taps[(size_t)k * L + (size_t)(((long long)u * M) % L)];
            NS_CUDA(cudaMalloc((void **)&d_taps4, taps4.size() * sizeof(float)));
            NS_CUDA(cudaMemcpy(d_taps4, taps4.data(), taps4.size() * sizeof(float), cudaMemcpyHostToDevice));
            g_sinc_tables_out_order[key] = d_taps4;
          } else {
            d_taps4 = it->second;
          }
        }
        if (smem > 48 * 1024)
          NS_CUDA(cudaFuncSetAttribute(ns_sinc_resample4_kernel<Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int vec_store = ((uintptr_t)d_out % 16) == 0 && (out_stride % 4) == 0;
        ns_sinc_resample4_kernel<Q><<<dim3((unsigned)tiles, (unsigned)n_streams), T, smem, st>>>(
            d_in, d_out, d_taps4, n_total, in_first, in_end_all, first_out, n_out, in_stride, out_stride, L, M, sinc_len, (int)span,
            vec_store);
        NS_CUDA(cudaGetLastError());
        return CRISPY_NS_OK;
      }
    }
  }
  // threads: a multiple of L near 160-256; outputs per thread Q in {8, 4, 2, 1} so the staged span fits
  int T = L * ((160 + L - 1) / L);
  if (T > 1024) T = L;
  const int per = T / L * M;  // input samples advanced per T outputs
  int Q = 8;
  auto span_of = [&](int q) { return (long long)per * q + sinc_len + 1; };
  while (Q > 1 && span_of(Q) * 4 > 96 * 1024) Q >>= 1;
  const long long span = span_of(Q);
  if (span * 4 > 200 * 1024) return fail(CRISPY_NS_EINVAL, "sinc_resample: decimation ratio too large for one tile");
  const size_t smem = (size_t)span * sizeof(float);
  const long long tiles = (n_out + (long long)T * Q - 1) / ((long long)T * Q);
  // samples of the recording the kernel may read: the caller's window, clipped to the recording
  const long long in_end = (in_first + n_in < n_total) ? in_first + n_in : n_total;
  if (tiles > 0x7fffffffll || n_streams > 65535) return fail(CRISPY_NS_EINVAL, "sinc_resample: too large for one call");
  dim3 grid((unsigned)tiles, (unsigned)n_streams);
#define NS_SINC_LAUNCH(QQ)                                                                               \
  do {                                                                                                   \
    if (smem > 48 * 1024)                                                                                \
      NS_CUDA(cudaFuncSetAttribute(ns_sinc_resample_kernel<QQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)smem));                                                          \
    ns_sinc_resample_kernel<QQ><<<grid, T, smem, st>>>(d_in, d_out, d_taps, n_total, in_first, in_end, first_out, n_out, \
                                                       in_stride, out_stride, L, M, sinc_len, (int)span); \
  } while (0)
  switch (Q) {
    case 8: NS_SINC_LAUNCH(8); break;
    case 4: NS_SINC_LAUNCH(4); break;
    case 2: NS_SINC_LAUNCH(2); break;
    default: NS_SINC_LAUNCH(1); break;
  }
#undef NS_SINC_LAUNCH
  NS_CUDA(cudaGetLastError());
  return CRISPY_NS_OK;
}

int sinc_resample(int device, const float *d_in, float *d_out, int n_streams, int64_t n_in,
                            int64_t in_stride, int64_t out_stride, int input_rate, int output_rate,
                            int sinc_len, float f_cutoff, void *cuda_stream) {
  if (n_in < 0) return fail(CRISPY_NS_EINVAL, "sinc_resample: bad argument");
  int L, M;
  if (!reduce_ratio(input_rate, output_rate, &L, &M))
    return fail(CRISPY_NS_EINVAL, "sinc_resample: output_rate/input_rate must reduce to L/M with L <= 1024");
  return sinc_resample_chunk(device, d_in, 0, n_in, n_in, d_out, 0,
                                       sinc_resample_count(input_rate, output_rate, n_in), n_streams, in_stride,
                                       out_stride, input_rate, output_rate, sinc_len, f_cutoff, cuda_stream);
}

int resample_host(int device, const float *h_in, float *h_out, int n_streams, int64_t n_in,
                            int64_t in_stride, int64_t out_stride, int input_rate, int output_rate, int kind) {
  if (!h_in || !h_out || n_streams < 1 || n_in < 0 || kind < 0 || kind > 2)
    return fail(CRISPY_NS_EINVAL, "resample_host: bad argument");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  const int64_t n_out = kind == 0   ? linear_resample_count((float)input_rate, (float)output_rate, n_in)
                        : kind == 1 ? sinc_resample_count(input_rate, output_rate, n_in)
                                    : resample_audio_count(n_in, input_rate, output_rate);
  if (n_in == 0 || n_out == 0) return CRISPY_NS_OK;
  NS_CUDA(cudaSetDevice(device));
  float *d_in = nullptr, *d_out = nullptr;
  NS_CUDA(cudaMalloc((void **)&d_in, (size_t)n_streams * n_in * sizeof(float)));
  if (cudaError_t e = cudaMalloc((void **)&d_out, (size_t)n_streams * n_out * sizeof(float)); e != cudaSuccess) {
    cudaFree(d_in);
    return fail(CRISPY_NS_ECUDA, std::string("resample_host: ") + cudaGetErrorString(e));
  }
  int rc = CRISPY_NS_OK;
  cudaError_t e = cudaMemcpy2D(d_in, (size_t)n_in * 4, h_in, (size_t)in_stride * 4, (size_t)n_in * 4, n_streams,
                               cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    rc = kind == 0   ? linear_resample(device, d_in, d_out, n_streams, n_in, n_in, n_out, (float)input_rate, (float)output_rate, nullptr)
         : kind == 1 ? sinc_resample(device, d_in, d_out, n_streams, n_in, n_in, n_out, input_rate, output_rate, 0, 0.f, nullptr)
                     : resample_audio(device, d_in, d_out, n_streams, n_in, n_in, n_out, input_rate, output_rate, nullptr);
    if (rc == CRISPY_NS_OK && cudaStreamSynchronize(nullptr) != cudaSuccess) rc = fail(CRISPY_NS_ECUDA, "resample_host: kernel failed");
    if (rc == CRISPY_NS_OK)
      e = cudaMemcpy2D(h_out, (size_t)out_stride * 4, d_out, (size_t)n_out * 4, (size_t)n_out * 4, n_streams,
                       cudaMemcpyDeviceToHost);
  }
  cudaFree(d_in);
  cudaFree(d_out);
  if (rc != CRISPY_NS_OK) return rc;
  if (e != cudaSuccess) return fail(CRISPY_NS_ECUDA, std::string("resample_host: ") + cudaGetErrorString(e));
  return CRISPY_NS_OK;
}

// ---- f3: WAV PCM16 -------------------------------------------------------------------------------
static void le16(uint8_t *p, uint32_t v) {
  p[0] = (uint8_t)v;
  p[1] = (uint8_t)(v >> 8);
}
static void le32(uint8_t *p, uint32_t v) {
  p[0] = (uint8_t)v;
  p[1] = (uint8_t)(v >> 8);
  p[2] = (uint8_t)(v >> 16);
  p[3] = (uint8_t)(v >> 24);
}
int wav_write_pcm16(const char *path, const int16_t *interleaved, int64_t n_frames, int channels,
                              int sample_rate) {
  if (!path || (!interleaved && n_frames > 0) || n_frames < 0 || channels < 1 || sample_rate < 1)
    return fail(CRISPY_NS_EINVAL, "wav_write: bad argument");
  const uint64_t data_bytes = (uint64_t)n_frames * channels * 2;
  if (data_bytes > 0xFFFFFFFFull - 36) return fail(CRISPY_NS_EINVAL, "wav_write: too large for RIFF");
  FILE *f = fopen(path, "wb");
  if (!f) return fail(CRISPY_NS_EIO, std::string("wav_write: cannot open ") + path);
  uint8_t h[44];
  memcpy(h, "RIFF", 4);
  le32(h + 4, (uint32_t)(36 + data_bytes));
  memcpy(h + 8, "WAVEfmt ", 8);
  le32(h + 16, 16);
  le16(h + 20, 1);
  le16(h + 22, (uint32_t)channels);
  le32(h + 24, (uint32_t)sample_rate);
  le32(h + 28, (uint32_t)(sample_rate * channels * 2));
  le16(h + 32, (uint32_t)(channels * 2));
  le16(h + 34, 16);
  memcpy(h + 36, "data", 4);
  le32(h + 40, (uint32_t)data_bytes);
  bool ok = fwrite(h, 1, 44, f) == 44;
  if (ok && data_bytes) ok = fwrite(interleaved, 1, data_bytes, f) == data_bytes;
  ok = (fclose(f) == 0) && ok;
  return ok ? CRISPY_NS_OK : fail(CRISPY_NS_EIO, "wav_write: short write");
}
int wav_read_pcm16(const char *path, int16_t *interleaved, int64_t cap_samples, int64_t *n_frames,
                             int *channels, int *sample_rate) {
  if (!path) return fail(CRISPY_NS_EINVAL, "wav_read: bad argument");
  FILE *f = fopen(path, "rb");
  if (!f) return fail(CRISPY_NS_EIO, std::string("wav_read: cannot open ") + path);
  uint8_t h[12];
  if (fread(h, 1, 12, f) != 12 || memcmp(h, "RIFF", 4) != 0 || memcmp(h + 8, "WAVE", 4) != 0) {
    fclose(f);
    return fail(CRISPY_NS_EIO, "wav_read: not a RIFF/WAVE file");
  }
  int ch = 0, sr = 0, bits = 0, fmt = 0;
  bool have_fmt = false;
  for (;;) {  // chunk walk, as get_wav_duration does (commands/recording.rs:385-460)
    uint8_t c[8];
    if (fread(c, 1, 8, f) != 8) break;
    const uint32_t sz = (uint32_t)c[4] | ((uint32_t)c[5] << 8) | ((uint32_t)c[6] << 16) | ((uint32_t)c[7] << 24);
    if (memcmp(c, "fmt ", 4) == 0) {
      uint8_t fm[40];
      const size_t take = sz < 40 ? sz : 40;
      if (sz < 16 || fread(fm, 1, take, f) != take) break;
      fmt = fm[0] | (fm[1] << 8);
      ch = fm[2] | (fm[3] << 8);
      sr = (int)((uint32_t)fm[4] | ((uint32_t)fm[5] << 8) | ((uint32_t)fm[6] << 16) | ((uint32_t)fm[7] << 24));
      bits = fm[14] | (fm[15] << 8);
      // WAVE_FORMAT_EXTENSIBLE (what hound and ffmpeg write for more than two channels): the sample format is the
      // first field of the sub-format GUID
      if (fmt == 0xFFFE && take >= 26) fmt = fm[24] | (fm[25] << 8);
      have_fmt = true;
      if (sz + (sz & 1) > take) fseek(f, (long)(sz + (sz & 1) - take), SEEK_CUR);
    } else if (memcmp(c, "data", 4) == 0) {
      if (!have_fmt || fmt != 1 || bits != 16 || ch < 1) {
        fclose(f);
        return fail(CRISPY_NS_EIO, "wav_read: only PCM16 is supported");
      }
      int64_t total = (int64_t)sz / 2;
      if (sz == 0xFFFFFFFFu) {  // a writer that could not seek back (ffmpeg to a pipe): the data runs to the end of the file
        const long pos = ftell(f);
        fseek(f, 0, SEEK_END);
        const long end = ftell(f);
        fseek(f, pos, SEEK_SET);
        total = (int64_t)(end > pos ? end - pos : 0) / 2;
      }
      total -= total % ch;
      if (n_frames) *n_frames = total / ch;
      if (channels) *channels = ch;
      if (sample_rate) *sample_rate = sr;
      if (interleaved) {
        const int64_t want = total < cap_samples ? total : cap_samples;
        if ((int64_t)fread(interleaved, 2, (size_t)want, f) != want) {
          fclose(f);
          return fail(CRISPY_NS_EIO, "wav_read: truncated data chunk");
        }
      }
      fclose(f);
      return CRISPY_NS_OK;
    } else {
      fseek(f, (long)(sz + (sz & 1)), SEEK_CUR);
    }
  }
  fclose(f);
  return fail(CRISPY_NS_EIO, "wav_read: no fmt/data chunk");
}


// ---- (e) several GPUs from one process ---------------------------------------------------------------
}  // namespace impl
struct crispy_ns_multi {
  int n_streams = 0;
  std::vector<int> device, first, count;
  std::vector<crispy_ns_batch *> batch;
};
namespace impl {

void multi_destroy(crispy_ns_multi *m) {
  if (!m) return;
  for (crispy_ns_batch *b : m->batch) batch_destroy(b);
  delete m;
}

int multi_create(const crispy_ns_model *model, const int *devices, int n_devices, int n_streams,
                           crispy_ns_multi **out) {
  if (!out || n_devices < 1 || n_streams < 1) return fail(CRISPY_NS_EINVAL, "multi_create: bad argument");
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  crispy_ns_multi *m = new crispy_ns_multi();
  m->n_streams = n_streams;
  // contiguous blocks whose sizes differ by at most one (crispy_b200/shard.py stream_block); devices beyond the
  // stream count stay empty and are skipped
  const int base = n_streams / n_devices, extra = n_streams % n_devices;
  for (int i = 0; i < n_devices; i++) {
    const int cnt = base + (i < extra ? 1 : 0);
    if (cnt == 0) continue;
    const int dev = devices ? devices[i] : i;
    if (dev < 0 || dev >= ndev) {
      multi_destroy(m);
      return fail(CRISPY_NS_ENODEV, "multi_create: device index out of range");
    }
    crispy_ns_batch *b = nullptr;
    const int rc = batch_create(model, dev, cnt, &b);
    if (rc != CRISPY_NS_OK) {
      multi_destroy(m);
      return rc;
    }
    m->device.push_back(dev);
    m->first.push_back(i * base + (i < extra ? i : extra));
    m->count.push_back(cnt);
    m->batch.push_back(b);
  }
  *out = m;
  return CRISPY_NS_OK;
}
int multi_n_devices(const crispy_ns_multi *m) { return m ? (int)m->batch.size() : 0; }
int multi_stream_range(const crispy_ns_multi *m, int i, int *device, int *first_stream, int *n_streams) {
  if (!m || i < 0 || i >= (int)m->batch.size()) return fail(CRISPY_NS_EINVAL, "multi_stream_range: bad argument");
  if (device) *device = m->device[i];
  if (first_stream) *first_stream = m->first[i];
  if (n_streams) *n_streams = m->count[i];
  return CRISPY_NS_OK;
}
int multi_reset(crispy_ns_multi *m) {
  if (!m) return fail(CRISPY_NS_EINVAL, "multi_reset: null handle");
  for (crispy_ns_batch *b : m->batch) {
    const int rc = batch_reset(b);
    if (rc != CRISPY_NS_OK) return rc;
  }
  return CRISPY_NS_OK;
}
// global stream ids -> (device block, local ids, entries); checked whole before anything is enqueued
static int multi_split(const crispy_ns_multi *m, const int *streams, int n, const char *what,
                       std::vector<std::vector<int>> &local, std::vector<std::vector<int>> &entry) {
  if (!m) return fail(CRISPY_NS_EINVAL, std::string(what) + ": null handle");
  if (n < 0 || n > m->n_streams || (n > 0 && !streams))
    return fail(CRISPY_NS_EINVAL, std::string(what) + ": the stream count must be in [0, n_streams] with a stream list");
  std::vector<char> seen((size_t)m->n_streams, 0);
  local.assign(m->batch.size(), {});
  entry.assign(m->batch.size(), {});
  for (int i = 0; i < n; i++) {
    const int s = streams[i];
    if (s < 0 || s >= m->n_streams) return fail(CRISPY_NS_EINVAL, std::string(what) + ": stream id out of range");
    if (seen[(size_t)s]) return fail(CRISPY_NS_EINVAL, std::string(what) + ": stream listed twice");
    seen[(size_t)s] = 1;
    for (size_t d = 0; d < m->batch.size(); d++)
      if (s >= m->first[d] && s < m->first[d] + m->count[d]) {
        local[d].push_back(s - m->first[d]);
        entry[d].push_back(i);
      }
  }
  return CRISPY_NS_OK;
}
int multi_set_controls(crispy_ns_multi *m, const int *streams, int n, const void *controls_v) {
  const crispy_ns_controls *controls = static_cast<const crispy_ns_controls *>(controls_v);
  std::vector<std::vector<int>> local, entry;
  if (int rc = multi_split(m, streams, n, "multi_set_controls", local, entry)) return rc;
  if (int rc = check_controls(controls, n, "multi_set_controls")) return rc;
  for (size_t d = 0; d < m->batch.size(); d++) {
    if (local[d].empty()) continue;
    std::vector<crispy_ns_controls> c;
    for (int i : entry[d]) c.push_back(controls[i]);
    if (int rc = batch_set_controls(m->batch[d], local[d].data(), (int)local[d].size(), c.data(), nullptr)) return rc;
    NS_CUDA(cudaStreamSynchronize(m->batch[d]->s_k[kNumKernels - 1]));
  }
  return CRISPY_NS_OK;
}
int multi_get_controls(crispy_ns_multi *m, const int *streams, int n, void *out_v) {
  crispy_ns_controls *out = static_cast<crispy_ns_controls *>(out_v);
  std::vector<std::vector<int>> local, entry;
  if (int rc = multi_split(m, streams, n, "multi_get_controls", local, entry)) return rc;
  if (n > 0 && !out) return fail(CRISPY_NS_EINVAL, "multi_get_controls: out is null");
  for (size_t d = 0; d < m->batch.size(); d++) {
    if (local[d].empty()) continue;
    std::vector<crispy_ns_controls> c(local[d].size());
    if (int rc = batch_get_controls(m->batch[d], local[d].data(), (int)local[d].size(), c.data())) return rc;
    for (size_t j = 0; j < c.size(); j++) out[entry[d][j]] = c[j];
  }
  return CRISPY_NS_OK;
}
int multi_process_streams_host(crispy_ns_multi *m, const void *h_in, void *h_out, float *h_vad,
                                         const float *h_app, int n_frames, int64_t in_stride, int64_t out_stride,
                                         int64_t vad_stride, int64_t app_stride, uint32_t flags, float volume) {
  if (!m || n_frames < 0 || (n_frames > 0 && (!h_in || !h_out))) return fail(CRISPY_NS_EINVAL, "multi_process_streams_host: bad argument");
  const size_t nd = m->batch.size();
  const size_t ie = in_elem(flags), oe = out_elem(flags);
  std::vector<int> rc(nd, CRISPY_NS_OK);
  std::vector<std::string> err(nd);
  auto work = [&](size_t i) {  // one host thread per device: its copies and launches never wait for another device
    const int64_t s0 = m->first[i];
    rc[i] = guard("multi_process_streams_host", [&]() -> int {
      return process_streams_host(m->batch[i], (const char *)h_in + (size_t)(s0 * in_stride) * ie,
                                            (char *)h_out + (size_t)(s0 * out_stride) * oe,
                                            h_vad ? h_vad + s0 * vad_stride : nullptr,
                                            h_app ? h_app + s0 * app_stride : nullptr, n_frames, in_stride, out_stride,
                                            vad_stride, app_stride, flags, volume);
    });
    if (rc[i] != CRISPY_NS_OK) {
      try {
        err[i] = g_err;  // thread-local: carry the message back to the caller's thread
      } catch (...) {
      }
    }
  };
  std::vector<std::thread> th;
  th.reserve(nd);
  for (size_t i = 1; i < nd; i++) {
    try {
      th.emplace_back(work, i);
    } catch (...) {  // no thread to be had: this device's share runs on the caller's thread (a joinable std::thread
      work(i);       // left behind by an exception would terminate the process)
    }
  }
  work(0);
  for (auto &t : th) t.join();
  for (size_t i = 0; i < nd; i++)
    if (rc[i] != CRISPY_NS_OK) return fail(rc[i], "device " + std::to_string(m->device[i]) + ": " + err[i]);
  return CRISPY_NS_OK;
}

// ---- f3 end to end: WAV files in, dual-mono WAV files out ---------------------------------------------
int denoise_wav_files(const crispy_ns_model *model, int device, const char *const *paths_in,
                                const char *const *paths_out, int n_files, uint32_t flags, float volume,
                                float *mean_vad) {
  if (!paths_in || !paths_out || n_files < 1) return fail(CRISPY_NS_EINVAL, "denoise_wav_files: bad argument");
  if (flags & ~(uint32_t)CRISPY_NS_DROP_FIRST_FRAME) return fail(CRISPY_NS_EINVAL, "denoise_wav_files: only CRISPY_NS_DROP_FIRST_FRAME is accepted");
  std::vector<int64_t> len((size_t)n_files, 0);
  std::vector<int> chans((size_t)n_files, 0);
  int64_t max_len = 0;
  for (int i = 0; i < n_files; i++) {
    if (!paths_in[i] || !paths_out[i]) return fail(CRISPY_NS_EINVAL, "denoise_wav_files: null path");
    int sr = 0;
    const int rc = wav_read_pcm16(paths_in[i], nullptr, 0, &len[(size_t)i], &chans[(size_t)i], &sr);
    if (rc != CRISPY_NS_OK) return rc;
    if (sr != 48000) return fail(CRISPY_NS_EINVAL, std::string("denoise_wav_files: ") + paths_in[i] + " is not 48 kHz (recording.rs:14)");
    if (len[(size_t)i] > max_len) max_len = len[(size_t)i];
  }
  const int64_t n_frames = (max_len + ns::kFrame - 1) / ns::kFrame;
  if (n_frames >= (1ll << 31) / ns::kFrame) return fail(CRISPY_NS_EINVAL, "denoise_wav_files: recording too long for one call");
  const bool drop = (flags & CRISPY_NS_DROP_FIRST_FRAME) != 0;
  const int64_t row = n_frames * ns::kFrame;
  struct Pinned {  // pinned staging: mono PCM16 in, stereo PCM16 out, VAD
    void *p = nullptr;
    ~Pinned() {
      if (p) cudaFreeHost(p);
    }
  } hin, hout, hvad;
  crispy_ns_batch *b = nullptr;
  int rc = batch_create(model, device, n_files, &b);
  if (rc != CRISPY_NS_OK) return rc;
  struct BatchGuard {
    crispy_ns_batch *b;
    ~BatchGuard() { batch_destroy(b); }
  } bg{b};
  if (n_frames == 0 || (drop && n_frames < 2)) {  // nothing to denoise: empty outputs
    for (int i = 0; i < n_files; i++) {
      rc = wav_write_pcm16(paths_out[i], nullptr, 0, 2, 48000);
      if (rc != CRISPY_NS_OK) return rc;
      if (mean_vad) mean_vad[i] = 0.f;
    }
    return CRISPY_NS_OK;
  }
  NS_CUDA(cudaHostAlloc(&hin.p, (size_t)n_files * row * sizeof(int16_t), cudaHostAllocDefault));
  NS_CUDA(cudaHostAlloc(&hout.p, (size_t)n_files * row * 2 * sizeof(int16_t), cudaHostAllocDefault));
  NS_CUDA(cudaHostAlloc(&hvad.p, (size_t)n_files * n_frames * sizeof(float), cudaHostAllocDefault));
  int16_t *in16 = (int16_t *)hin.p, *out16 = (int16_t *)hout.p;
  float *vad = (float *)hvad.p;
  {
    std::vector<int16_t> tmp;
    for (int i = 0; i < n_files; i++) {
      const int ch = chans[(size_t)i];
      const int64_t n = len[(size_t)i];
      tmp.resize((size_t)(n * ch));
      int64_t nf = 0;
      rc = wav_read_pcm16(paths_in[i], tmp.data(), n * ch, &nf, nullptr, nullptr);
      if (rc != CRISPY_NS_OK) return rc;
      int16_t *dst = in16 + (size_t)i * row;
      for (int64_t k = 0; k < n; k++) dst[k] = tmp[(size_t)(k * ch)];  // channel 0 (commands/transcription.rs:310-312)
      memset(dst + n, 0, (size_t)(row - n) * sizeof(int16_t));
    }
  }
  rc = process_streams_host(b, in16, out16, vad, nullptr, (int)n_frames, row, row, n_frames, 0,
                                      CRISPY_NS_IN_I16 | CRISPY_NS_UNIT_SCALE | CRISPY_NS_MIX_STEREO_I16 | flags, volume);
  if (rc != CRISPY_NS_OK) return rc;
  for (int i = 0; i < n_files; i++) {
    int64_t n_out = len[(size_t)i] - (drop ? ns::kFrame : 0);
    if (n_out < 0) n_out = 0;
    rc = wav_write_pcm16(paths_out[i], out16 + (size_t)i * row * 2, n_out, 2, 48000);
    if (rc != CRISPY_NS_OK) return rc;
    if (mean_vad) {
      const int64_t fr = (len[(size_t)i] + ns::kFrame - 1) / ns::kFrame;
      double acc = 0.0;
      for (int64_t t = 0; t < fr; t++) acc += vad[(size_t)i * n_frames + t];
      mean_vad[i] = fr > 0 ? (float)(acc / (double)fr) : 0.f;
    }
  }
  return CRISPY_NS_OK;
}

// ---- measurement aid: FP32 burst -------------------------------------------------------------------------
}  // namespace impl
template <bool FUSED>
__global__ void __launch_bounds__(256) ns_fp32_burst_kernel(float *out, int iters, float y0) {
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; i++) a[i] = (float)(threadIdx.x + i);
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      if (FUSED)
        a[i] = fmaf(a[(i + 1) & 7], y0, a[i]);
      else
        a[i] = __fadd_rn(a[i], __fmul_rn(a[(i + 1) & 7], y0));
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) s += a[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
namespace impl {
int measure_fp32(int device, double *ffma_tflops, double *unfused_tmacs) {
  const int ndev = device_count();
  if (ndev == 0) return fail(CRISPY_NS_ENODEV, "no CUDA device: libcrispy_ns has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(CRISPY_NS_ENODEV, "device index out of range");
  NS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  NS_CUDA(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 20000;
  float *d = nullptr;
  NS_CUDA(cudaMalloc((void **)&d, (size_t)blocks * threads * sizeof(float)));
  cudaEvent_t a = nullptr, b = nullptr;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  double best[2] = {1e30, 1e30};
  cudaError_t e = cudaSuccess;
  for (int mode = 0; mode < 2 && e == cudaSuccess; mode++) {
    for (int rep = 0; rep < 4 && e == cudaSuccess; rep++) {
      cudaEventRecord(a, 0);
      if (mode == 0)
        ns_fp32_burst_kernel<true><<<blocks, threads>>>(d, rep == 0 ? 64 : iters, 1e-6f);
      else
        ns_fp32_burst_kernel<false><<<blocks, threads>>>(d, rep == 0 ? 64 : iters, 1e-6f);
      cudaEventRecord(b, 0);
      e = cudaEventSynchronize(b);
      float ms = 0.f;
      if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, a, b);
      if (rep > 0 && ms < best[mode]) best[mode] = ms;
    }
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(d);
  if (e != cudaSuccess) return fail(CRISPY_NS_ECUDA, std::string("measure_fp32: ") + cudaGetErrorString(e));
  const double macs = (double)blocks * threads * 8.0 * iters;
  if (ffma_tflops) *ffma_tflops = 2.0 * macs / (best[0] * 1e-3) / 1e12;
  if (unfused_tmacs) *unfused_tmacs = macs / (best[1] * 1e-3) / 1e12;
  return CRISPY_NS_OK;
}

}  // namespace impl

#include "crispy_ns_abi.inc"

#ifdef NS_PHASE_CLOCKS
extern "C" int crispy_ns_debug_pitch_phase_cycles(unsigned long long *out24, int reset) {
  if (out24 && cudaMemcpyFromSymbol(out24, ns::g_pitch_phase_cycles, 24 * sizeof(unsigned long long)) != cudaSuccess) return -1;
  if (reset) {
    unsigned long long z[24] = {0};
    if (cudaMemcpyToSymbol(ns::g_pitch_phase_cycles, z, sizeof(z)) != cudaSuccess) return -1;
  }
  return 0;
}
#endif
