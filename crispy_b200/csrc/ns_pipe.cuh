// ns_pipe.cuh -- device code of the phased RNNoise pipeline behind
// nnnoiseless::DenoiseState::process_frame (/root/reference/src-tauri/src/audio.rs:268).
//
// One chunk of frames of every stream goes through seven kernels (DESIGN.md has the data flow):
//   K0 highpass   serial-in-time biquad, one lane per stream (f32 state, f64 intermediates: a6)
//   K1 pitch      parallel over (stream, run of R frames): pitch_downsample, pitch_search and every
//                 inner product remove_doubling can ask for (a9-a11) -> candidate table
//   K2 pitchscan  serial-in-time threshold walk of remove_doubling (last_period / last_gain), one
//                 warp per stream, one lane per candidate
//   K3 spectrum   parallel over (stream, frame): windowed rFFT960 of the frame and of the
//                 pitch-lagged window, band energies / correlation, cepstrum (a7, a8, a12, a13)
//   K3b features  serial-in-time cepstral ring, delta features, spectral variability (a13), one warp per
//                 stream; emits the 42 features as bf16 hi + lo MMA fragments
//   K4 rnn        serial-in-time recurrent core on the tensor pipe (mma.sync bf16 hi + lo), 16 streams per
//                 CTA: dense -> 3 GRUs -> dense, gain smoothing (a14)
//   K5 synthesis  per (stream, run of frames): pitch filter, gain interpolation, inverse FFT, overlap-add
//                 (a15, a16); the next frame's spectra arrive by TMA bulk copies
//
// EXACTNESS CONTRACT.  Everything that feeds a discrete pitch decision (K0, K1, K2) is computed
// with the oracle's operation order and roundings: this translation unit is compiled with
// -fmad=false (nvcc) / -ffp-contract=off (host emulation), so a*b+c is a rounded product followed by
// a rounded sum unless fmaf() is spelled out; fmaf() appears only in K3-K5 (spectra, RNN), whose
// results are continuous in their inputs.  Pitch indices therefore match the oracle bit for bit.
//
// The same source compiles for sm_100a (nvcc) and for the host SIMT emulation (NS_HOST_EMU, tests).
#pragma once
#include <type_traits>

#include "ns_common.h"
#include "ns_simt.h"

namespace ns {

NS_DEV f4 ld4(const float *p) { return *reinterpret_cast<const f4 *>(p); }

// =================================================================================================
// K0: a6 biquad high-pass.  upstream denoise.c biquad(): y = x + mem0 (f32);
// mem0 = (f32)(mem1 + (b0 x - a0 y)), mem1 = (f32)(b1 x - a1 y) with f64 intermediates.  The f32
// rounding of the state makes the recursion non-linear (two trajectories a few ulps apart never
// merge: measured, scripts/micro), so it runs serially, one lane per stream, and nothing else may
// sit on that lane's critical path.
// =================================================================================================
// One CTA = 32 streams = three specialised warps that meet only through shared-memory flags (a
// bar.sync would make the recursion wait for the other warps' global memory traffic):
//   warp 1 (loader)   : cp.async (LDGSTS) tiles of 96 samples x 32 streams into a ring, two tiles ahead
//   warp 0 (recursion): one lane per stream runs the biquad over its row of the tile in place
//   warp 2 (storer)   : copies the stream history to the front of the hp rows, then writes every
//                       finished tile to the hp workspace (and the chunk's tail to the state's history)
// Flags hold "tile index + 1" per ring slot: landed (loader -> recursion), done (recursion ->
// storer), freed (storer -> loader).
constexpr int kHpThreads = 96;
// Tile length: 96 samples x 4 stages = 51 KB.  Smaller rings were measured (-DNS_HP_TILE=48: 27 KB, fits beside three
// pitch CTAs; 24: 14 KB) and bought nothing -- the pipeline ran 47.15 / 51.3 ms per 1,536 frames against 46.9 -- while
// the recursion warp pays ~500 cycles of hand-over per tile (isolated 617 -> 641 -> 790 us per chunk), so the long tile stays.
#ifndef NS_HP_TILE
#define NS_HP_TILE 96
#endif
constexpr int kHpTile = NS_HP_TILE;  // samples per tile; 480 = 5 tiles
constexpr int kHpPitch = kHpTile + 4;  // floats per row in shared memory: rows 4 (mod 32) banks apart for LDS.128
constexpr int kHpStages = 4;
constexpr int kHpAhead = 2;        // tiles the loader keeps in flight beyond the one it is publishing
// byte offset of a row's raw PCM16 samples: 16-byte aligned, 4c + 16 <= kHpRaw16 + 2(c + 4) for every c < kHpTile
constexpr int kHpRaw16 = (2 * kHpTile - 8 + 15) / 16 * 16;
static_assert(kFrame % kHpTile == 0 && kHpTile % 8 == 0 && kHpPitch % 32 != 0 && kHpPitch % 4 == 0, "tile geometry");
static_assert(kHpRaw16 % 16 == 0 && kHpRaw16 + 2 * kHpTile <= kHpPitch * 4 && 2 * kHpTile - 8 <= kHpRaw16, "PCM16 staging");
struct HpSmem {
  float tile[kHpStages][32][kHpPitch];
  int landed[kHpStages], done[kHpStages], freed[kHpStages];
};

NS_DEV float load_sample(const Params &p, int stream, long long idx) {
  const long long off = (long long)stream * p.in_stride + idx;
  if (p.flags & kFlagInI16) return (float)reinterpret_cast<const int16_t *>(p.in)[off];
  return reinterpret_cast<const float *>(p.in)[off];
}

// tile `n` of the chunk -> ring slot; fast path: 16-byte cp.async (lanes 0..23 cover one 384-byte row
// segment per instruction), else plain loads
NS_DEV void hp_fetch_tile(const Params &p, HpSmem &sm, int s0, int nrows, long long in0, int n, bool fast, int lane) {
  float(*dst)[kHpPitch] = sm.tile[n % kHpStages];
  const long long idx0 = in0 + (long long)n * kHpTile;
  if (fast && (p.flags & kFlagInI16)) {
    // PCM16 rows (192 B) land raw in the upper part of their float row (byte kHpRaw16 on); the recursion
    // converts four samples at a time and writes y over the row from the front, always behind its reads
    if (lane < kHpTile / 8) {
      const int16_t *src = reinterpret_cast<const int16_t *>(p.in) + (long long)s0 * p.in_stride + idx0 + 8 * lane;
      char *d = reinterpret_cast<char *>(&dst[0][0]) + kHpRaw16 + 16 * lane;
#pragma unroll 8
      for (int r = 0; r < nrows; r++, src += p.in_stride, d += kHpPitch * sizeof(float)) Simt::cp_async16(d, src);
    }
  } else if (fast) {
    if (lane < kHpTile / 4) {
      const float *src = reinterpret_cast<const float *>(p.in) + (long long)s0 * p.in_stride + idx0 + 4 * lane;
      float *d = &dst[0][4 * lane];
#pragma unroll 8
      for (int r = 0; r < nrows; r++, src += p.in_stride, d += kHpPitch) Simt::cp_async16(d, src);
    }
  } else {
    for (int q = lane; q < 32 * kHpTile; q += 32) {
      const int r = q / kHpTile, c = q - r * kHpTile;
      dst[r][c] = (r < nrows) ? load_sample(p, s0 + r, idx0 + c) : 0.f;
    }
  }
}

NS_DEV void hp_copy_rows(const float *src, long long src_stride, float *dst, long long dst_stride, int nrows, int lane) {
  for (int r = 0; r < nrows; r++) {  // kHist floats per row, batched so the loads overlap
    const f4 *__restrict__ s = reinterpret_cast<const f4 *>(src + (long long)r * src_stride);
    f4 *__restrict__ d = reinterpret_cast<f4 *>(dst + (long long)r * dst_stride);
    f4 v[6];
    for (int i0 = 0; i0 < kHist / 4; i0 += 6 * 32) {
#pragma unroll
      for (int u = 0; u < 6; u++)
        if (i0 + u * 32 + lane < kHist / 4) v[u] = s[i0 + u * 32 + lane];
#pragma unroll
      for (int u = 0; u < 6; u++)
        if (i0 + u * 32 + lane < kHist / 4) d[i0 + u * 32 + lane] = v[u];
    }
  }
}

// F32 (CRISPY_NS_BIQUAD_F32): the recursion in f32 arithmetic alone, every product and sum rounded to f32 --
//   mem0 = mem1 + (b0 x - a0 y), mem1 = b1 x - a1 y -- the form a port that widens nothing would compute.
template <bool F32 = false>
NS_DEV void highpass_body(const Params &p, HpSmem &sm) {
  const int tid = Simt::tid();
  const int lane = tid & 31, warp = tid >> 5;
  const int s0 = Simt::cta() * 32;
  const int nrows = (p.n_streams - s0) < 32 ? (p.n_streams - s0) : 32;
  const int nsamp = p.n_frames * kFrame;
  const int ntiles = nsamp / kHpTile;
  const bool tail_direct = nsamp >= kHist;  // the new history is the chunk's own tail
  if (tid < kHpStages) sm.landed[tid] = sm.done[tid] = sm.freed[tid] = 0;
  Simt::cta_sync();
  const long long in0 = (long long)p.frame0 * kFrame;
  const bool in16 = (p.flags & kFlagInI16) != 0;
  const int amask = in16 ? 7 : 3;  // samples per 16 bytes - 1
  const bool fast = (p.in_stride & amask) == 0 && (in0 & amask) == 0 && (reinterpret_cast<uintptr_t>(p.in) & 15) == 0;
  const bool raw16 = fast && in16;
  if (warp == 1) {  // ---- loader
    for (int n = 0; n < ntiles + kHpAhead; n++) {
      if (n < ntiles) {
        if (n >= kHpStages) Simt::flag_wait(&sm.freed[n % kHpStages], n - kHpStages + 1, true);
        hp_fetch_tile(p, sm, s0, nrows, in0, n, fast, lane);
      }
      Simt::cp_async_commit();
      if (n >= kHpAhead) {  // tile n - kHpAhead has landed in every lane's view: publish it
        Simt::cp_async_wait<kHpAhead>();
        if (raw16) {
          // PCM16 rows were staged raw in the upper part of their float row: this warp, which only issues copies
          // otherwise, turns them into floats in place (lane = row, four samples at a time, writing always behind its
          // reads) so that the conversion stays off the recursion warp's chain
          Simt::warp_sync();
          if (lane < nrows) {
            float *row = sm.tile[(n - kHpAhead) % kHpStages][lane];
#pragma unroll 4
            for (int c = 0; c < kHpTile; c += 4) {
              const uint32_t *rw = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(row) + kHpRaw16 + 2 * c);
              const uint32_t r0 = rw[0], r1 = rw[1];
              *reinterpret_cast<f4 *>(row + c) = f4{(float)(int16_t)(r0 & 0xFFFFu), (float)(int16_t)(r0 >> 16),
                                                    (float)(int16_t)(r1 & 0xFFFFu), (float)(int16_t)(r1 >> 16)};
            }
          }
        }
        Simt::fence_cta();
        Simt::warp_sync();
        if (lane == 0) Simt::flag_set(&sm.landed[(n - kHpAhead) % kHpStages], n - kHpAhead + 1);
      }
    }
  } else if (warp == 0) {  // ---- recursion
    const float scale = ((p.flags & kFlagUnitScale) && !(p.flags & kFlagInI16)) ? 32768.0f : 1.0f;  // audio.rs:264
    const bool valid = lane < nrows;
    float *st = p.state + (long long)(s0 + (valid ? lane : 0)) * kStateFloats;
    float m0 = valid ? st[kStHp] : 0.f, m1 = valid ? st[kStHp + 1] : 0.f;
    const double na0 = -(double)-1.99599f, na1 = -(double)0.99600f;
    for (int n = 0; n < ntiles; n++) {
      const int slot = n % kHpStages;
      Simt::flag_wait(&sm.landed[slot], n + 1, false);
      if (valid) {
        float *row = sm.tile[slot][lane];
#pragma unroll 2
        for (int c = 0; c < kHpTile; c += 4) {
          float x[4];
          {
            const f4 xv = ld4(row + c);  // PCM16 input arrives here as floats too (converted by the loader warp)
            x[0] = xv.x * scale, x[1] = xv.y * scale, x[2] = xv.z * scale, x[3] = xv.w * scale;
          }
          float y[4];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const float xi = x[i];
            const float yi = xi + m0;
            if constexpr (F32) {
              const float b0 = -2.f, b1 = 1.f, a0 = -1.99599f, a1 = .99600f;
              m0 = m1 + (b0 * xi - a0 * yi);
              m1 = b1 * xi - a1 * yi;
            } else {
              const double xd = (double)xi, yd = (double)yi;
              // a0*y and a1*y are exact in f64 (24 x 24 bit), so the fused forms round exactly like
              // upstream's  mem1 + (b0*x - a0*y)  and  b1*x - a1*y
              m0 = (float)((double)m1 + fma(na0, yd, -2.0 * xd));
              m1 = (float)fma(na1, yd, xd);
            }
            y[i] = yi;
          }
          *reinterpret_cast<f4 *>(row + c) = f4{y[0], y[1], y[2], y[3]};
        }
      }
      Simt::fence_cta();
      Simt::warp_sync();
      if (lane == 0) Simt::flag_set(&sm.done[slot], n + 1);
    }
    if (valid) {
      st[kStHp] = m0;
      st[kStHp + 1] = m1;
    }
  } else {  // ---- storer
    hp_copy_rows(p.state + (long long)s0 * kStateFloats + kStHist, kStateFloats, p.hp + (long long)s0 * p.hp_stride,
                 p.hp_stride, nrows, lane);
    Simt::warp_sync();  // the old history has been read: the tail tiles may overwrite it
    for (int n = 0; n < ntiles; n++) {
      const int slot = n % kHpStages;
      Simt::flag_wait(&sm.done[slot], n + 1, true);
      float(*tile)[kHpPitch] = sm.tile[slot];
      const int base = n * kHpTile;
      if (lane < kHpTile / 4) {
        const int c = 4 * lane;
        float *dsth = p.hp + (long long)s0 * p.hp_stride + kHist + base + c;
        const int hidx = base + c - (nsamp - kHist);
        if (tail_direct && hidx >= 0) {
          float *dsts = p.state + (long long)s0 * kStateFloats + kStHist + hidx;
          for (int r = 0; r < nrows; r++, dsth += p.hp_stride, dsts += kStateFloats) {
            const f4 v = ld4(&tile[r][c]);
            *reinterpret_cast<f4 *>(dsth) = v;
            *reinterpret_cast<f4 *>(dsts) = v;
          }
        } else {
#pragma unroll 8
          for (int r = 0; r < nrows; r++, dsth += p.hp_stride) *reinterpret_cast<f4 *>(dsth) = ld4(&tile[r][c]);
        }
      }
      Simt::warp_sync();
      if (lane == 0) Simt::flag_set(&sm.freed[slot], n + 1);
    }
    if (!tail_direct) {  // short chunk: last kHist samples of [history | chunk] -> state, staged through registers
      Simt::fence_cta();
      Simt::warp_sync();
      for (int r = 0; r < nrows; r++) {
        const float *src = p.hp + (long long)(s0 + r) * p.hp_stride + nsamp;
        float *dst = p.state + (long long)(s0 + r) * kStateFloats + kStHist;
        float v[kHist / 32];
#pragma unroll
        for (int i = 0; i < kHist / 32; i++) v[i] = src[lane + 32 * i];
#pragma unroll
        for (int i = 0; i < kHist / 32; i++) dst[lane + 32 * i] = v[i];
      }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// K0, second form (ns_highpass_par_kernel; what small batches run): THE SAME RECURSION, PARALLEL IN TIME.
//
// The single recursion warp above spends its 74 cycles per sample on the f64 side of its SM sub-partition: five F2F
// conversions (one warp issues one per ~13-19 cycles, scripts/micro/fp64_rate.cu) and four f64 operations, on a chain of
// FADD -> F2F -> DFMA -> DADD -> F2F (scripts/micro/hp_latency.cu; speculating mem0 in f32 on the same warp while it
// still verifies in f64 is therefore SLOWER: 81 cycles, variants 5 / 6).  Here the f64 work leaves the serial warp:
//   warp 0          : runs the recursion SPECULATIVELY in error-free f32 arithmetic, no f64 at all (43 cycles a
//                     sample: ~20 FADD / FMUL / FFMA / FSEL, whose dependent latency is ~5.8 cycles on this part), and
//                     only records its state at the start of every 24-sample segment (and at the tile's end);
//   warps 3, 5, 6, 7: segment v of every tile by upstream's own f64 expression (exact_run), STARTING FROM THE RECORDED
//                     STATE, four segments in parallel on the other sub-partitions; they write y, and compare the
//                     state they end in, bit for bit, with the state recorded for the next segment;
//   warp 1 / warp 2 : loader and storer as before (y now has a ring of its own: x must survive a repair).
// By induction over the segments, every y the storer sees comes out of upstream's expression from a start state that
// is upstream's: the result is upstream's bits BY CONSTRUCTION, whatever the speculation does.  Where a segment's
// end state differs from the record (any bit, the sign of a zero included), warp 0 takes the segment's exact end
// state, recomputes the rest of that tile exactly, and speculates the next tile again, before the next tile is
// released to the exact warps (`settle`).
// The f32 speculation: a0 y = ph + pl exactly (FMUL + FFMA), m1 - 2x = ch + cl exactly, ch + ph = s1 + e1 exactly
// (error terms by a two-sided FastTwoSum), and RN32(s1 + ((cl + pl) + e1)) is upstream's
// RN32(RN53(m1 + RN53(a0 y - 2x))) unless the sum sits within ~2^-22 ulp of a rounding boundary or the low product
// underflows; mem1 = RN32(x - a1 y) is a single f32 FMA.  On the host: no mismatch in 1e9 samples of speech-like, white, DC, tonal,
// PCM16 and tiny inputs; ~300 per decay into digital silence (the state crossing 2^-126); subnormal limit cycles that
// cross -0 miss once per ~800 samples; 0.08 % of the bench workload's tiles need a repair.
// Measured (B200, 1,024 streams x 32 frames, the kernel alone): 613 -> 424 us; per tile the speculation warp works
// 4,160 cycles, waits 130 for the loader and spends 610 in `settle` (-DNS_HP_CLOCKS).  In the pipeline it is worth
// +3 % at 768 streams, +18 % at 512, +37 % at 256, and nothing beside the pitch CTAs of a full batch, where K0 is not
// the longest stage and its eight warps take issue slots from them: crispy_ns.cu picks the form by batch size.
// Warp 4 would share warp 0's sub-partition and exits at once.
// -------------------------------------------------------------------------------------------------
#ifndef NS_HP_PAR
#define NS_HP_PAR 1
#endif
constexpr int kHpSeg = 4;                     // exact warps = segments per tile
constexpr int kHpSegLen = kHpTile / kHpSeg;   // 24 samples
constexpr int kHpYStages = 2;                 // y ring: one tile being written, one being stored
constexpr int kHpParThreads = 256;
// The loader publishes tile n once tile n + kHpParAhead has been issued, and a ring slot is held until its tile has
// been settled (one tile later than in the first form): with two tiles ahead the speculation warp waited ~1,000 cycles
// per tile for `landed` (measured with -DNS_HP_CLOCKS); with one, tile n is published two tiles before it is needed.
constexpr int kHpParAhead = 1;
static_assert(kHpTile % (4 * kHpSeg) == 0, "segments are whole 16-byte groups");
#ifdef NS_HOST_EMU
// test hook of the host emulation: tiles whose speculation had to be repaired (tests assert the path is taken)
inline long long g_hp_respeculated = 0;
#define NS_HP_COUNT_RESPEC() __atomic_add_fetch(&::ns::g_hp_respeculated, 1, __ATOMIC_RELAXED)
#else
#define NS_HP_COUNT_RESPEC() ((void)0)
#endif
#if defined(NS_HP_CLOCKS) && defined(__CUDACC__) && !defined(NS_HOST_EMU)
#define NS_HP_T0() const long long hp_t0_ = clock64()
#define NS_HP_ACC(var) var += clock64() - hp_t0_
#else
#define NS_HP_T0() ((void)0)
#define NS_HP_ACC(var) ((void)0)
#endif
struct HpParSmem {
  HpSmem x;                                  // the x ring and the loader's flags (done[] unused)
  float y[kHpYStages][32][kHpPitch];         // the y ring
  float spec[2][kHpSeg + 1][32][2];          // speculated (mem0, mem1) at the start of segment v / at the tile's end
  float exact[2][kHpSeg][32][2];             // upstream's (mem0, mem1) at the end of segment v
  alignas(16) int bad[2][32][kHpSeg];        // 1: segment v ended in a state that is not the recorded one
  int go;                                    // tiles < go are speculated and every earlier tile is settled
  int ver;                                   // kHpSeg x the number of tiles every exact warp is through
  int ydone;                                 // tiles < ydone are final in the y ring
  int yfreed;                                // tiles < yfreed have been stored
};

// a + b - RN32(a + b), exactly: FastTwoSum both ways round; the one whose first operand is the larger is exact
// (scripts/micro/hp_latency.cu variant 16: 45.8 cycles a sample; TwoSum 47.3, operands ordered first 50.3)
NS_DEV float hp_fast_err(float a, float b, float s) {
  const float ea = b - (s - a), eb = a - (s - b);
  return fabsf(a) >= fabsf(b) ? ea : eb;
}

NS_DEV void highpass_par_body(const Params &p, HpParSmem &sm) {
  const int tid = Simt::tid();
  const int lane = tid & 31, warp = tid >> 5;
  const int s0 = Simt::cta() * 32;
  const int nrows = (p.n_streams - s0) < 32 ? (p.n_streams - s0) : 32;
  const int nsamp = p.n_frames * kFrame;
  const int ntiles = nsamp / kHpTile;
  const bool tail_direct = nsamp >= kHist;  // the new history is the chunk's own tail
  if (tid < kHpStages) sm.x.landed[tid] = sm.x.done[tid] = sm.x.freed[tid] = 0;
  if (tid == 0) sm.ver = sm.go = sm.ydone = sm.yfreed = 0;
  Simt::cta_sync();
  const long long in0 = (long long)p.frame0 * kFrame;
  const bool in16 = (p.flags & kFlagInI16) != 0;
  const int amask = in16 ? 7 : 3;  // samples per 16 bytes - 1
  const bool fast = (p.in_stride & amask) == 0 && (in0 & amask) == 0 && (reinterpret_cast<uintptr_t>(p.in) & 15) == 0;
  const bool raw16 = fast && in16;
  const float scale = ((p.flags & kFlagUnitScale) && !in16) ? 32768.0f : 1.0f;  // audio.rs:264
  const bool valid = lane < nrows;
  float m0 = 0.f, m1 = 0.f;
  long long t_work = 0, t_wait = 0, t_wait2 = 0;  // -DNS_HP_CLOCKS: cycles per role (CTA 0 prints them)
  (void)t_work, (void)t_wait, (void)t_wait2;
  const long long t_begin = 0;
  (void)t_begin;
  const double na0 = -(double)-1.99599f, na1 = -(double)0.99600f;
  // n4 16-byte groups by upstream's own expression (f32 state, f64 intermediates): the definition of the result.
  // a0*y and a1*y are exact in f64 (24 x 24 bit), so the fused forms round exactly like upstream's
  // mem1 + (b0*x - a0*y)  and  b1*x - a1*y
  auto exact_run = [&](const float *xrow, float *yrow, int n4) {
#pragma unroll 2
    for (int c = 0; c < 4 * n4; c += 4) {
      const f4 xv = ld4(xrow + c);
      const float x[4] = {xv.x * scale, xv.y * scale, xv.z * scale, xv.w * scale};
      float y[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const float xi = x[i];
        const float yi = xi + m0;
        const double xd = (double)xi, yd = (double)yi;
        m0 = (float)((double)m1 + fma(na0, yd, -2.0 * xd));
        m1 = (float)fma(na1, yd, xd);
        y[i] = yi;
      }
      *reinterpret_cast<f4 *>(yrow + c) = f4{y[0], y[1], y[2], y[3]};
    }
  };
  if (warp == 1) {  // ---- loader (as in the first form)
    for (int n = 0; n < ntiles + kHpParAhead; n++) {
      if (n < ntiles) {
        if (n >= kHpStages) {
          NS_HP_T0();
          Simt::flag_wait(&sm.x.freed[n % kHpStages], n - kHpStages + 1, true);
          NS_HP_ACC(t_wait);
        }
        hp_fetch_tile(p, sm.x, s0, nrows, in0, n, fast, lane);
      }
      Simt::cp_async_commit();
      if (n >= kHpParAhead) {
        Simt::cp_async_wait<kHpParAhead>();
        if (raw16) {
          Simt::warp_sync();
          if (lane < nrows) {
            float *row = sm.x.tile[(n - kHpParAhead) % kHpStages][lane];
#pragma unroll 4
            for (int c = 0; c < kHpTile; c += 4) {
              const uint32_t *rw = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(row) + kHpRaw16 + 2 * c);
              const uint32_t r0 = rw[0], r1 = rw[1];
              *reinterpret_cast<f4 *>(row + c) = f4{(float)(int16_t)(r0 & 0xFFFFu), (float)(int16_t)(r0 >> 16),
                                                    (float)(int16_t)(r1 & 0xFFFFu), (float)(int16_t)(r1 >> 16)};
            }
          }
        }
        Simt::fence_cta();
        Simt::warp_sync();
        if (lane == 0) Simt::flag_set(&sm.x.landed[(n - kHpParAhead) % kHpStages], n - kHpParAhead + 1);
      }
    }
  } else if (warp == 0) {  // ---- speculation in f32, and the repair of what it misses
    float *st = p.state + (long long)(s0 + (valid ? lane : 0)) * kStateFloats;
    if (valid) m0 = st[kStHp], m1 = st[kStHp + 1];
    const float a0f = 1.99599f, na1f = -0.99600f;
    auto spec_tile = [&](int n) {
      const float *row = sm.x.tile[n % kHpStages][lane];
      float(*rec)[32][2] = sm.spec[n & 1];
      for (int v = 0; v < kHpSeg; v++) {
        rec[v][lane][0] = m0, rec[v][lane][1] = m1;
#pragma unroll 2
        for (int c = v * kHpSegLen; c < (v + 1) * kHpSegLen; c += 4) {
          const f4 xv = ld4(row + c);
          const float x[4] = {xv.x * scale, xv.y * scale, xv.z * scale, xv.w * scale};
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const float xi = x[i];
            const float yi = xi + m0;
            // mem0' = RN32(m1 - 2x + a0 y): a0 y = ph + pl, m1 - 2x = ch + cl, ch + ph = s1 + e1, all exactly
            const float ph = a0f * yi, pl = fmaf(a0f, yi, -ph);
            const float b = -2.0f * xi;
            const float ch = fmaf(-2.0f, xi, m1), cl = hp_fast_err(m1, b, ch);
            const float s1 = ch + ph;
            const float e1 = hp_fast_err(ch, ph, s1);
            m0 = s1 + ((cl + pl) + e1);
            // mem1' = RN32(x - a1 y) is ONE f32 FMA: exact product, one rounding (upstream rounds to 53 bits first,
            // which matters with probability ~2^-29 -- and then the exact warps notice)
            m1 = fmaf(na1f, yi, xi);
          }
        }
      }
      rec[kHpSeg][lane][0] = m0, rec[kHpSeg][lane][1] = m1;
    };
    // tile k has been through the exact warps: repair it if a segment ended off the record, then hand it on
    auto settle = [&](int k, bool next_speculated) {
      Simt::flag_poll(&sm.ver, kHpSeg * (k + 1), false);  // the exact warps are at most one tile apart: a sum will do
      Simt::fence_cta();
      if (valid) {
        static_assert(kHpSeg == 4, "one 16-byte load fetches a lane's four flags");
        struct alignas(16) I4 {
          int x, y, z, w;
        };
        const I4 bd = *reinterpret_cast<const I4 *>(sm.bad[k & 1][lane]);
        const int v0 = bd.x ? 0 : bd.y ? 1 : bd.z ? 2 : bd.w ? 3 : -1;
        if (v0 >= 0) {
          NS_HP_COUNT_RESPEC();
          m0 = sm.exact[k & 1][v0][lane][0], m1 = sm.exact[k & 1][v0][lane][1];  // upstream's state after segment v0
          const int c0 = (v0 + 1) * kHpSegLen;
          exact_run(sm.x.tile[k % kHpStages][lane] + c0, sm.y[k % kHpYStages][lane] + c0, (kHpTile - c0) / 4);
          if (next_speculated) spec_tile(k + 1);
        }
      }
      Simt::fence_cta();  // one fence for the repaired y, the records of the next tile and the three flags
      Simt::warp_sync();
      if (lane == 0) {
        Simt::flag_store(&sm.ydone, k + 1);
        Simt::flag_store(&sm.x.freed[k % kHpStages], k + 1);
        if (next_speculated) Simt::flag_store(&sm.go, k + 2);
      }
    };
    for (int n = 0; n < ntiles; n++) {
      {
        NS_HP_T0();
        Simt::flag_wait(&sm.x.landed[n % kHpStages], n + 1, false);
        NS_HP_ACC(t_wait);
      }
      {
        NS_HP_T0();
        if (valid) spec_tile(n);
        NS_HP_ACC(t_work);
      }
      if (n >= 1) {
        NS_HP_T0();
        settle(n - 1, true);  // raises go = n + 1 as well
        NS_HP_ACC(t_wait2);
      } else {
        Simt::fence_cta();
        Simt::warp_sync();
        if (lane == 0) Simt::flag_store(&sm.go, 1);
      }
    }
    if (ntiles > 0) settle(ntiles - 1, false);
    if (valid) {
      st[kStHp] = m0;
      st[kStHp + 1] = m1;
    }
  } else if (warp == 2) {  // ---- storer (as in the first form, from the y ring)
    hp_copy_rows(p.state + (long long)s0 * kStateFloats + kStHist, kStateFloats, p.hp + (long long)s0 * p.hp_stride,
                 p.hp_stride, nrows, lane);
    Simt::warp_sync();  // the old history has been read: the tail tiles may overwrite it
    for (int n = 0; n < ntiles; n++) {
      {
        NS_HP_T0();
        Simt::flag_wait(&sm.ydone, n + 1, true);
        NS_HP_ACC(t_wait);
      }
      NS_HP_T0();
      float(*tile)[kHpPitch] = sm.y[n % kHpYStages];
      const int base = n * kHpTile;
      if (lane < kHpTile / 4) {
        const int c = 4 * lane;
        float *dsth = p.hp + (long long)s0 * p.hp_stride + kHist + base + c;
        const int hidx = base + c - (nsamp - kHist);
        if (tail_direct && hidx >= 0) {
          float *dsts = p.state + (long long)s0 * kStateFloats + kStHist + hidx;
          for (int r = 0; r < nrows; r++, dsth += p.hp_stride, dsts += kStateFloats) {
            const f4 v = ld4(&tile[r][c]);
            *reinterpret_cast<f4 *>(dsth) = v;
            *reinterpret_cast<f4 *>(dsts) = v;
          }
        } else {
#pragma unroll 8
          for (int r = 0; r < nrows; r++, dsth += p.hp_stride) *reinterpret_cast<f4 *>(dsth) = ld4(&tile[r][c]);
        }
      }
      Simt::warp_sync();
      NS_HP_ACC(t_work);
      if (lane == 0) Simt::flag_set(&sm.yfreed, n + 1);
    }
    if (!tail_direct) {  // short chunk: last kHist samples of [history | chunk] -> state, staged through registers
      Simt::fence_cta();
      Simt::warp_sync();
      for (int r = 0; r < nrows; r++) {
        const float *src = p.hp + (long long)(s0 + r) * p.hp_stride + nsamp;
        float *dst = p.state + (long long)(s0 + r) * kStateFloats + kStHist;
        float v[kHist / 32];
#pragma unroll
        for (int i = 0; i < kHist / 32; i++) v[i] = src[lane + 32 * i];
#pragma unroll
        for (int i = 0; i < kHist / 32; i++) dst[lane + 32 * i] = v[i];
      }
    }
  } else if (warp != 4) {  // ---- segment v of every tile by upstream's expression, from the recorded state
    const int v = warp == 3 ? 0 : warp - 4;  // warps 3, 5, 6, 7
    for (int n = 0; n < ntiles; n++) {
      {
        NS_HP_T0();
        Simt::flag_wait(&sm.go, n + 1, true);
        NS_HP_ACC(t_wait);
      }
      if (n >= kHpYStages) {
        NS_HP_T0();
        Simt::flag_wait(&sm.yfreed, n - kHpYStages + 1, true);
        NS_HP_ACC(t_wait2);
      }
      NS_HP_T0();
      if (valid) {
        m0 = sm.spec[n & 1][v][lane][0], m1 = sm.spec[n & 1][v][lane][1];
        exact_run(sm.x.tile[n % kHpStages][lane] + v * kHpSegLen, sm.y[n % kHpYStages][lane] + v * kHpSegLen, kHpSegLen / 4);
        sm.exact[n & 1][v][lane][0] = m0, sm.exact[n & 1][v][lane][1] = m1;
        sm.bad[n & 1][lane][v] =
            (f2u(m0) != f2u(sm.spec[n & 1][v + 1][lane][0])) | (f2u(m1) != f2u(sm.spec[n & 1][v + 1][lane][1]));
      }
      Simt::fence_cta();
      Simt::warp_sync();
      NS_HP_ACC(t_work);
      if (lane == 0) Simt::atomic_add_shared(&sm.ver, 1);
    }
  }
#if defined(NS_HP_CLOCKS) && defined(__CUDACC__) && !defined(NS_HOST_EMU)
  if (Simt::cta() == 0 && lane == 0 && warp != 4)
    printf("K0 warp %d: %d tiles, work %lld, wait %lld, wait2 %lld cycles\n", warp, ntiles, t_work, t_wait, t_wait2);
#endif
}

// =================================================================================================
// K1: pitch analysis of R consecutive frames of one stream.  Every sum below is accumulated in the
// oracle's order (ascending index, rounded product then rounded add), one lane per sum; under sum policies
// 1 and 2 the inner products the oracle sums as dot4 are split into four partial sums (Acc4).
// =================================================================================================
template <int R>
struct PitchSmem {
  static constexpr int kHLen = R * kFrame + 1248;
  static constexpr int kXlpFloats = (R * kLpStride > kHLen) ? R * kLpStride : kHLen;
  alignas(16) float xr[R * kLpStride];  // raw downsampled rows; after the FIR each row holds y4[432] | yy_lookup[388]
  alignas(16) float xlp[kXlpFloats];    // first the high-passed window, then the whitened rows x_lp
  alignas(16) float ac[R][8];
  alignas(16) float lpc2[R][8];
  alignas(16) float fx[R][12];
  alignas(16) int fi[R][12];
  alignas(16) float xx[R];
  alignas(16) float s10[R][12];   // fine pass: Syy before each of the (at most ten) candidate lags (chain warp B, in P7's shadow)
#ifdef NS_PITCH_PAD_BYTES
  char pad[NS_PITCH_PAD_BYTES];  // measurement builds: forces fewer resident CTAs per SM
#endif
  int best0[R], best1[R], T0[R], nk[R];
  int n_tri[4], n_sgl[4];                   // [0] used: one list each (the alignment buckets are gone)
  // The coarse search's arrays (P5, P6) and remove_doubling's (P10 .. P12) are never live together: one region
  union {
    struct {
      alignas(16) float xc[R][152];
      alignas(16) float sb6[R][148];  // Syy before every coarse lag (helper warp, in the coarse search's shadow)
    };
    struct {
      // work lists of remove_doubling's inner products: frame | lag << 5 | k << 14
      uint32_t tri[4][R * 16], sgl[4][R * 16];  // <= 15 triples and <= 14 singles per frame, stored flat from tri[0] / sgl[0]
      alignas(16) float dots[R][64];   // 0: T0-1, 1: T0+1; for k >= 2 at 2+4(k-2): T1-1, T1, T1+1, T1b
    };
  };
};

struct Best2 {
  float n0, d0, n1, d1;
  int p0, p1;
};
NS_DEV void best_init(Best2 &b) {
  b.n0 = b.n1 = -1.f;
  b.d0 = b.d1 = 0.f;
  b.p0 = 0;
  b.p1 = 1;
}
NS_DEV void best_insert(Best2 &b, float num, float syy, int i) {  // pitch.c find_best_pitch
  if (num * b.d1 > b.n1 * syy) {
    if (num * b.d0 > b.n0 * syy) {
      b.n1 = b.n0;
      b.d1 = b.d0;
      b.p1 = b.p0;
      b.n0 = num;
      b.d0 = syy;
      b.p0 = i;
    } else {
      b.n1 = num;
      b.d1 = syy;
      b.p1 = i;
    }
  }
}

// the same update without branches (the serial search lanes run it on every lag): `valid` gates it
NS_DEV void best_insert_sel(Best2 &b, bool valid, float num, float syy, int i) {
  const bool c1 = valid && (num * b.d1 > b.n1 * syy);
  const bool c0 = c1 && (num * b.d0 > b.n0 * syy);
  b.n1 = c0 ? b.n0 : (c1 ? num : b.n1);
  b.d1 = c0 ? b.d0 : (c1 ? syy : b.d1);
  b.p1 = c0 ? b.p0 : (c1 ? i : b.p1);
  b.n0 = c0 ? num : b.n0;
  b.d0 = c0 ? syy : b.d0;
  b.p0 = c0 ? i : b.p0;
}

constexpr int kDotXy0 = 62;  // slot of xy(T0) in PitchSmem::dots (candidates use 0..57)
NS_DEV int rd_T1(int k, int T0) { return (2 * T0 + k) / (2 * k); }
NS_DEV int rd_T1b(int k, int T0, int T1) {
  if (k == 2) return (T1 + T0 > 384) ? T0 : T0 + T1;
  const int sc = (k == 6 || k == 12) ? 5 : ((k & 1) ? 2 : 3);  // second_check[k]
  return (2 * sc * T0 + k) / (2 * k);
}
NS_DEV float pitch_gain_f(float xy, float xx, float yy) { return xy / sqrtf(1.f + xx * yy); }

// sum_{j<N} x[j] * y[j] with y = yrow + yoff, accumulated in ascending j as a rounded product followed
// by a rounded add (the oracle's order).  x and yrow are 16-byte aligned, y has arbitrary alignment:
// the lane walks aligned float4s and shifts a two-vector window in registers, so one LDS.128 feeds
// four taps and the only serial dependency is the chain of adds (a scalar loop pays the ~29-cycle
// shared-memory latency on every tap and ~3.5 bank-conflict wavefronts between lanes with different
// lags).  Reads up to 3 floats before y[0] and 11 past y[N-1]: row padding / neighbouring rows.
#ifndef NS_DOT_UNROLL
#define NS_DOT_UNROLL 4
#endif
#define NS_PRAGMA(x) _Pragma(#x)
#define NS_UNROLL(n) NS_PRAGMA(unroll n)
// The chain of adds of one inner product, fed tap j as add(j & 3, x[j] y[j]) with j ascending from 0.  D4 = false:
// one accumulator in ascending j (xiph's celt_inner_prod / xcorr_kernel, sum policy 0).  D4 = true: four partial sums
// s[j & 3] reduced as ((s0 + s1) + s2) + s3 -- the oracle's dot4 (rnnoise_oracle.c, sum policies 1 and 2).  Every
// length summed here is a multiple of 4, so dot4's sequential tail never runs.
template <bool D4>
struct Acc4 {
  float s = 0.f;
  NS_DEV void add(int, float v) { s += v; }
  NS_DEV float sum() const { return s; }
};
template <>
struct Acc4<true> {
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  NS_DEV void add(int t, float v) { s[t] += v; }
  NS_DEV float sum() const { return ((s[0] + s[1]) + s[2]) + s[3]; }
};
// K1's summation policy (CRISPY_NS_SUM_*): which of its inner products are summed as dot4
template <int SP>
constexpr bool kSpDot4 = SP >= 1;  // celt_inner_prod / dual_inner_prod
template <int SP>
constexpr bool kSpDot4Xcorr = SP >= 2;  // celt_pitch_xcorr (coarse search, autocorrelation)

template <int N, bool D4 = false>
NS_DEV float dot_shifted(const float *x, const float *yrow, int yoff) {
  static_assert(N % 4 == 0, "whole float4s");
  const float *ya = yrow + (yoff & ~3);
  const bool p1 = (yoff & 1) != 0, p2 = (yoff & 2) != 0;
  f4 lo = ld4(ya), hi = ld4(ya + 4), xv = ld4(x);
  Acc4<D4> sum;
  NS_UNROLL(NS_DOT_UNROLL)
  for (int j = 0; j < N; j += 4) {
    // the next trip's operands are requested before this trip's chain of adds (the over-read of the
    // last trip stays inside the shared-memory rows)
    const f4 hi_n = ld4(ya + j + 8), xv_n = ld4(x + j + 4);
    const float a0 = p1 ? lo.y : lo.x, a1 = p1 ? lo.z : lo.y, a2 = p1 ? lo.w : lo.z, a3 = p1 ? hi.x : lo.w,
                a4 = p1 ? hi.y : hi.x, a5 = p1 ? hi.z : hi.y;
    const float y0 = p2 ? a2 : a0, y1 = p2 ? a3 : a1, y2 = p2 ? a4 : a2, y3 = p2 ? a5 : a3;
    sum.add(0, xv.x * y0);
    sum.add(1, xv.y * y1);
    sum.add(2, xv.z * y2);
    sum.add(3, xv.w * y3);
    lo = hi;
    hi = hi_n;
    xv = xv_n;
  }
  return sum.sum();
}
// the same with the shift S = (y - ya) known at compile time: no selects (used where a whole warp shares it)
template <int N, int S, bool D4 = false>
NS_DEV float dot_fixed_shift(const float *x, const float *ya) {
  f4 lo = ld4(ya), hi = ld4(ya + 4), xv = ld4(x);
  Acc4<D4> sum;
  NS_UNROLL(NS_DOT_UNROLL)
  for (int j = 0; j < N; j += 4) {
    const f4 hi_n = ld4(ya + j + 8), xv_n = ld4(x + j + 4);
    const float w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    sum.add(0, xv.x * w[S]);
    sum.add(1, xv.y * w[S + 1]);
    sum.add(2, xv.z * w[S + 2]);
    sum.add(3, xv.w * w[S + 3]);
    lo = hi;
    hi = hi_n;
    xv = xv_n;
  }
  return sum.sum();
}
// three inner products at once for the consecutive lags whose windows start at ya + S, ya + S + 1 and
// ya + S + 2: one pass over x and one stream of y feed three independent chains of adds
template <int N, int S>
NS_DEV void dot3_fixed_shift(const float *x, const float *ya, float &s0, float &s1, float &s2) {
  f4 w0 = ld4(ya), w1 = ld4(ya + 4), w2 = ld4(ya + 8), xv = ld4(x);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  NS_UNROLL(NS_DOT_UNROLL)
  for (int j = 0; j < N; j += 4) {
    const f4 w2_n = ld4(ya + j + 12), xv_n = ld4(x + j + 4);
    const float w[12] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w};
    a0 += xv.x * w[S];
    a1 += xv.x * w[S + 1];
    a2 += xv.x * w[S + 2];
    a0 += xv.y * w[S + 1];
    a1 += xv.y * w[S + 2];
    a2 += xv.y * w[S + 3];
    a0 += xv.z * w[S + 2];
    a1 += xv.z * w[S + 3];
    a2 += xv.z * w[S + 4];
    a0 += xv.w * w[S + 3];
    a1 += xv.w * w[S + 4];
    a2 += xv.w * w[S + 5];
    w0 = w1;
    w1 = w2;
    w2 = w2_n;
    xv = xv_n;
  }
  s0 = a0;
  s1 = a1;
  s2 = a2;
}
// the same three inner products with the shift S = yoff & 3 known only at run time: the six window elements a quad of
// taps needs come out of a two-level select network (shift by one, then by two) over the twelve loaded floats.
// Fourteen selects per four taps buy full lanes: with compile-time shifts a warp only holds the items of one
// alignment bucket (a quarter of a CTA's ~56 triples per warp-pass, seven active lanes on average).
template <int N, bool D4 = false>
NS_DEV void dot3_shifted(const float *x, const float *yrow, int yoff, float &s0, float &s1, float &s2) {
  const float *ya = yrow + (yoff & ~3);
  const bool p1 = (yoff & 1) != 0, p2 = (yoff & 2) != 0;
  f4 w0 = ld4(ya), w1 = ld4(ya + 4), w2 = ld4(ya + 8), xv = ld4(x);
  Acc4<D4> a2, a1, a0;  // this order keeps the sequential instantiation's SASS what it was before Acc4
  NS_UNROLL(NS_DOT_UNROLL)
  for (int j = 0; j < N; j += 4) {
    const f4 w2_n = ld4(ya + j + 12), xv_n = ld4(x + j + 4);
    // b[i] = w[i + (S & 1)], i < 8;  y[i] = b[i + (S & 2)], i < 6
    const float b0 = p1 ? w0.y : w0.x, b1 = p1 ? w0.z : w0.y, b2 = p1 ? w0.w : w0.z, b3 = p1 ? w1.x : w0.w,
                b4 = p1 ? w1.y : w1.x, b5 = p1 ? w1.z : w1.y, b6 = p1 ? w1.w : w1.z, b7 = p1 ? w2.x : w1.w;
    const float y0 = p2 ? b2 : b0, y1 = p2 ? b3 : b1, y2 = p2 ? b4 : b2, y3 = p2 ? b5 : b3, y4 = p2 ? b6 : b4,
                y5 = p2 ? b7 : b5;
    a0.add(0, xv.x * y0);
    a1.add(0, xv.x * y1);
    a2.add(0, xv.x * y2);
    a0.add(1, xv.y * y1);
    a1.add(1, xv.y * y2);
    a2.add(1, xv.y * y3);
    a0.add(2, xv.z * y2);
    a1.add(2, xv.z * y3);
    a2.add(2, xv.z * y4);
    a0.add(3, xv.w * y3);
    a1.add(3, xv.w * y4);
    a2.add(3, xv.w * y5);
    w0 = w1;
    w1 = w2;
    w2 = w2_n;
    xv = xv_n;
  }
  s0 = a0.sum();
  s1 = a1.sum();
  s2 = a2.sum();
}
template <bool D4 = false>
NS_DEV float dot480_shifted(const float *row, int yoff) { return dot_shifted<480, D4>(row + 384, row, yoff); }

// find_best_pitch's running energy: out[i] = Syy before lag i, Syy <- max(1, Syy + y[i+len]^2 - y[i]^2), for
// i < n (rounded up to 4).  y, out 16-byte aligned; out may alias y[0..n) (each y[i] is read before out[i]
// is written and never again).  Four lags per trip: loads and products are off the chain of adds.
NS_DEV void syy_recurrence(float syy, const float *y, int len, int n, float *out) {
  for (int i0 = 0; i0 < n; i0 += 4) {
    const f4 ya = ld4(y + i0 + len), yb = ld4(y + i0);
    const float d0 = ya.x * ya.x - yb.x * yb.x, d1 = ya.y * ya.y - yb.y * yb.y, d2 = ya.z * ya.z - yb.z * yb.z,
                d3 = ya.w * ya.w - yb.w * yb.w;
    f4 o;
    o.x = syy;
    syy += d0;
    syy = syy < 1.f ? 1.f : syy;
    o.y = syy;
    syy += d1;
    syy = syy < 1.f ? 1.f : syy;
    o.z = syy;
    syy += d2;
    syy = syy < 1.f ? 1.f : syy;
    o.w = syy;
    syy += d3;
    syy = syy < 1.f ? 1.f : syy;
    *reinterpret_cast<f4 *>(out + i0) = o;
  }
}

// acc + sum_{j<N} y[j]^2 in ascending j (y 16-byte aligned), loads batched four taps at a time
template <int N>
NS_DEV float sumsq_from(float acc, const float *y) {
  static_assert(N % 4 == 0, "whole float4s");
#pragma unroll 4
  for (int j = 0; j < N; j += 4) {
    const f4 v = ld4(y + j);
    acc += v.x * v.x;
    acc += v.y * v.y;
    acc += v.z * v.z;
    acc += v.w * v.w;
  }
  return acc;
}

#if defined(NS_PHASE_CLOCKS) && defined(__CUDACC__) && !defined(NS_HOST_EMU)
// measurement build only: cycles between K1's barriers, summed over CTAs (thread 0 of each CTA)
__device__ unsigned long long g_pitch_phase_cycles[24];
#define NS_PHASE_BEGIN() long long ns_pc_ = clock64()
#define NS_PHASE_MARK(i)                                                       \
  do {                                                                         \
    if (tid == 0) {                                                            \
      const long long now_ = clock64();                                        \
      atomicAdd(&g_pitch_phase_cycles[i], (unsigned long long)(now_ - ns_pc_)); \
      ns_pc_ = now_;                                                           \
    }                                                                          \
  } while (0)
#else
#define NS_PHASE_BEGIN() do {} while (0)
#define NS_PHASE_MARK(i) do {} while (0)
#endif
// SP: the summation policy (CRISPY_NS_SUM_*, kSpDot4 / kSpDot4Xcorr above); 0 is xiph's sequential order
template <int R, int NT, int SP = 0>
NS_DEV void pitch_body(const Params &p, PitchSmem<R> &sm) {
  const int tid = Simt::tid();
  NS_PHASE_BEGIN();
  const int runs_per_stream = (p.n_frames + R - 1) / R;
  const int stream = Simt::cta() / runs_per_stream;
  const int t0 = (Simt::cta() % runs_per_stream) * R;
  const int nfr = (p.n_frames - t0) < R ? (p.n_frames - t0) : R;
  const float *row = p.hp + (long long)stream * p.hp_stride + 192 + (long long)t0 * kFrame;
  float *h = sm.xlp;

  // P0: the window of high-passed samples these frames' pitch buffers cover
  if (tid < 4) sm.n_tri[tid] = sm.n_sgl[tid] = 0;
  {
    const int n4 = (nfr * kFrame + 1248) / 4;
    const f4 *src = reinterpret_cast<const f4 *>(row);
    f4 *dst = reinterpret_cast<f4 *>(h);
    for (int i = tid; i < n4; i += NT) dst[i] = src[i];
  }
  Simt::cta_sync();
  NS_PHASE_MARK(1);
  // P1: a9 2x downsample, pitch_buf[j] of frame f = h[480 f + j]
  for (int it = tid; it < nfr * (kLpLen / 4); it += NT) {  // four outputs per lane from two float4s (+ one scalar)
    const int f = it / (kLpLen / 4), i0 = 4 * (it - f * (kLpLen / 4));
    const float *x = h + f * kFrame + 2 * i0;
    const f4 b4 = ld4(x), c4 = ld4(x + 4);
    f4 v;
    if (i0 == 0)
      v.x = .5f * (.5f * b4.y + b4.x);
    else
      v.x = .5f * (.5f * (x[-1] + b4.y) + b4.x);
    v.y = .5f * (.5f * (b4.y + b4.w) + b4.z);
    v.z = .5f * (.5f * (b4.w + c4.y) + c4.x);
    v.w = .5f * (.5f * (c4.y + c4.w) + c4.z);
    *reinterpret_cast<f4 *>(sm.xr + f * kLpStride + i0) = v;
  }
  Simt::cta_sync();
  NS_PHASE_MARK(2);
  // P2: _celt_autocorr, lags 0..4.  One lane per (frame, lag) chain, twenty chains per warp (four frames x five
  // lags: their rows sit 8 banks apart and the lags 1 bank apart, so the scalar reads of x[i + k] do not
  // conflict and x[i] arrives as one broadcast LDS.128 per frame); operands are fetched one quad ahead of the
  // chain of adds.
  if (R <= 8 && NT >= 64) {
    if (tid < 64) {
      const int l = tid & 31, fl = l / 5, k = l - 5 * fl, f = 4 * (tid >> 5) + fl;
      if (l < 20 && f < nfr) {
        const float *x = sm.xr + f * kLpStride;
        const float *y = x + k;
        f4 xv = ld4(x);
        float y0 = y[0], y1 = y[1], y2 = y[2], y3 = y[3];
        Acc4<kSpDot4Xcorr<SP>> sum;
        NS_UNROLL(NS_DOT_UNROLL)
        for (int i = 0; i < kLpLen - 4; i += 4) {  // the last trip's over-read stays inside the padded row
          const f4 xn = ld4(x + i + 4);
          const float n0 = y[i + 4], n1 = y[i + 5], n2 = y[i + 6], n3 = y[i + 7];
          sum.add(0, xv.x * y0);
          sum.add(1, xv.y * y1);
          sum.add(2, xv.z * y2);
          sum.add(3, xv.w * y3);
          xv = xn;
          y0 = n0, y1 = n1, y2 = n2, y3 = n3;
        }
        float d = 0.f;
        for (int i = k + kLpLen - 4; i < kLpLen; i++) d += x[i] * x[i - k];
        sm.ac[f][k] = sum.sum() + d;
      }
    }
  } else if (NT >= 5 * 32 && R <= 32) {
    const int k = tid >> 5, f = tid & 31;
    if (k < 5 && f < nfr) {
      const float *x = sm.xr + f * kLpStride;
      float sum;
      switch (k) {
        case 0: sum = dot_fixed_shift<kLpLen - 4, 0, kSpDot4Xcorr<SP>>(x, x); break;
        case 1: sum = dot_fixed_shift<kLpLen - 4, 1, kSpDot4Xcorr<SP>>(x, x); break;
        case 2: sum = dot_fixed_shift<kLpLen - 4, 2, kSpDot4Xcorr<SP>>(x, x); break;
        case 3: sum = dot_fixed_shift<kLpLen - 4, 3, kSpDot4Xcorr<SP>>(x, x); break;
        default: sum = dot_fixed_shift<kLpLen - 4, 0, kSpDot4Xcorr<SP>>(x, x + 4); break;
      }
      float d = 0.f;
      for (int i = k + kLpLen - 4; i < kLpLen; i++) d += x[i] * x[i - k];
      sm.ac[f][k] = sum + d;
    }
  } else {
    for (int it = tid; it < nfr * 5; it += NT) {
      const int f = it / 5, k = it - f * 5;
      const float *x = sm.xr + f * kLpStride;
      const float sum = dot_shifted<kLpLen - 4, kSpDot4Xcorr<SP>>(x, x, k);
      float d = 0.f;
      for (int i = k + kLpLen - 4; i < kLpLen; i++) d += x[i] * x[i - k];
      sm.ac[f][k] = sum + d;
    }
  }
  Simt::cta_sync();
  NS_PHASE_MARK(3);
  // P3: lag window, _celt_lpc (order 4), bandwidth expansion, the extra zero
  if (tid < nfr) {
    const int f = tid;
    float ac[5], lpc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 5; k++) ac[k] = sm.ac[f][k];
    ac[0] *= 1.0001f;
#pragma unroll
    for (int i = 1; i <= 4; i++) ac[i] -= ac[i] * (.008f * i) * (.008f * i);
    float error = ac[0];
    if (ac[0] != 0.f) {
      for (int i = 0; i < 4; i++) {
        float rr = 0.f;
        for (int j = 0; j < i; j++) rr += lpc[j] * ac[i - j];
        rr += ac[i + 1];
        const float r = -rr / error;
        lpc[i] = r;
        for (int j = 0; j < ((i + 1) >> 1); j++) {
          const float t1 = lpc[j], t2 = lpc[i - 1 - j];
          lpc[j] = t1 + r * t2;
          lpc[i - 1 - j] = t2 + r * t1;
        }
        error = error - r * r * error;
        if (error < .001f * ac[0]) break;
      }
    }
    float tmp = 1.f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      tmp = .9f * tmp;
      lpc[i] = lpc[i] * tmp;
    }
    sm.lpc2[f][0] = lpc[0] + .8f;
    sm.lpc2[f][1] = lpc[1] + .8f * lpc[0];
    sm.lpc2[f][2] = lpc[2] + .8f * lpc[1];
    sm.lpc2[f][3] = lpc[3] + .8f * lpc[2];
    sm.lpc2[f][4] = .8f * lpc[3];
  }
  Simt::cta_sync();
  NS_PHASE_MARK(4);
  // P4: celt_fir5 with zero initial memory -> x_lp (overwrites the window h, which is dead now)
  for (int it = tid; it < nfr * (kLpLen / 4); it += NT) {  // four outputs per lane from three float4s
    const int f = it / (kLpLen / 4), i0 = 4 * (it - f * (kLpLen / 4));
    const float *x = sm.xr + f * kLpStride + i0;
    const float *n = sm.lpc2[f];
    const f4 z4 = f4{0.f, 0.f, 0.f, 0.f};
    const f4 p4 = (i0 >= 8) ? ld4(x - 8) : z4, q4 = (i0 >= 4) ? ld4(x - 4) : z4, r4 = ld4(x);
    const float w[9] = {p4.w, q4.x, q4.y, q4.z, q4.w, r4.x, r4.y, r4.z, r4.w};  // x[i0-5 .. i0+3]
    const float n0 = n[0], n1 = n[1], n2 = n[2], n3 = n[3], n4 = n[4];
    float o[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      float sum = w[5 + u];
      sum += n0 * w[4 + u];
      sum += n1 * w[3 + u];
      sum += n2 * w[2 + u];
      sum += n3 * w[1 + u];
      sum += n4 * w[u];
      o[u] = sum;
    }
    *reinterpret_cast<f4 *>(sm.xlp + f * kLpStride + i0) = f4{o[0], o[1], o[2], o[3]};
  }
  Simt::cta_sync();
  NS_PHASE_MARK(5);
  // P4b: 4x-decimated copy y4[m] = x_lp[2m] (x4[j] = y4[192 + j]); zero pad to 432+8
  for (int it = tid; it < nfr * 440; it += NT) {
    const int f = it / 440, m = it - f * 440;
    sm.xr[f * kLpStride + m] = (m < 432) ? sm.xlp[f * kLpStride + 2 * m] : 0.f;
  }
  Simt::cta_sync();
  NS_PHASE_MARK(6);
  // ---- the two long serial chains that only need x_lp run on their own warps in the shadow of P5..P7, a
  // budgeted number of 16-element blocks per phase (state stays in registers across the barriers):
  //   B (warp NW-2, lane = frame): find_best_pitch's running energy of the fine pass, Syy = 1 + sum_{j<480} y[j]^2
  //     (P5/P6), then, once P6 has named the candidate lags, Syy <- max(1, Syy + y[i+480]^2 - y[i]^2) up to the last
  //     candidate, keeping the value before each candidate lag (sm.s10) for P8;
  //   C (warp NW-3, lane = frame): remove_doubling's xx = sum x[j]^2 and its yy_lookup recurrence.
  // Both are complete before their consumers: B before P8, C before P12 (the P7 call finishes both).
  constexpr int NW = NT / 32;
  static_assert(NW >= 4, "chain warps B and C, the coarse helper and at least one worker warp");
  const int chain_lane = tid & 31;
  const bool chain_b = (tid >> 5) == NW - 2 && chain_lane < nfr, chain_c = (tid >> 5) == NW - 3 && chain_lane < nfr;
  float ch_acc = chain_b ? 1.f : 0.f;
  float ch_p1 = 0.f, ch_p2 = 0.f, ch_p3 = 0.f;  // chain C's partial sums of taps j = 1, 2, 3 (mod 4) under dot4
  int ch_blk = 0;  // blocks done: 30 for the sum of squares, then 19 (B) / 24 (C) for the recurrence
  auto chain_run = [&](int budget, bool recur_b) {
    if (!chain_b && !chain_c) return;
    const int f = chain_lane;
    const float *y = sm.xlp + f * kLpStride + (chain_c ? 384 : 0);
    for (; budget > 0 && ch_blk < 30; budget--, ch_blk++) {
      const float *q = y + 16 * ch_blk;
      const f4 v0 = ld4(q), v1 = ld4(q + 4), v2 = ld4(q + 8), v3 = ld4(q + 12);
      if constexpr (kSpDot4<SP>) {
        if (chain_c) {  // xx is dual_inner_prod's: dot4 (chain B's Syy belongs to find_best_pitch and stays sequential)
          ch_acc += v0.x * v0.x, ch_p1 += v0.y * v0.y, ch_p2 += v0.z * v0.z, ch_p3 += v0.w * v0.w;
          ch_acc += v1.x * v1.x, ch_p1 += v1.y * v1.y, ch_p2 += v1.z * v1.z, ch_p3 += v1.w * v1.w;
          ch_acc += v2.x * v2.x, ch_p1 += v2.y * v2.y, ch_p2 += v2.z * v2.z, ch_p3 += v2.w * v2.w;
          ch_acc += v3.x * v3.x, ch_p1 += v3.y * v3.y, ch_p2 += v3.z * v3.z, ch_p3 += v3.w * v3.w;
          if (ch_blk == 29) ch_acc = ((ch_acc + ch_p1) + ch_p2) + ch_p3;
        }
      }
      if (!kSpDot4<SP> || !chain_c) {
        ch_acc += v0.x * v0.x, ch_acc += v0.y * v0.y, ch_acc += v0.z * v0.z, ch_acc += v0.w * v0.w;
        ch_acc += v1.x * v1.x, ch_acc += v1.y * v1.y, ch_acc += v1.z * v1.z, ch_acc += v1.w * v1.w;
        ch_acc += v2.x * v2.x, ch_acc += v2.y * v2.y, ch_acc += v2.z * v2.z, ch_acc += v2.w * v2.w;
        ch_acc += v3.x * v3.x, ch_acc += v3.y * v3.y, ch_acc += v3.z * v3.z, ch_acc += v3.w * v3.w;
      }
      if (ch_blk == 29 && chain_c) {
        sm.xx[f] = ch_acc;
        sm.xr[f * kLpStride + 432] = ch_acc;  // yy_lookup[0]
      }
    }
    if (chain_b) {
      if (ch_blk < 30 || !recur_b) return;  // the recurrence waits for P6's candidates
      // candidate runs exactly as P8 walks them
      const int lo0 = 2 * sm.best0[f] - 2, lo1 = 2 * sm.best1[f] - 2;
      const int r1 = lo0 < lo1 ? lo0 : lo1, r2 = lo0 < lo1 ? lo1 : lo0;
      auto clampi = [](int v) { return v < 0 ? 0 : (v > 294 ? 294 : v); };
      const int a0 = clampi(r1), b0 = clampi(r2 > r1 + 5 ? r2 : r1 + 5), last = clampi(r2 + 5);
      float syy = ch_acc;
      for (int i0 = 0; i0 < last; i0 += 4) {
        const f4 ya = ld4(y + i0 + 480), yb = ld4(y + i0);
        const float d[4] = {ya.x * ya.x - yb.x * yb.x, ya.y * ya.y - yb.y * yb.y, ya.z * ya.z - yb.z * yb.z,
                            ya.w * ya.w - yb.w * yb.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int i = i0 + u;
          if ((unsigned)(i - a0) < 5u) sm.s10[f][i - a0] = syy;
          if ((unsigned)(i - b0) < 5u) sm.s10[f][5 + i - b0] = syy;
          syy += d[u];
          syy = syy < 1.f ? 1.f : syy;
        }
      }
      ch_blk = 1000;
    } else {
      float *yyl = sm.xr + f * kLpStride + 432;  // yy_lookup[0..384]
      for (; budget > 0 && ch_blk < 30 + 24; budget--, ch_blk++) {
        const int i1 = 1 + 16 * (ch_blk - 30);
        float yy = ch_acc;
#pragma unroll
        for (int h = 0; h < 4; h++) {  // lags i0..i0+3: x[-i] and x[480-i] come as two aligned float4s
          const int i0 = i1 + 4 * h;
          const f4 a = ld4(y - i0 - 3), c = ld4(y + 477 - i0);
          const float av[4] = {a.w * a.w, a.z * a.z, a.y * a.y, a.x * a.x};
          const float cv[4] = {c.w * c.w, c.z * c.z, c.y * c.y, c.x * c.x};
#pragma unroll
          for (int u = 0; u < 4; u++) {
            yy = yy + av[u] - cv[u];
            yyl[i0 + u] = yy < 0.f ? 0.f : yy;
          }
        }
        ch_acc = yy;
      }
    }
  };
  // P5: a10 coarse cross-correlation, 147 lags x 240 taps, eight lags per lane.  In its shadow the
  // last warp (idle when NT > 19 R + 32) runs the coarse find_best_pitch's Syy recurrence (it only needs y4).
  if (tid >= NT - 32) {
    const int l = tid - (NT - 32);
    if (l < nfr) {
      const float *y4 = sm.xr + l * kLpStride;
      syy_recurrence(sumsq_from<240>(1.f, y4), y4, 240, 147, sm.sb6[l]);
    }
  }
  // Under dot4 a lag holds four partial sums: four lags per lane keep the accumulators at sixteen registers.
  constexpr bool kD4x = kSpDot4Xcorr<SP>;
  constexpr int kLpl = kD4x ? 4 : 8, kQpf = 152 / kLpl;  // lags per lane, lanes per frame
  for (int it = tid; it < nfr * kQpf; it += NT) {  // eight lags per lane: one new float4 of y and one of x feed 32 MACs
    const int f = it / kQpf, q = it - f * kQpf;
    const float *y4 = sm.xr + f * kLpStride;
    const float *x4 = y4 + 192;
    const float *yb = y4 + kLpl * q;
    Acc4<kD4x> a[kLpl];
    f4 w0 = ld4(yb), w1 = ld4(yb + 4);
#pragma unroll 2
    for (int j = 0; j < 240; j += 4) {
      const f4 xv = ld4(x4 + j), w2 = ld4(yb + j + 8);
      const float w[12] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w};
      const float xt[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int l = 0; l < kLpl; l++) a[l].add(t, xt[t] * w[l + t]);
      w0 = w1;
      w1 = w2;
    }
    float *dst = sm.xc[f] + kLpl * q;
#pragma unroll
    for (int l = 0; l < kLpl; l += 4)
      *reinterpret_cast<f4 *>(dst + l) = f4{a[l].sum(), a[l + 1].sum(), a[l + 2].sum(), a[l + 3].sum()};
  }
  chain_run(25, false);
  Simt::cta_sync();
  NS_PHASE_MARK(7);
  // P6: find_best_pitch on the coarse correlation.  The serial scan (147 dependent insertions per frame) only has to
  // be replayed over the lags that can end up among its two winners: warp f scores its frame's 147 lags in parallel
  // (num / Syy, five lags per lane), takes the second best score, and runs the oracle's insertion, in lag order and
  // with the oracle's cross-multiplied comparisons, over the lags within 2e-4 of it -- two or three on speech and on
  // noise alike.  A lag further below loses every comparison against the two winners by a margin a thousand times
  // the float32 rounding of either side, and a lag that cannot win does not change which lags do, so the result is
  // the full scan's, bit for bit.  Where that margin means nothing -- the threshold lag's num = (xc 1e-12)^2 near the
  // float32 underflow range (a signal decaying through the denormals), or more than 32 lags within the margin --
  // lane 0 runs the full scan.
  if (NW > R && (tid >> 5) < R) {
    const int f = tid >> 5, lane = tid & 31;
    if (f < nfr) {
      float sc[5], xcv[5], syv[5];
      float t0v = -1.f, t1v = -1.f, t1num = 0.f, t0num = 0.f;  // two best scores and their nums
      int nvalid = 0;
#pragma unroll
      for (int u = 0; u < 5; u++) {
        const int i = lane + 32 * u;
        const bool in = i < 147;
        xcv[u] = in ? sm.xc[f][i] : 0.f;
        syv[u] = in ? sm.sb6[f][i] : 1.f;
        const float x16 = xcv[u] * 1e-12f, num = x16 * x16;
        const bool valid = in && xcv[u] > 0.f;
        sc[u] = valid ? num / syv[u] : -1.f;
        nvalid += valid ? 1 : 0;
        const bool a = sc[u] > t0v, bb = sc[u] > t1v;
        t1v = a ? t0v : (bb ? sc[u] : t1v);
        t1num = a ? t0num : (bb ? num : t1num);
        t0v = a ? sc[u] : t0v;
        t0num = a ? num : t0num;
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        const float o0 = Simt::shfl_xor(t0v, d), o1 = Simt::shfl_xor(t1v, d), n0 = Simt::shfl_xor(t0num, d), n1 = Simt::shfl_xor(t1num, d);
        nvalid += Simt::shfl_xor(nvalid, d);
        // merge (o0, o1) into (t0v, t1v)
        bool a = o0 > t0v, bb = o0 > t1v;
        t1v = a ? t0v : (bb ? o0 : t1v);
        t1num = a ? t0num : (bb ? n0 : t1num);
        t0v = a ? o0 : t0v;
        t0num = a ? n0 : t0num;
        bb = o1 > t1v;
        t1num = bb ? n1 : t1num;
        t1v = bb ? o1 : t1v;
      }
      const float thr = nvalid >= 2 ? t1v * (1.f - 2e-4f) : -1.f;
      unsigned mine = 0u;
      int cnt = 0;
#pragma unroll
      for (int u = 0; u < 5; u++)
        if (sc[u] >= 0.f && sc[u] >= thr) mine |= 1u << u, cnt++;
      int total = cnt;
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) total += Simt::shfl_xor(total, d);
      Best2 b;
      best_init(b);
      if (total > 32 || (nvalid >= 2 && !(t1num >= 1e-30f))) {  // the margin argument does not apply: full scan
        if (lane == 0) {
          for (int i = 0; i < 147; i++) {
            const float xc = sm.xc[f][i];
            const float x16 = xc * 1e-12f;
            best_insert_sel(b, xc > 0.f, x16 * x16, sm.sb6[f][i], i);
          }
        }
      } else {
        for (int s = 0; s < total; s++) {  // the candidates in ascending lag order: every lane replays the insertion
          int mn = 0x7FFFFFFF;
#pragma unroll
          for (int u = 0; u < 5; u++)
            if (mine & (1u << u)) {
              const int i = lane + 32 * u;
              mn = i < mn ? i : mn;
            }
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) {
            const int o = Simt::shfl_xor(mn, d);
            mn = o < mn ? o : mn;
          }
          const int src = mn & 31, u = mn >> 5;
          float xc = 0.f, sy = 1.f;
#pragma unroll
          for (int uu = 0; uu < 5; uu++)
            if (uu == u) xc = xcv[uu], sy = syv[uu];
          xc = Simt::shfl(xc, src);
          sy = Simt::shfl(sy, src);
          const float x16 = xc * 1e-12f;
          best_insert_sel(b, xc > 0.f, x16 * x16, sy, mn);
          if (lane == src) mine &= ~(1u << u);
        }
      }
      if (lane == 0) {
        sm.best0[f] = b.p0;
        sm.best1[f] = b.p1;
      }
    }
  } else if (NW <= R && tid < nfr) {  // narrow CTAs (measurement variants, the host emulation's small build): one lane per frame
    const int f = tid;
    Best2 b;
    best_init(b);
    for (int i0 = 0; i0 < 147; i0 += 4) {  // Syy per lag comes from the helper warp
      const f4 xc4 = ld4(sm.xc[f] + i0), sy4 = ld4(sm.sb6[f] + i0);
      const float xcv[4] = {xc4.x, xc4.y, xc4.z, xc4.w}, syv[4] = {sy4.x, sy4.y, sy4.z, sy4.w};
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (i0 + u < 147) {
          const float x16 = xcv[u] * 1e-12f;
          best_insert_sel(b, xcv[u] > 0.f, x16 * x16, syv[u], i0 + u);
        }
      }
    }
    sm.best0[f] = b.p0;
    sm.best1[f] = b.p1;
  }
  chain_run(20, false);  // B's sum of squares completes here; C keeps a share for P7
  Simt::cta_sync();
  NS_PHASE_MARK(8);
  // P7: fine search, at most ten lags around 2*best0 and 2*best1 (chain C finishes in its shadow)
  for (int it = tid; it < nfr * 10; it += NT) {
    const int f = it / 10, c = it - f * 10;
    const float *lp = sm.xlp + f * kLpStride;
    const int c0 = 2 * sm.best0[f], c1 = 2 * sm.best1[f];
    const int i = (c < 5) ? (c0 - 2 + c) : (c1 - 2 + (c - 5));
    const int dd = i - c0;
    const bool ok = (i >= 0) && (i < 294) && (c < 5 || dd > 2 || dd < -2);
    float sum = 0.f;
    if (ok) sum = dot480_shifted<kSpDot4<SP>>(lp, i);
    sm.fi[f][c] = ok ? i : -1;
    sm.fx[f][c] = sum < -1.f ? -1.f : sum;
  }
  chain_run(1000, true);
  Simt::cta_sync();
  NS_PHASE_MARK(9);
  // P8: find_best_pitch on the fine correlation (zero outside the candidates), pseudo-interpolation
  if (tid < nfr) {
    const int f = tid;
    const float *y = sm.xlp + f * kLpStride;
    const int lo0 = 2 * sm.best0[f] - 2, lo1 = 2 * sm.best1[f] - 2;
    auto xcorr_at = [&](int i) -> float {
      const int d0 = i - lo0, d1 = i - lo1;
      if (d0 >= 0 && d0 < 5 && sm.fi[f][d0] == i) return sm.fx[f][d0];
      if (d1 >= 0 && d1 < 5 && sm.fi[f][5 + d1] == i) return sm.fx[f][5 + d1];
      return 0.f;
    };
    Best2 b;
    best_init(b);
    // only the two runs of five candidate lags are compared; Syy before each of them came from chain B
    const int r1 = lo0 < lo1 ? lo0 : lo1, r2 = lo0 < lo1 ? lo1 : lo0;
    auto clampi = [](int v) { return v < 0 ? 0 : (v > 294 ? 294 : v); };
    const int a0 = clampi(r1), a1 = clampi(r1 + 5), b0 = clampi(r2 > r1 + 5 ? r2 : r1 + 5), b1 = clampi(r2 + 5);
    auto checked = [&](int from, int to, const float *syy) {
      for (int i = from; i < to; i++) {
        const float xc = xcorr_at(i);
        const float x16 = xc * 1e-12f;
        best_insert_sel(b, xc > 0.f, x16 * x16, syy[i - from], i);
      }
    };
    checked(a0, a1, sm.s10[f]);
    checked(b0, b1, sm.s10[f] + 5);
    const int bp = b.p0;
    int offset = 0;
    if (bp > 0 && bp < 293) {
      const float a = xcorr_at(bp - 1), bb = xcorr_at(bp), cc = xcorr_at(bp + 1);
      if ((cc - a) > .7f * (bb - a))
        offset = 1;
      else if ((a - cc) > .7f * (bb - cc))
        offset = -1;
    }
    const int pitch_index = kPitchMax - (2 * bp - offset);
    int T0 = pitch_index / 2;
    if (T0 >= 384) T0 = 383;
    sm.T0[f] = T0;
  }
  Simt::cta_sync();
  NS_PHASE_MARK(10);
  // P9 (a11 remove_doubling): xx came from the helper warp above; xy(T0) is one more item of the work list
  // P10: the candidate work list, one lane per (frame, k).  k is examined iff T0/k stays >= 30 (T1 is
  // non-increasing in k, so this equals upstream's break).  Every k contributes the three consecutive
  // lags T-1, T, T+1 (one "triple": their lagged windows overlap, so one pass over x and y feeds all
  // three sums) and, for k >= 2, the single lag T1b.  Items are bucketed by the alignment of their
  // window so that a whole warp shares a compile-time shift in P11.
  for (int it = tid; it < nfr * 16; it += NT) {
    const int f = it >> 4, k = it & 15;
    if (k == 0) continue;
    const int T0 = sm.T0[f];
    if (k > 1 && rd_T1(k, T0) < 30) continue;
    if (k == kMaxK || rd_T1(k + 1, T0) < 30) sm.nk[f] = k;
    const int Tc = (k == 1) ? T0 : rd_T1(k, T0);
    {
      const int idx = Simt::atomic_add_shared(&sm.n_tri[0], 1);
      (&sm.tri[0][0])[idx] = (uint32_t)(f | (Tc << 5) | (k << 14));
    }
    if (k > 1) {
      const int T1b = rd_T1b(k, T0, Tc);
      const int idx = Simt::atomic_add_shared(&sm.n_sgl[0], 1);
      (&sm.sgl[0][0])[idx] = (uint32_t)(f | (T1b << 5) | (k << 14));
    }
  }
  Simt::cta_sync();
  NS_PHASE_MARK(11);
  // P11: the inner products, one lane per item whatever its window alignment (dot3_shifted): full warps.  Triples
  // first (three chains each), the singles on the warps after them.
  {
    const int w = tid >> 5, lane = tid & 31;
    const int n_tri = sm.n_tri[0], n_sgl = sm.n_sgl[0];
    const int tri_warps = (n_tri + 31) >> 5, sgl_warps = (n_sgl + 31) >> 5;
    for (int job = w; job < tri_warps + sgl_warps; job += NW) {
      if (job < tri_warps) {
        const int it = job * 32 + lane;
        if (it < n_tri) {
          const int e = (&sm.tri[0][0])[it];
          const int f = e & 31, Tc = (e >> 5) & 0x1FF, k = e >> 14;
          const float *row = sm.xlp + f * kLpStride;
          float sp, sc, sm1;  // lags Tc+1, Tc, Tc-1
          dot3_shifted<480, kSpDot4<SP>>(row + 384, row, 384 - Tc - 1, sp, sc, sm1);
          const int d = 2 + 4 * (k - 2);
          sm.dots[f][k == 1 ? 0 : d] = sm1;
          sm.dots[f][k == 1 ? kDotXy0 : d + 1] = sc;
          sm.dots[f][k == 1 ? 1 : d + 2] = sp;
        }
      } else {
        const int it = (job - tri_warps) * 32 + lane;
        if (it < n_sgl) {
          const int e = (&sm.sgl[0][0])[it];
          const int f = e & 31, lag = (e >> 5) & 0x1FF, k = e >> 14;
          const float *row = sm.xlp + f * kLpStride;
          sm.dots[f][2 + 4 * (k - 2) + 3] = dot_shifted<480, kSpDot4<SP>>(row + 384, row, 384 - lag);
        }
      }
    }
  }
  Simt::cta_sync();
  NS_PHASE_MARK(12);
  // P12: per candidate k: gain, the pitch gain it would report, refined pitch index -> table
  for (int it = tid; it < nfr * 16; it += NT) {
    const int f = it >> 4, k = it & 15;  // k == 0 writes the header
    uint32_t *tab = p.tab + ((long long)stream * p.chunk_cap + (t0 + f)) * kTabWords;
    const int T0 = sm.T0[f], nk = sm.nk[f];
    if (k == 0) {
      tab[0] = (uint32_t)T0 | ((uint32_t)nk << 16);
      tab[1] = 0u;
      continue;
    }
    if (k > nk) continue;
    const float *yyl = sm.xr + f * kLpStride + 432;
    const float xx = sm.xx[f];
    float xy, yy, c0, c1, c2;
    int T;
    if (k == 1) {
      T = T0;
      xy = sm.dots[f][kDotXy0];
      yy = yyl[T0];
      c0 = sm.dots[f][0];
      c1 = xy;
      c2 = sm.dots[f][1];
    } else {
      const int d = 2 + 4 * (k - 2);
      T = rd_T1(k, T0);
      const int T1b = rd_T1b(k, T0, T);
      c0 = sm.dots[f][d];
      c1 = sm.dots[f][d + 1];
      c2 = sm.dots[f][d + 2];
      xy = .5f * (c1 + sm.dots[f][d + 3]);
      yy = .5f * (yyl[T] + yyl[T1b]);
    }
    const float g = pitch_gain_f(xy, xx, yy);
    const float bxy = xy < 0.f ? 0.f : xy;
    float pg = (yy <= bxy) ? 1.f : bxy / (yy + 1.f);
    if (pg > g) pg = g;
    int offset = 0;
    if ((c2 - c0) > .7f * (c1 - c0))
      offset = 1;
    else if ((c0 - c2) > .7f * (c1 - c2))
      offset = -1;
    int pi = 2 * T + offset;
    if (pi < kPitchMin) pi = kPitchMin;
    uint32_t *e = tab + 2 + 3 * (k - 1);
    e[0] = (uint32_t)T | ((uint32_t)pi << 16);
    e[1] = f2u(g);
    e[2] = f2u(pg);
  }
  NS_PHASE_MARK(13);
}

// =================================================================================================
// K2: the serial part of remove_doubling.  One warp per stream; lane k-1 judges candidate k against
// the threshold that depends on the previous frame's period and gain; the last passing k wins.
// =================================================================================================
NS_DEV void pitchscan_body(const Params &p, int warps_per_cta) {
  const int lane = Simt::tid() & 31;
  const int stream = Simt::cta() * warps_per_cta + (Simt::tid() >> 5);
  if (stream >= p.n_streams) return;
  float *st = p.state + (long long)stream * kStateFloats;
  int last_period = reinterpret_cast<int *>(st)[kStLastPeriod];
  float last_gain = st[kStLastGain];
  const uint32_t *tab = p.tab + (long long)stream * p.chunk_cap * kTabWords;
  float *rec = p.rec + (long long)stream * p.chunk_cap * kRecFloats;
  const int k = lane + 1;
  for (int t = 0; t < p.n_frames; t++, tab += kTabWords, rec += kRecFloats) {
    const uint32_t hdr = tab[0];
    const int T0 = (int)(hdr & 0xFFFFu), nk = (int)(hdr >> 16);
    uint32_t w0 = 0u;
    float g1 = 0.f, pg = 0.f;
    if (k <= nk) {
      w0 = tab[2 + 3 * lane];
      g1 = u2f(tab[3 + 3 * lane]);
      pg = u2f(tab[4 + 3 * lane]);
    }
    const float g0 = Simt::shfl(g1, 0);
    const int T1 = (int)(w0 & 0xFFFFu);
    const int prev_period = last_period / 2;
    bool pass = (k == 1);
    if (k >= 2 && k <= nk) {
      const int dT = T1 > prev_period ? T1 - prev_period : prev_period - T1;
      float cont;
      if (dT <= 1)
        cont = last_gain;
      else if (dT <= 2 && 5 * k * k < T0)
        cont = .5f * last_gain;
      else
        cont = 0.f;
      float thresh = .7f * g0 - cont;
      if (thresh < .3f) thresh = .3f;
      if (T1 < 90) {
        thresh = .85f * g0 - cont;
        if (thresh < .4f) thresh = .4f;
      } else if (T1 < 60) {
        thresh = .9f * g0 - cont;
        if (thresh < .5f) thresh = .5f;
      }
      pass = g1 > thresh;
    }
    const unsigned m = Simt::ballot(pass);
    int win = 0;
    for (int b = 14; b > 0; b--)
      if (m & (1u << b)) {
        win = b;
        break;
      }
    const int pi = (int)(Simt::shfl((int)w0, win) >> 16) & 0xFFFF;
    const float gain = Simt::shfl(pg, win);
    last_period = pi;
    last_gain = gain;
    if (lane == 0) {
      reinterpret_cast<int *>(rec)[kRecPitchIndex] = pi;
      rec[kRecPitchGain] = gain;
    }
  }
  if (lane == 0) {
    reinterpret_cast<int *>(st)[kStLastPeriod] = last_period;
    st[kStLastGain] = last_gain;
  }
}

// =================================================================================================
// spectra: 480-point complex FFT (forward), Stockham radices 4,4,5,6 through registers, by a
// 128-thread group that meets on its own named barrier
// =================================================================================================
// K3 / K5 view of the constant tables: the FFT twiddles are indexed irregularly per lane, so they live in
// shared memory; the window, DCT and band tables are read in order (coalesced) and come through L1 with
// read-only loads, which frees the shared memory for the staging buffers of the next frame.
struct SpecTw {
  cf w480[480];
  cf w960[244];
#ifndef NS_FFT3  // four stages 4.4.5.6: the product.  -DNS_FFT3 builds three stages 8.10.6 (a quarter fewer trips through shared
                 // memory, one barrier fewer, but only 60 / 48 / 80 busy lanes per stage): measured no faster on B200
                 // (spectrum 224 vs 214 us, synthesis 171 vs 171 us per 32,768 frames), so it stays a variant
  cf tw3[64];  // third FFT stage (radix 5, 16 sub-transforms): w480[6 r k] for r = 1..4, k < 16, contiguous in k --
               // read straight from w480 the sixteen lanes of a half-warp stride 48 r bytes (up to 8-way conflicts)
#else          // three stages 8.10.6: second stage (radix 10, 8 sub-transforms): w480[6 r k], r = 1..9, k < 8, contiguous in k
  cf tw3[72];
#endif
};
struct Tab {
  const SpecTw *s;
  const Tables *g;
  NS_DEV cf w480(int i) const { return s->w480[i]; }
  NS_DEV cf w960(int i) const { return s->w960[i]; }
#ifndef NS_FFT3
  NS_DEV cf tw3(int r, int k) const { return s->tw3[(r - 1) * 16 + k]; }
#else
  NS_DEV cf tw3(int r, int k) const { return s->tw3[(r - 1) * 8 + k]; }
#endif
  NS_DEV float win(int i) const { return Simt::ldg(g->win + i); }
  NS_DEV float dct(int i) const { return Simt::ldg(g->dct + i); }
  NS_DEV int bin_band(int i) const { return Simt::ldg(g->bin_band + i); }
  NS_DEV int eband(int i) const { return Simt::ldg(g->eband + i); }
  NS_DEV f4 win4(int i) const { return ldg_f4(g->win + i); }
  NS_DEV f4 bin_frac4(int i) const { return ldg_f4(g->bin_frac + i); }
  static NS_DEV f4 ldg_f4(const float *p) {
#if defined(__CUDACC__) && !defined(NS_HOST_EMU)
    const float4 v = Simt::ldg4(p);
    return f4{v.x, v.y, v.z, v.w};
#else
    return *reinterpret_cast<const f4 *>(p);
#endif
  }
};

struct Grp {
  int tid, lane, warp, bar;
};
NS_DEV void gsync(const Grp &g) { Simt::group_sync(g.bar, kGroupThreads); }
NS_DEV cf cmul(cf a, cf b) {
  cf c;
  c.x = fmaf(a.x, b.x, -(a.y * b.y));
  c.y = fmaf(a.x, b.y, a.y * b.x);
  return c;
}
NS_DEV cf cadd(cf a, cf b) { return cf{a.x + b.x, a.y + b.y}; }
NS_DEV cf csub(cf a, cf b) { return cf{a.x - b.x, a.y - b.y}; }
NS_DEV cf mul_neg_i(cf a) { return cf{a.y, -a.x}; }  // a * (-i)
NS_DEV cf mul_pos_i(cf a) { return cf{-a.y, a.x}; }  // a * (+i)

template <int R>
struct Dft;
template <>
struct Dft<3> {
  static NS_DEV void run(cf *v) {
    const float s = 0.86602540378443864676f;
    cf a = cadd(v[1], v[2]), b = csub(v[1], v[2]);
    cf m = cf{fmaf(-0.5f, a.x, v[0].x), fmaf(-0.5f, a.y, v[0].y)};
    cf n = cf{s * b.x, s * b.y};
    v[0] = cadd(v[0], a);
    v[1] = cadd(m, mul_neg_i(n));
    v[2] = cadd(m, mul_pos_i(n));
  }
};
template <>
struct Dft<4> {
  static NS_DEV void run(cf *v) {
    cf t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
    cf t2 = cadd(v[1], v[3]), t3 = mul_neg_i(csub(v[1], v[3]));
    v[0] = cadd(t0, t2);
    v[2] = csub(t0, t2);
    v[1] = cadd(t1, t3);
    v[3] = csub(t1, t3);
  }
};
template <>
struct Dft<5> {
  static NS_DEV void run(cf *v) {
    const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
    const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
    cf a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
    cf b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
    cf m1 = cf{fmaf(c2, a2.x, fmaf(c1, a1.x, v[0].x)), fmaf(c2, a2.y, fmaf(c1, a1.y, v[0].y))};
    cf m2 = cf{fmaf(c1, a2.x, fmaf(c2, a1.x, v[0].x)), fmaf(c1, a2.y, fmaf(c2, a1.y, v[0].y))};
    cf n1 = cf{fmaf(s2, b2.x, s1 * b1.x), fmaf(s2, b2.y, s1 * b1.y)};
    cf n2 = cf{fmaf(-s1, b2.x, s2 * b1.x), fmaf(-s1, b2.y, s2 * b1.y)};
    v[0] = cf{v[0].x + a1.x + a2.x, v[0].y + a1.y + a2.y};
    v[1] = cadd(m1, mul_neg_i(n1));
    v[4] = cadd(m1, mul_pos_i(n1));
    v[2] = cadd(m2, mul_neg_i(n2));
    v[3] = cadd(m2, mul_pos_i(n2));
  }
};
template <>
struct Dft<6> {
  static NS_DEV void run(cf *v) {
    cf e[3] = {v[0], v[2], v[4]};
    cf o[3] = {v[1], v[3], v[5]};
    Dft<3>::run(e);
    Dft<3>::run(o);
    const cf w1 = cf{0.5f, -0.86602540378443864676f};   // W6
    const cf w2 = cf{-0.5f, -0.86602540378443864676f};  // W6^2
    o[1] = cmul(o[1], w1);
    o[2] = cmul(o[2], w2);
    v[0] = cadd(e[0], o[0]);
    v[1] = cadd(e[1], o[1]);
    v[2] = cadd(e[2], o[2]);
    v[3] = csub(e[0], o[0]);
    v[4] = csub(e[1], o[1]);
    v[5] = csub(e[2], o[2]);
  }
};

template <>
struct Dft<8> {
  static NS_DEV void run(cf *v) {
    const float h = 0.70710678118654752440f;
    cf e[4] = {v[0], v[2], v[4], v[6]};
    cf o[4] = {v[1], v[3], v[5], v[7]};
    Dft<4>::run(e);
    Dft<4>::run(o);
    // W8^1 = (1 - i) / sqrt 2, W8^2 = -i, W8^3 = (-1 - i) / sqrt 2
    const cf o1 = cf{h * (o[1].x + o[1].y), h * (o[1].y - o[1].x)};
    const cf o2 = mul_neg_i(o[2]);
    const cf o3 = cf{h * (o[3].y - o[3].x), -h * (o[3].x + o[3].y)};
    v[0] = cadd(e[0], o[0]);
    v[4] = csub(e[0], o[0]);
    v[1] = cadd(e[1], o1);
    v[5] = csub(e[1], o1);
    v[2] = cadd(e[2], o2);
    v[6] = csub(e[2], o2);
    v[3] = cadd(e[3], o3);
    v[7] = csub(e[3], o3);
  }
};
template <>
struct Dft<10> {
  static NS_DEV void run(cf *v) {
    cf e[5] = {v[0], v[2], v[4], v[6], v[8]};
    cf o[5] = {v[1], v[3], v[5], v[7], v[9]};
    Dft<5>::run(e);
    Dft<5>::run(o);
    // W10^k = exp(-2 pi i k / 10), k = 1..4
    const cf w1 = cf{0.80901699437494742410f, -0.58778525229247312917f};
    const cf w2 = cf{0.30901699437494742410f, -0.95105651629515357212f};
    const cf w3 = cf{-0.30901699437494742410f, -0.95105651629515357212f};
    const cf w4 = cf{-0.80901699437494742410f, -0.58778525229247312917f};
    o[1] = cmul(o[1], w1);
    o[2] = cmul(o[2], w2);
    o[3] = cmul(o[3], w3);
    o[4] = cmul(o[4], w4);
#pragma unroll
    for (int k = 0; k < 5; k++) {
      v[k] = cadd(e[k], o[k]);
      v[k + 5] = csub(e[k], o[k]);
    }
  }
};

// Stockham scatter of one butterfly's outputs, ordered so that the lanes of one shared-memory transaction hit
// different banks:
//  * first stage (NS = 1, R = 4): a thread owns 32 contiguous bytes and writes them as two 16-byte stores; the
//    upper half of every quarter-warp writes its two halves in the other order (straight order is 2-way conflicted);
//  * second stage (R = 4, NS = 4): output r of butterfly j = 4g + k goes to bin 16g + k + 4r, so for a fixed r the
//    sixteen lanes of a half-warp cover only four bank groups (4-way conflict); lane group g therefore writes
//    its outputs rotated by g, r = (s + g) mod 4 at step s, which makes the sixteen addresses distinct mod 16 bins.
// The rotations are selects on registers (no dynamic indexing).
template <int R, int NS_>
NS_DEV void fft_store(cf *buf, int j, int k, const cf (&v)[R]) {
  const int j0 = (j - k) * R + k;
  if (NS_ == 1 && R == 4) {
    f4 *d = reinterpret_cast<f4 *>(buf + j0);
    const bool sw = (j & 4) != 0;
    const f4 lo = f4{v[0].x, v[0].y, v[1].x, v[1].y}, hi = f4{v[2].x, v[2].y, v[3].x, v[3].y};
    d[sw ? 1 : 0] = sw ? hi : lo;
    d[sw ? 0 : 1] = sw ? lo : hi;
  } else if (NS_ == 1 && R == 8) {
    // a thread owns 64 contiguous bytes (four 16-byte chunks); a quarter-warp's lanes are 64 B apart, so chunk c of
    // lane l sits in bank group (4 l + c) mod 8: lane l writes chunk (s + l / 2) mod 4 at step s -> eight distinct groups
    f4 *d = reinterpret_cast<f4 *>(buf + j0);
    const int rot = (j >> 1) & 3;
    f4 c[4] = {f4{v[0].x, v[0].y, v[1].x, v[1].y}, f4{v[2].x, v[2].y, v[3].x, v[3].y}, f4{v[4].x, v[4].y, v[5].x, v[5].y},
               f4{v[6].x, v[6].y, v[7].x, v[7].y}};
    if (rot & 1) {
      const f4 t0 = c[0];
      c[0] = c[1], c[1] = c[2], c[2] = c[3], c[3] = t0;
    }
    if (rot & 2) {
      const f4 t0 = c[0], t1 = c[1];
      c[0] = c[2], c[1] = c[3], c[2] = t0, c[3] = t1;
    }
#pragma unroll
    for (int st = 0; st < 4; st++) d[(st + rot) & 3] = c[st];  // c[st] holds chunk (st + rot) & 3
  } else if (NS_ == 4 && R == 4) {
    const int rot = (j >> 2) & 3;
    cf w[4] = {v[0], v[1], v[2], v[3]};
    if (rot & 1) {  // w[s] <- w[s + 1]
      const cf t0 = w[0];
      w[0] = w[1], w[1] = w[2], w[2] = w[3], w[3] = t0;
    }
    if (rot & 2) {  // w[s] <- w[s + 2]
      const cf t0 = w[0], t1 = w[1];
      w[0] = w[2], w[1] = w[3], w[2] = t0, w[3] = t1;
    }
#pragma unroll
    for (int s = 0; s < 4; s++) buf[j0 + ((s + rot) & 3) * 4] = w[s];  // w[s] == v[(s + rot) & 3]
  } else if (NS_ == 1 && (R & 1) == 0) {
    f4 *d = reinterpret_cast<f4 *>(buf + j0);
#pragma unroll
    for (int r = 0; r < R; r += 2) d[r >> 1] = f4{v[r].x, v[r].y, v[r + 1].x, v[r + 1].y};
  } else {
#pragma unroll
    for (int r = 0; r < R; r++) buf[j0 + r * NS_] = v[r];
  }
}

// the stage whose twiddles come from the compact table SpecTw::tw3
#ifndef NS_FFT3
template <int R, int NS_>
constexpr bool kTw3Stage = (R == 5 && NS_ == 16);
#else
template <int R, int NS_>
constexpr bool kTw3Stage = (R == 10 && NS_ == 8);
#endif

// PP ("ping-pong"): the stage stores into a buffer it does not load from, so the barrier between the loads and the
// stores is not needed
template <int R, int NS_, bool PP = false, class Load>
NS_DEV void fft_stage(const Grp &g, const Tab &T, cf *buf, Load load) {
  constexpr int M = 480 / R;
  constexpr int TSTEP = 480 / (NS_ * R);
  cf v[R];
  const int j = g.tid;
  const bool act = j < M;
  int k = 0;
  if (act) {
    k = j % NS_;
    v[0] = load(j);
#pragma unroll
    for (int r = 1; r < R; r++) {
      cf x = load(j + r * M);
      v[r] = (NS_ == 1) ? x : cmul(x, kTw3Stage<R, NS_> ? T.tw3(r, k) : T.w480(r * k * TSTEP));
    }
    Dft<R>::run(v);
  }
  if (!PP) gsync(g);
  if (act) fft_store<R, NS_>(buf, j, k, v);
  gsync(g);
}

// two independent transforms side by side (same twiddles, same barriers): K3's frame and pitch-lag spectra
template <int R, int NS_, bool PP = false, class Load2>
NS_DEV void fft_stage2(const Grp &g, const Tab &T, cf *bufA, cf *bufB, Load2 load2) {
  constexpr int M = 480 / R;
  constexpr int TSTEP = 480 / (NS_ * R);
  cf va[R], vb[R];
  const int j = g.tid;
  const bool act = j < M;
  int k = 0;
  if (act) {
    k = j % NS_;
    load2(j, va[0], vb[0]);
#pragma unroll
    for (int r = 1; r < R; r++) {
      load2(j + r * M, va[r], vb[r]);
      if (NS_ != 1) {
        const cf w = kTw3Stage<R, NS_> ? T.tw3(r, k) : T.w480(r * k * TSTEP);
        va[r] = cmul(va[r], w);
        vb[r] = cmul(vb[r], w);
      }
    }
    Dft<R>::run(va);
    Dft<R>::run(vb);
  }
  if (!PP) gsync(g);
  if (act) {
    fft_store<R, NS_>(bufA, j, k, va);
    fft_store<R, NS_>(bufB, j, k, vb);
  }
  gsync(g);
}

// two independent transforms, one per half of the group (threads 0..63: A, 64..127: B): the stages with at most 64
// butterflies per transform (radix 8: 60, radix 10: 48)
template <int R, int NS_, bool PP = false, class LoadA, class LoadB>
NS_DEV void fft_stage_split(const Grp &g, const Tab &T, cf *bufA, cf *bufB, LoadA loadA, LoadB loadB) {
  constexpr int M = 480 / R;
  constexpr int TSTEP = 480 / (NS_ * R);
  static_assert(M <= 64, "one half of the group per transform");
  cf v[R];
  const int j = g.tid & 63;
  const bool second = g.tid >= 64, act = j < M;
  int k = 0;
  if (act) {
    k = j % NS_;
#pragma unroll
    for (int r = 0; r < R; r++) {
      const cf x = second ? loadB(j + r * M) : loadA(j + r * M);
      v[r] = (NS_ == 1 || r == 0) ? x : cmul(x, kTw3Stage<R, NS_> ? T.tw3(r, k) : T.w480(r * k * TSTEP));
    }
    Dft<R>::run(v);
  }
  if (!PP) gsync(g);
  if (act) fft_store<R, NS_>(second ? bufB : bufA, j, k, v);
  gsync(g);
}

// a7 / a12: X <- rFFT960(window . src[0..960)) / 960 (bins 0..480) for two windows at once (X of the frame, P of the
// pitch-lagged window): shared window, twiddle and barrier traffic
// (XA, XB) receive the result; (YA, YB) are scratch of the same size: the four stages ping-pong between them
NS_DEV void rfft960_windowed2(const Grp &g, const Tab &T, const float *win, const float *__restrict__ srcA,
                              const float *__restrict__ srcB, cf *XA, cf *XB, cf *YA, cf *YB) {
  auto load = [&](int n, cf &a, cf &b) {  // win: the half window in shared memory; srcA / srcB in HBM / L2
    const int i0 = 2 * n;  // even: both taps sit in the same half of the symmetric window -> one 8-byte read
    const bool up = i0 < kFrame;
    const cf wp = *reinterpret_cast<const cf *>(win + (up ? i0 : kWindow - 2 - i0));
    const float w0 = up ? wp.x : wp.y, w1 = up ? wp.y : wp.x;
    a = cf{srcA[i0] * w0, srcA[i0 + 1] * w1};
    b = cf{srcB[i0] * w0, srcB[i0 + 1] * w1};
  };
  auto from_x = [&](int n, cf &a, cf &b) {
    a = XA[n];
    b = XB[n];
  };
  auto from_y = [&](int n, cf &a, cf &b) {
    a = YA[n];
    b = YB[n];
  };
#ifndef NS_FFT3
  fft_stage2<4, 1, true>(g, T, YA, YB, load);
  fft_stage2<4, 4, true>(g, T, XA, XB, from_y);
  fft_stage2<5, 16, true>(g, T, YA, YB, from_x);
  fft_stage2<6, 80, true>(g, T, XA, XB, from_y);
#else
  // three stages 8 . 10 . 6: a quarter fewer trips of both spectra through shared memory and one barrier fewer; the
  // first two stages have at most 60 butterflies per transform, so each half of the group takes one transform
  auto loadA = [&](int n) -> cf {
    cf a, b;
    (void)b;
    const int i0 = 2 * n;
    const bool up = i0 < kFrame;
    const cf wp = *reinterpret_cast<const cf *>(win + (up ? i0 : kWindow - 2 - i0));
    const float w0 = up ? wp.x : wp.y, w1 = up ? wp.y : wp.x;
    a = cf{srcA[i0] * w0, srcA[i0 + 1] * w1};
    return a;
  };
  auto loadB = [&](int n) -> cf {
    const int i0 = 2 * n;
    const bool up = i0 < kFrame;
    const cf wp = *reinterpret_cast<const cf *>(win + (up ? i0 : kWindow - 2 - i0));
    const float w0 = up ? wp.x : wp.y, w1 = up ? wp.y : wp.x;
    return cf{srcB[i0] * w0, srcB[i0 + 1] * w1};
  };
  (void)load;
  fft_stage_split<8, 1, true>(g, T, XA, XB, loadA, loadB);
  fft_stage_split<10, 8, true>(g, T, YA, YB, [&](int n) -> cf { return XA[n]; }, [&](int n) -> cf { return XB[n]; });
  fft_stage2<6, 80, true>(g, T, XA, XB, from_y);
#endif
  const float norm = 1.0f / kWindow;
  for (int k = g.tid; k <= 240; k += kGroupThreads) {
    const cf w = T.w960(k);
#pragma unroll
    for (int q = 0; q < 2; q++) {
      cf *X = q ? XB : XA;
      const cf a = X[k], b = X[k == 0 ? 0 : 480 - k];
      const float er = .5f * (a.x + b.x), ei = .5f * (a.y - b.y);
      const float orr = .5f * (a.x - b.x), oi = .5f * (a.y + b.y);
      const float tr = fmaf(orr, w.x, -(oi * w.y)), ti = fmaf(orr, w.y, oi * w.x);
      X[k] = cf{(er + ti) * norm, (ei - tr) * norm};
      X[480 - k] = cf{(er - ti) * norm, (-ei - tr) * norm};
    }
  }
  gsync(g);
}

// a16: unscaled inverse of the Hermitian spectrum X[0..480]; result left in X as 480 complex
// z[m] with x[2m] = z[m].x and x[2m+1] = -z[m].y (the conjugate of a forward FFT).
NS_DEV void irfft960_inplace(const Grp &g, const Tab &T, cf *X, cf *Y) {  // Y: scratch of 481 cf (ping-pong partner)
#ifndef NS_FFT3
  cf *Z = X;  // four stages end where they started
#else
  cf *Z = Y;  // three stages: the Hermitian fold goes to the partner so that the last stage lands in X
#endif
  for (int k = g.tid; k <= 240; k += kGroupThreads) {
    const cf a = X[k], b = X[480 - k], w = T.w960(k);
    const float ex = a.x + b.x, ey = a.y - b.y;
    const float ox = a.x - b.x, oy = a.y + b.y;
    const float tr = fmaf(ox, w.x, oy * w.y), ti = fmaf(-ox, w.y, oy * w.x);
    Z[k] = cf{ex - ti, -(ey + tr)};
    if (k != 0) Z[480 - k] = cf{ex + ti, ey - tr};
  }
  gsync(g);
  auto from_x = [&](int n) -> cf { return X[n]; };
  auto from_y = [&](int n) -> cf { return Y[n]; };
#ifndef NS_FFT3
  fft_stage<4, 1, true>(g, T, Y, from_x);
  fft_stage<4, 4, true>(g, T, X, from_y);
  fft_stage<5, 16, true>(g, T, Y, from_x);
  fft_stage<6, 80, true>(g, T, X, from_y);
#else
  fft_stage<8, 1, true>(g, T, X, from_y);
  fft_stage<10, 8, true>(g, T, Y, from_x);
  fft_stage<6, 80, true>(g, T, X, from_y);
#endif
}

// a8: 22 triangular bands over bins 0..400.  Every band edge is a multiple of four bins, so bins
// 4s..4s+3 ("slot" s < 100, = one eband5ms unit) lie in one interval between two band centres.
// band_slots: thread s < 100 visits its four bins once, for NQ quantities at a time, and leaves the
// interval's two triangular partial sums (weight 1-f towards the lower band, f towards the upper one)
// in part[2q][s], part[2q+1][s].  band_reduce (after a group barrier): 88 threads, band = tid/4, four
// lanes add the partials of the two intervals that touch the band in a fixed order; results are valid
// in lanes with (tid & 3) == 0, tid < 88.
constexpr int kSlots = 100;
// a thread's slot = 32 contiguous bytes (four complex bins) as two 16-byte accesses; the upper half of every
// quarter-warp takes them in the other order so that the eight lanes of a transaction cover all 32 banks
NS_DEV void ld_slot(const cf *slot, bool sw, f4 &lo, f4 &hi) {
  const f4 *q = reinterpret_cast<const f4 *>(slot);
  const f4 a = q[sw ? 1 : 0], b = q[sw ? 0 : 1];
  lo = sw ? b : a;
  hi = sw ? a : b;
}
NS_DEV void st_slot(cf *slot, bool sw, f4 lo, f4 hi) {
  f4 *q = reinterpret_cast<f4 *>(slot);
  q[sw ? 1 : 0] = sw ? hi : lo;
  q[sw ? 0 : 1] = sw ? lo : hi;
}
constexpr int kPartStride = 100;
template <int NQ, class BinVal>
NS_DEV void band_slots(const Grp &g, const Tab &T, float *part, BinVal val) {
  if (g.tid < kSlots) {
    const int k0 = 4 * g.tid;
    const f4 fr4 = T.bin_frac4(k0);
    const float fr[4] = {fr4.x, fr4.y, fr4.z, fr4.w};
    float s0[NQ], s1[NQ];
#pragma unroll
    for (int q = 0; q < NQ; q++) s0[q] = s1[q] = 0.f;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      float v[NQ];
      val(u, v);
#pragma unroll
      for (int q = 0; q < NQ; q++) {
        s0[q] += v[q];
        s1[q] = fmaf(fr[u], v[q], s1[q]);
      }
    }
#pragma unroll
    for (int q = 0; q < NQ; q++) {
      part[(2 * q) * kPartStride + g.tid] = s0[q] - s1[q];
      part[(2 * q + 1) * kPartStride + g.tid] = s1[q];
    }
  }
}
template <int NQ>
NS_DEV void band_reduce(const Grp &g, const Tab &T, const float *part, float (&acc)[NQ]) {
#pragma unroll
  for (int q = 0; q < NQ; q++) acc[q] = 0.f;
  const int b = g.tid >> 2, sub = g.tid & 3;
  if (g.tid < 4 * kBands) {
    const int lo = (b >= 1) ? (T.eband(b - 1) >> 2) : 0;  // slots
    const int mid = T.eband(b) >> 2;
    const int hi = (b <= kBands - 2) ? (T.eband(b + 1) >> 2) : mid;
    for (int sl = mid + sub; sl < hi; sl += 4) {  // interval b: this band is its lower one
#pragma unroll
      for (int q = 0; q < NQ; q++) acc[q] += part[(2 * q) * kPartStride + sl];
    }
    for (int sl = lo + sub; sl < mid; sl += 4) {  // interval b-1: this band is its upper one
#pragma unroll
      for (int q = 0; q < NQ; q++) acc[q] += part[(2 * q + 1) * kPartStride + sl];
    }
  }
#pragma unroll
  for (int q = 0; q < NQ; q++) {
    acc[q] += Simt::shfl_xor(acc[q], 1);
    acc[q] += Simt::shfl_xor(acc[q], 2);
    if (b == 0 || b == kBands - 1) acc[q] *= 2.f;
  }
}

struct SpecSmem {
  SpecTw tw;
  // K3: spec[0] = X | P of the frame in work, spec[1] = the next task's raw windows (960 + 968 floats).
  // K5: the two halves hold X | P of the frame in work and of the next frame (double buffer by frame parity).
  cf spec[2][2 * kSpecStride];
  float rec_s[2][kRecFloats];  // K5: the frames' records, staged with the spectra
  float Ex[24], Ep[24], Exp[24], Ly[24], g[24], graw[24], r[24], nrm[24], newE[24];
  float synth[kFrame];
  float part[6 * kPartStride];  // band_slots -> band_reduce
  int pitch_index, silence;
  alignas(8) uint64_t mbar;  // completion of the bulk copies that stage the next frame
};
static_assert(sizeof(SpecSmem) <= 28160, "eight resident CTAs per SM: 8 x (sizeof + 1 KB) <= 228 KB");
static_assert(2 * kSpecStride * sizeof(cf) >= (960 + 968) * sizeof(float), "raw window staging fits one spectra buffer");

NS_DEV void load_twiddles(const Params &p, SpecTw &dst, int tid, int nthr) {
  static_assert(offsetof(Tables, w480) == 0 && offsetof(Tables, w960) == sizeof(cf) * 480, "twiddles lead the tables");
  const uint32_t *src = reinterpret_cast<const uint32_t *>(p.tables);
  uint32_t *d = reinterpret_cast<uint32_t *>(&dst);
  for (int i = tid; i < (int)(offsetof(SpecTw, tw3) / 4); i += nthr) d[i] = src[i];
#ifndef NS_FFT3
  for (int i = tid; i < 64; i += nthr) dst.tw3[i] = p.tables->w480[6 * ((i >> 4) + 1) * (i & 15)];
#else
  for (int i = tid; i < 72; i += nthr) dst.tw3[i] = p.tables->w480[6 * ((i >> 3) + 1) * (i & 7)];
#endif
}

// spectra of frame t: X of [prev | cur], P of the window lagged by pitch_index, Ex / Ep / raw Exp
// `res` selects the half of s.spec that receives X | P; the other half is the FFT's ping-pong partner.  With three FFT
// stages the first one already writes the result half, so consecutive tasks alternate `res`: the threads that race
// ahead into the next frame must not overwrite spectra the slower ones are still copying out.
NS_DEV void frame_spectra(const Grp &g, const Tab &T, SpecSmem &s, const float *hp_row, int t, int pitch_index, int res = 0) {
  const float *cur = hp_row + kHist - kFrame + (long long)t * kFrame;  // [analysis_mem | frame]
  cf *X = s.spec[res], *P = s.spec[res] + kSpecStride;
  // K3 keeps the window where K5 keeps synthesis_mem
  rfft960_windowed2(g, T, s.synth, cur, cur - pitch_index, X, P, s.spec[res ^ 1], s.spec[res ^ 1] + kSpecStride);
  {
    f4 xl, xh, pl, ph;
    const int sl = g.tid < kSlots ? g.tid : 0;
    const bool sw = (g.tid & 4) != 0;
    ld_slot(X + 4 * sl, sw, xl, xh);
    ld_slot(P + 4 * sl, sw, pl, ph);
    const cf xs[4] = {cf{xl.x, xl.y}, cf{xl.z, xl.w}, cf{xh.x, xh.y}, cf{xh.z, xh.w}};
    const cf ps[4] = {cf{pl.x, pl.y}, cf{pl.z, pl.w}, cf{ph.x, ph.y}, cf{ph.z, ph.w}};
    band_slots<3>(g, T, s.part, [&](int u, float (&v)[3]) {  // u: bin within the slot
      const cf x = xs[u], p = ps[u];
      v[0] = fmaf(x.x, x.x, x.y * x.y);
      v[1] = fmaf(p.x, p.x, p.y * p.y);
      v[2] = fmaf(x.x, p.x, x.y * p.y);
    });
  }
  gsync(g);
  float acc[3];
  band_reduce<3>(g, T, s.part, acc);
  if (g.tid < 4 * kBands && (g.tid & 3) == 0) {
    s.Ex[g.tid >> 2] = acc[0];
    s.Ep[g.tid >> 2] = acc[1];
    s.Exp[g.tid >> 2] = acc[2];
  }
  gsync(g);
}

// =================================================================================================
// K3: per (stream, frame): spectra -> band features that do not depend on recurrent state
// =================================================================================================
NS_DEV void spectrum_body(const Params &p, SpecSmem &s) {
  Grp g;
  g.tid = Simt::tid();
  g.lane = g.tid & 31;
  g.warp = g.tid >> 5;
  g.bar = 1;
  load_twiddles(p, s.tw, g.tid, kGroupThreads);
  for (int i = g.tid; i < kFrame; i += kGroupThreads) s.synth[i] = p.tables->win[i];
  Simt::cta_sync();
  const Tab T{&s.tw, p.tables};
  const float dct_scale = 0.30151134457776363f;  // sqrt(2/22)
  // a CTA's tasks are n_ctas apart: (stream, t) advance by (dq, dr) with a carry, no division per task
  const int dq = Simt::n_ctas() / p.n_frames, dr = Simt::n_ctas() - dq * p.n_frames;
  int stream = Simt::cta() / p.n_frames, t = Simt::cta() - stream * p.n_frames;
  int task_parity = 0;
  (void)task_parity;
  for (; stream < p.n_streams; stream += dq, t += dr) {
    if (t >= p.n_frames) {
      t -= p.n_frames;
      stream += 1;
      if (stream >= p.n_streams) break;
    }
    const long long fidx = (long long)stream * p.chunk_cap + t;
    float *rec = p.rec + fidx * kRecFloats;
    const int pitch_index = reinterpret_cast<const int *>(rec)[kRecPitchIndex];
#ifndef NS_FFT3
    const int res = 0;
#else
    const int res = task_parity;
    task_parity ^= 1;
#endif
    frame_spectra(g, T, s, p.hp + (long long)stream * p.hp_stride, t, pitch_index, res);
    {  // spectra -> workspace (K5 reads them back instead of redoing two FFTs)
      f4 *dst4 = reinterpret_cast<f4 *>(p.spec + fidx * (2 * kSpecStride));
      const f4 *src4 = reinterpret_cast<const f4 *>(s.spec[res]);  // X[482] | P[482]: 482 float4
      for (int k = g.tid; k < kSpecStride; k += kGroupThreads) dst4[k] = src4[k];
    }
    // band features: warp 0 alone, meeting on warp barriers, while the other warps finish the spectra store and
    // start on the next frame (nothing written below is touched again before several group barriers have passed,
    // and warp 0 joins the next frame's first barrier only after it is done here)
    if (g.warp == 0) {
      const int i = g.lane;
      if (i < kBands) {
        s.Exp[i] = s.Exp[i] / (float)sqrt(.001 + (double)(s.Ex[i] * s.Ep[i]));
        s.Ly[i] = (float)log10(1e-2 + (double)s.Ex[i]);
      }
      Simt::warp_sync();
      if (i == 0) {
        float logMax = -2.f, follow = -2.f, E = 0.f;
        for (int j = 0; j < kBands; j++) {
          float ly = s.Ly[j];
          ly = fmaxf(logMax - 7.f, fmaxf(follow - 1.5f, ly));
          logMax = fmaxf(logMax, ly);
          follow = fmaxf(follow - 1.5f, ly);
          s.Ly[j] = ly;
          E += s.Ex[j];
        }
        s.silence = (E < 0.04f) ? 1 : 0;
      }
      Simt::warp_sync();
      if (i < kBands) {
        float sum = 0.f;
        for (int j = 0; j < kBands; j++) sum += s.Ly[j] * T.dct(j * kBands + i);
        float c = sum * dct_scale;
        if (i == 0) c -= 12.f;
        if (i == 1) c -= 4.f;
        rec[kRecCeps + i] = c;
        rec[kRecExp + i] = s.Exp[i];
        rec[kRecEx + i] = s.Ex[i];
        rec[kRecEp + i] = s.Ep[i];
        if (p.dbg) {
          float *d = p.dbg + ((long long)stream * p.n_frames_call + p.frame0 + t) * kDbgFloats;
          d[kDbgEx + i] = s.Ex[i];
          d[kDbgEp + i] = s.Ep[i];
          d[kDbgExp + i] = s.Exp[i];
        }
      } else if (i < kBands + kDeltaCeps) {
        const int c6 = i - kBands;
        float sum = 0.f;
        for (int j = 0; j < kBands; j++) sum += s.Exp[j] * T.dct(j * kBands + c6);
        float c = sum * dct_scale;
        if (c6 == 0) c -= 1.3f;
        if (c6 == 1) c -= 0.9f;
        rec[kRecTail + c6] = c;
      } else if (i == kBands + kDeltaCeps) {
        rec[kRecTail + kDeltaCeps] = .01f * (float)(pitch_index - 300);
        reinterpret_cast<int *>(rec)[kRecSilence] = s.silence;
      }
      Simt::warp_sync();  // the next frame's band sums overwrite Ex / Ep / Exp: every lane is done reading first
    }
  }
}

// =================================================================================================
// activations (rnn.c tansig_approx / sigmoid_approx / relu)
// =================================================================================================
// tansig_approx without branches: |x| is clamped to 8, where the table ends at exactly 1.0 with zero
// slope, so x >= 8 (and NaN) give +-1 as upstream's early returns do; floor(.5 + 25|x|) is a truncation.
// The recurrent core is continuous in its inputs (no decision hangs on the last bit of an activation), so the
// multiply-adds are fused here: 12 instead of 16 instructions per activation on the kernel's busiest path.
NS_DEV float tansig_approx(const float *tab, float x) {
  const float ax = fminf(fabsf(x), 8.f);
  const int i = (int)fmaf(25.f, ax, .5f);
  const float d = fmaf(-.04f, (float)i, ax);
  float y = tab[i];
  const float dy = fmaf(-y, y, 1.f);
  y = fmaf(d * dy, fmaf(-y, d, 1.f), y);
  return copysignf(y, x);
}
NS_DEV float sigmoid_approx(const float *tab, float x) { return fmaf(.5f, tansig_approx(tab, .5f * x), .5f); }
NS_DEV float activate(const float *tab, int act, float x) {
  if (act == 1) return sigmoid_approx(tab, x);
  if (act == 0) return tansig_approx(tab, x);
  return x < 0.f ? 0.f : x;
}
// N activations of one kind: the (uniform) choice is made once, so the N table look-ups and polynomial chains
// interleave instead of running one after the other behind a branch each
template <int N>
NS_DEV void activate_n(const float *tab, int act, const float *x, float *y) {
  if (act == 1) {
#pragma unroll
    for (int j = 0; j < N; j++) y[j] = sigmoid_approx(tab, x[j]);
  } else if (act == 0) {
#pragma unroll
    for (int j = 0; j < N; j++) y[j] = tansig_approx(tab, x[j]);
  } else {
#pragma unroll
    for (int j = 0; j < N; j++) y[j] = x[j] < 0.f ? 0.f : x[j];
  }
}

// bf16 (round to nearest even) bit pattern of a finite float, and the hi + lo split of an activation
NS_DEV uint32_t bf16_rn_bits(float x) {
  const uint32_t u = f2u(x);
  return (u + 0x7FFFu + ((u >> 16) & 1u)) >> 16;
}
NS_DEV void bf16_split(float x, uint32_t &hi, uint32_t &lo) {
  hi = bf16_rn_bits(x);
  lo = bf16_rn_bits(x - u2f(hi << 16));
}
// two activations -> one word of the hi plane and one of the lo plane (v0 in the low halfword)
NS_DEV void bf16_split2(float v0, float v1, uint32_t &hi, uint32_t &lo) {
  hi = Simt::bf16x2_rn(v0, v1);
  lo = Simt::bf16x2_rn(v0 - u2f(hi << 16), v1 - u2f(hi & 0xFFFF0000u));
}
struct alignas(16) u4 {
  uint32_t x, y, z, w;
};
struct alignas(8) u2 {
  uint32_t x, y;
};

// =================================================================================================
// K3b: a13 cepstral ring, delta features, spectral variability.  One warp per stream walks the
// chunk's frames (the ring only advances on non-silent frames) and emits the 42 features already
// split into bf16 hi + lo and laid out as the recurrent core's A fragments (ns_common.h).
// =================================================================================================
constexpr int kFeatWarps = 4;
struct FeatSmem {
  float ring[kFeatWarps][kCepsMem][24];
  float dist[kFeatWarps][64];
  float cin[kFeatWarps][32];
  float feat[kFeatWarps][48];
};

NS_DEV void features_body(const Params &p, FeatSmem &sm) {
  const int lane = Simt::tid() & 31, warp = Simt::tid() >> 5;
  const int stream = Simt::cta() * kFeatWarps + warp;
  const int n_pad = (p.n_streams + kMmaStreams - 1) / kMmaStreams * kMmaStreams;
  if (stream >= n_pad) return;
  const int group = stream / kMmaStreams, row = stream % kMmaStreams;
  uint32_t *blk = p.featq + (long long)group * p.chunk_cap * kFeatBlockWords;
  // feature pair q = lane (features 2q, 2q+1) of this stream's row lands in this word of a plane
  const int q = lane;
  const int widx = ((q >> 3) * 32 + (row & 7) * 4 + (q & 3)) * 4 + (row >> 3) + 2 * ((q & 7) >> 2);
  if (stream >= p.n_streams) {  // padding rows of the last group: zero features, flagged silent
    for (int t = 0; t < p.n_frames; t++) {
      uint32_t *b = blk + (long long)t * kFeatBlockWords;
      if (lane < 24) {
        b[widx] = 0u;
        b[kFeatKt * kKtWords + widx] = 0u;
      }
      if (lane == 24) b[2 * kFeatKt * kKtWords + row] = 1u;
    }
    return;
  }
  float(*ring)[24] = sm.ring[warp];
  float *dist = sm.dist[warp], *cin = sm.cin[warp], *feat = sm.feat[warp];
  float *st = p.state + (long long)stream * kStateFloats;
  for (int i = lane; i < kCepsMem * kBands; i += 32) ring[i / kBands][i % kBands] = st[kStCeps + i];
  int memid = reinterpret_cast<const int *>(st)[kStMemId];
  for (int i = lane; i < 48; i += 32) feat[i] = 0.f;
  Simt::warp_sync();
  for (int it = lane; it < 64; it += 32) {  // pairwise cepstral distances of the ring
    const int a = it >> 3, b = it & 7;
    float d = 0.f;
    for (int k = 0; k < kBands; k++) {
      const float tt = ring[a][k] - ring[b][k];
      d += tt * tt;
    }
    dist[it] = d;
  }
  Simt::warp_sync();
  for (int t = 0; t < p.n_frames; t++) {
    const float *rec = p.rec + ((long long)stream * p.chunk_cap + t) * kRecFloats;
    const bool silent = reinterpret_cast<const int *>(rec)[kRecSilence] != 0;
    uint32_t *b = blk + (long long)t * kFeatBlockWords;
    if (!silent) {
      if (lane < kBands) {
        const float c = rec[kRecCeps + lane];
        ring[memid][lane] = c;
        cin[lane] = c;
      } else if (lane < 29) {
        cin[lane] = rec[kRecTail + lane - kBands];
      }
      Simt::warp_sync();
      if (lane < kCepsMem) {  // distances to the new ring row
        const int a = memid, bb = lane;
        float d = 0.f;
        for (int k = 0; k < kBands; k++) {
          const float tt = ring[a][k] - ring[bb][k];
          d += tt * tt;
        }
        dist[(a << 3) + bb] = d;
        dist[(bb << 3) + a] = d;
      }
      const int m0 = memid, m1 = (m0 + 7) & 7, m2 = (m0 + 6) & 7;
      for (int i = lane; i < 41; i += 32) {  // features[0..40]
        float v;
        if (i < kDeltaCeps) {
          v = ring[m0][i] + ring[m1][i] + ring[m2][i];
        } else if (i < kBands) {
          v = cin[i];
        } else if (i < kBands + kDeltaCeps) {
          const int j = i - kBands;
          v = ring[m0][j] - ring[m2][j];
        } else if (i < kBands + 2 * kDeltaCeps) {
          const int j = i - kBands - kDeltaCeps;
          v = ring[m0][j] - 2.f * ring[m1][j] + ring[m2][j];
        } else {
          v = cin[kBands + (i - kBands - 2 * kDeltaCeps)];
        }
        feat[i] = v;
      }
      Simt::warp_sync();
      float mind = 1e15f;  // spectral variability: sum over ring rows of the distance to the nearest other row
      if (lane < kCepsMem)
        for (int bb = 0; bb < kCepsMem; bb++)
          if (bb != lane) mind = fminf(mind, dist[(lane << 3) + bb]);
      float sv = 0.f;
      for (int a = 0; a < kCepsMem; a++) sv += Simt::shfl(mind, a);
      if (lane == 0) feat[41] = sv / kCepsMem - 2.1f;
      memid = (memid + 1) & 7;
      Simt::warp_sync();
    }
    if (lane < 24) {
      uint32_t h0 = 0u, l0 = 0u, h1 = 0u, l1 = 0u;
      if (!silent) {
        bf16_split(feat[2 * q], h0, l0);
        bf16_split(feat[2 * q + 1], h1, l1);
      }
      b[widx] = h0 | (h1 << 16);
      b[kFeatKt * kKtWords + widx] = l0 | (l1 << 16);
    }
    if (lane == 24) b[2 * kFeatKt * kKtWords + row] = silent ? 1u : 0u;
    if (p.dbg) {
      float *d = p.dbg + ((long long)stream * p.n_frames_call + p.frame0 + t) * kDbgFloats + kDbgFeatures;
      for (int i = lane; i < kFeatures; i += 32) d[i] = silent ? 0.f : feat[i];
    }
    Simt::warp_sync();
  }
  for (int i = lane; i < kCepsMem * kBands; i += 32) st[kStCeps + i] = ring[i / kBands][i % kBands];
  if (lane == 0) reinterpret_cast<int *>(st)[kStMemId] = memid;
}

// Voice gate (crispy_ns_controls): a frame is voiced if its returned VAD >= threshold; a voiced frame opens the gate
// for `hold` more frames; G = 1 while open, else the gate gain.  Serial in time per stream, so both recurrent cores
// run it where they write the VAD and hand G of the frame and of the one before to K5 in the record (K5's runs of a
// chunk are concurrent and could not carry it).  A zeroed state row is threshold 0: every frame voiced, G = 1.
struct GateState {
  float thr, gain, shut_gain;
  int hold, left, shut;
};
NS_DEV GateState gate_load(const float *st) {
  const int *sti = reinterpret_cast<const int *>(st);
  return GateState{st[kStCtlGateThr], st[kStCtlGateGain], st[kStGateShutGain], sti[kStCtlGateHold], sti[kStGateLeft],
                   sti[kStGateShut]};
}
NS_DEV void gate_step(GateState &q, float vad, float *rec) {
  bool open = true;
  if (!(vad < q.thr))  // vad >= thr; a NaN VAD (non-finite input) counts as voiced, so an unset gate never closes
    q.left = q.hold;
  else if (q.left > 0)
    q.left -= 1;
  else
    open = false;
  rec[kRecGatePrev] = q.shut ? q.shut_gain : 1.f;
  rec[kRecGate] = open ? 1.f : q.gain;
  q.shut = open ? 0 : 1;
  q.shut_gain = open ? 0.f : q.gain;
}
NS_DEV void gate_save(const GateState &q, float *st) {
  int *sti = reinterpret_cast<int *>(st);
  sti[kStGateLeft] = q.left;
  sti[kStGateShut] = q.shut;
  st[kStGateShutGain] = q.shut_gain;
}

// =================================================================================================
// K4: a14 the recurrent core on the tensor pipe, 16 streams per CTA, serial over the chunk's frames.
// All weights stay in shared memory as bf16 B fragments for the whole launch; every activation
// vector lives in shared memory as bf16 hi + lo A fragments; the GRU states, update gates and
// lastg stay in the registers of the lanes whose accumulator fragments own them.  Each of the
// eight matrix products of a frame is one pass of mma.sync.m16n8k16 over its k-tiles (twice: hi and
// lo plane) followed by an in-register epilogue (bias, activation, GRU algebra) that writes the
// next products' A fragments; one block barrier separates consecutive products.
// Neuron tile j (8 neurons) of a GRU belongs to warp j % 8 in both its z|r and candidate products.
// =================================================================================================
struct RnnSmem {
  uint32_t w[kMmaWords];
  uint32_t ahi[kKtResident * kKtWords];
  uint32_t alo[kKtResident * kKtWords];
  uint32_t fq[2][kFeatBlockWords];
  float bias[kMmaBias];
  float tansig[204];
  int act[kNumMmaJobs];
};
static_assert(sizeof(RnnSmem) <= 232448, "recurrent-core shared memory exceeds the 227 KB a CTA may use");

// product J for this warp's `nact` (<= NACC) n-tiles `tiles[]`: every k-tile of the job's compile-time
// list, hi and lo planes into separate accumulators (two independent MMA chains per n-tile).  All
// shared-memory offsets except the warp's tile bases are immediates.
template <int J, int NACC, int... KT>
NS_DEV void mma_run_list(const RnnSmem &r, const uint32_t *fcur, const int (&tiles)[NACC], int nact, int lane,
                         float (&acc)[NACC][2][4], KtList<KT...>) {
  constexpr int NNT = MmaShape<J>::nnt;
#pragma unroll
  for (int n = 0; n < NACC; n++)
#pragma unroll
    for (int e = 0; e < 4; e++) acc[n][0][e] = acc[n][1][e] = 0.f;
  const uint32_t *wb[NACC];
#pragma unroll
  for (int n = 0; n < NACC; n++) wb[n] = r.w + MmaOff<J>::w + tiles[n] * 64 + lane * 2;
  const uint32_t *res_hi = r.ahi + lane * 4, *res_lo = r.alo + lane * 4, *f_hi = fcur + lane * 4;
  int i = 0;
  auto step = [&](auto vt) {
    constexpr int v = decltype(vt)::value;
    const uint32_t *ph = (v < kKtResident) ? res_hi + v * kKtWords : f_hi + (v - kKtF) * kKtWords;
    const uint32_t *pl = (v < kKtResident) ? res_lo + v * kKtWords : f_hi + (kFeatKt + v - kKtF) * kKtWords;
    const u4 ah4 = *reinterpret_cast<const u4 *>(ph), al4 = *reinterpret_cast<const u4 *>(pl);
    const uint32_t ah[4] = {ah4.x, ah4.y, ah4.z, ah4.w}, al[4] = {al4.x, al4.y, al4.z, al4.w};
#pragma unroll
    for (int n = 0; n < NACC; n++) {
      if (n < nact) {
        const u2 b2 = *reinterpret_cast<const u2 *>(wb[n] + i * NNT * 64);
        const uint32_t b[2] = {b2.x, b2.y};
        Simt::mma_bf16_16816(acc[n][0], ah, b);
        Simt::mma_bf16_16816(acc[n][1], al, b);
      }
    }
    i++;
  };
  (step(IntC<KT>{}), ...);
}
template <int J, int NACC>
NS_DEV void mma_run(const RnnSmem &r, const uint32_t *fcur, const int (&tiles)[NACC], int nact, int lane,
                    float (&acc)[NACC][2][4]) {
  mma_run_list<J, NACC>(r, fcur, tiles, nact, lane, acc, typename MmaShape<J>::Kt{});
}

// S * (bias + sum) of the four accumulator elements of n-tile `tile`: rows lane/4 (e < 2) and
// lane/4 + 8, output columns tile*8 + 2*(lane%4) + (e & 1)
template <int J>
NS_DEV void mma_pre(const RnnSmem &r, const float (&acc)[2][4], int tile, int lane, float (&x)[4]) {
  const float *b = r.bias + MmaOff<J>::b + tile * 8 + 2 * (lane & 3);
  const float b0 = b[0], b1 = b[1];
  x[0] = ((acc[0][0] + acc[1][0]) + b0) * (1.f / 256);
  x[1] = ((acc[0][1] + acc[1][1]) + b1) * (1.f / 256);
  x[2] = ((acc[0][2] + acc[1][2]) + b0) * (1.f / 256);
  x[3] = ((acc[0][3] + acc[1][3]) + b1) * (1.f / 256);
}

// write this lane's four values (rows lane/4 and lane/4+8, inputs k0 + 2*(lane%4) + {0,1}) of the
// 8 inputs starting at resident position k0 (a multiple of 8) as hi/lo A fragments
NS_DEV void store_frag(RnnSmem &r, int k0, int lane, const float (&v)[4]) {
  uint32_t h0, l0, h1, l1;
  bf16_split2(v[0], v[1], h0, l0);
  bf16_split2(v[2], v[3], h1, l1);
  const int off = ((k0 >> 4) * 32 + lane) * 4 + ((k0 >> 3) & 1) * 2;
  *reinterpret_cast<u2 *>(r.ahi + off) = u2{h0, h1};
  *reinterpret_cast<u2 *>(r.alo + off) = u2{l0, l1};
}

// resident positions (k index = k-tile * 16 + kk) of the activation vectors
constexpr int kPosDense = kKtDV * 16, kPosVadH = kKtDV * 16 + 24, kPosDense2 = kKtDVR * 16,
              kPosVadR = kKtDVR * 16 + 24, kPosNoiseH = kKtNH * 16, kPosNoiseR = kKtNR * 16,
              kPosDenH = kKtDH * 16, kPosDenR = kKtDR * 16;

NS_DEV void rnn_body(const Params &p, RnnSmem &r) {
  const int tid = Simt::tid(), lane = tid & 31, warp = tid >> 5;
  const int NT = kMmaThreads;
  const int g = lane >> 2, c2 = 2 * (lane & 3);
  const int s0 = Simt::cta() * kMmaStreams;
  const int srow[2] = {s0 + g, s0 + g + 8};
  const bool live[2] = {srow[0] < p.n_streams, srow[1] < p.n_streams};
  {  // weights, biases, tables -> shared memory; activation fragments cleared
    const RnnHeader &H = *p.rnn_hdr;
    const u4 *src = reinterpret_cast<const u4 *>(p.rnn_words);
    u4 *dst = reinterpret_cast<u4 *>(r.w);
    for (int i = tid; i < kMmaWords / 4; i += NT) dst[i] = src[i];
    for (int i = tid; i < kMmaBias; i += NT) r.bias[i] = p.rnn_bias[i];
    for (int i = tid; i < 204; i += NT) r.tansig[i] = p.tables->tansig[i];
    if (tid < kNumMmaJobs) r.act[tid] = H.activation[tid];
    for (int i = tid; i < kKtResident * kKtWords; i += NT) r.ahi[i] = r.alo[i] = 0u;
  }
  const uint32_t *fq_src = p.featq + (long long)Simt::cta() * p.chunk_cap * kFeatBlockWords;
  auto fetch = [&](int t) {  // feature block of frame t -> fq[t & 1]
    if (tid < kFeatBlockWords / 4) Simt::cp_async16(&r.fq[t & 1][tid * 4], fq_src + (long long)t * kFeatBlockWords + tid * 4);
    Simt::cp_async_commit();
  };
  if (p.n_frames > 0) fetch(0);
  // recurrent state -> registers of the owning lanes.  hv: vad (warps 0-2), hn: noise (warps 0-5),
  // hd[0]: denoise tile `warp`, hd[1]: denoise tile warp + 8 (warps 0-3); lastg: warps 0-2
  float hv[4], hn[4], hd[2][4], lastg[4];
  auto load4 = [&](float (&h)[4], int st_off, int n0, int n_max) {
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int n = n0 + (e & 1);
      h[e] = (live[e >> 1] && n < n_max) ? p.state[(long long)srow[e >> 1] * kStateFloats + st_off + n] : 0.f;
    }
  };
  auto save4 = [&](const float (&h)[4], int st_off, int n0, int n_max) {
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int n = n0 + (e & 1);
      if (live[e >> 1] && n < n_max) p.state[(long long)srow[e >> 1] * kStateFloats + st_off + n] = h[e];
    }
  };
  load4(hv, kStHVad, warp * 8 + c2, warp < 3 ? 24 : 0);
  load4(hn, kStHNoise, warp * 8 + c2, warp < 6 ? 48 : 0);
  load4(hd[0], kStHDen, warp * 8 + c2, 96);
  load4(hd[1], kStHDen, (warp + 8) * 8 + c2, warp < 4 ? 96 : 0);
  load4(lastg, kStLastG, warp * 8 + c2, warp < 3 ? kBands : 0);
  // the voice gate runs on the lanes that write the VAD (warp 7, lane % 4 == 0: streams srow[0], srow[1])
  const bool gate_lane = warp == 7 && (lane & 3) == 0;
  GateState gate[2] = {};
#pragma unroll
  for (int h = 0; h < 2; h++)
    if (gate_lane && live[h]) gate[h] = gate_load(p.state + (long long)srow[h] * kStateFloats);
  Simt::cta_sync();  // the fragments were cleared
  if (warp < 3) store_frag(r, kPosVadH + warp * 8, lane, hv);
  if (warp < 6) store_frag(r, kPosNoiseH + warp * 8, lane, hn);
  store_frag(r, kPosDenH + warp * 8, lane, hd[0]);
  if (warp < 4) store_frag(r, kPosDenH + (warp + 8) * 8, lane, hd[1]);
  Simt::cp_async_wait<0>();
  Simt::cta_sync();
  const float *tab = r.tansig;
  const int act_dense = r.act[kJDense], act_vad = r.act[kJVadC], act_noise = r.act[kJNoiseC], act_den = r.act[kJDenC],
            act_out = r.act[kJOut], act_vadout = r.act[kJVadOut];
  // GRU update of the four (row, neuron) elements this lane owns
  auto gru_update = [&](float (&h)[4], const float (&z)[4], const float (&x)[4], int act, const bool (&sil)[2]) {
    float cnd[4];
    activate_n<4>(tab, act, x, cnd);
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const float hnew = z[e] * h[e] + (1.f - z[e]) * cnd[e];
      if (!sil[e >> 1]) h[e] = hnew;
    }
  };
  for (int t = 0; t < p.n_frames; t++) {
    const uint32_t *fcur = r.fq[t & 1];
    if (t + 1 < p.n_frames) fetch(t + 1);
    const u4 *flags4 = reinterpret_cast<const u4 *>(fcur + 2 * kFeatKt * kKtWords);
    uint32_t all_silent = 1u;
#pragma unroll
    for (int i = 0; i < kMmaStreams / 4; i++) {
      const u4 f = flags4[i];
      all_silent &= f.x & f.y & f.z & f.w;
    }
    const uint32_t *flags = fcur + 2 * kFeatKt * kKtWords;
    const bool sil[2] = {flags[g] != 0u, flags[g + 8] != 0u};
    float vad[2] = {0.f, 0.f};
    float gout[4] = {0.f, 0.f, 0.f, 0.f}, graw[4] = {0.f, 0.f, 0.f, 0.f};
    if (!all_silent) {
      float x[4], z[2][4];
      if (warp < 3) {  // input_dense: features -> dense (both copies)
        float acc[1][2][4];
        const int tiles[1] = {warp};
        mma_run<kJDense, 1>(r, fcur, tiles, 1, lane, acc);
        mma_pre<kJDense>(r, acc[0], warp, lane, x);
        float y[4];
        activate_n<4>(tab, act_dense, x, y);
        store_frag(r, kPosDense + warp * 8, lane, y);
        store_frag(r, kPosDense2 + warp * 8, lane, y);
      }
      Simt::cta_sync();
      if (warp < 3) {  // vad_gru z | r
        float acc[2][2][4];
        const int tiles[2] = {warp, 3 + warp};
        mma_run<kJVadZR, 2>(r, fcur, tiles, 2, lane, acc);
        float rh[4];
        mma_pre<kJVadZR>(r, acc[0], tiles[0], lane, x);
#pragma unroll
        for (int e = 0; e < 4; e++) z[0][e] = sigmoid_approx(tab, x[e]);
        mma_pre<kJVadZR>(r, acc[1], tiles[1], lane, x);
#pragma unroll
        for (int e = 0; e < 4; e++) rh[e] = hv[e] * sigmoid_approx(tab, x[e]);
        store_frag(r, kPosVadR + warp * 8, lane, rh);
      }
      Simt::cta_sync();
      if (warp < 3) {  // vad_gru candidate
        float acc[1][2][4];
        const int tiles[1] = {warp};
        mma_run<kJVadC, 1>(r, fcur, tiles, 1, lane, acc);
        mma_pre<kJVadC>(r, acc[0], warp, lane, x);
        gru_update(hv, z[0], x, act_vad, sil);
        store_frag(r, kPosVadH + warp * 8, lane, hv);
      }
      Simt::cta_sync();
      if (warp < 6) {  // noise_gru z | r (warps 0-5); vad_output on the settled vad state (warp 7)
        float acc[2][2][4];
        const int tiles[2] = {warp, 6 + warp};
        mma_run<kJNoiseZR, 2>(r, fcur, tiles, 2, lane, acc);
        float rh[4];
        mma_pre<kJNoiseZR>(r, acc[0], tiles[0], lane, x);
#pragma unroll
        for (int e = 0; e < 4; e++) z[0][e] = sigmoid_approx(tab, x[e]);
        mma_pre<kJNoiseZR>(r, acc[1], tiles[1], lane, x);
#pragma unroll
        for (int e = 0; e < 4; e++) rh[e] = hn[e] * sigmoid_approx(tab, x[e]);
        store_frag(r, kPosNoiseR + warp * 8, lane, rh);
      } else if (warp == 7) {
        float acc[1][2][4];
        const int tiles[1] = {0};
        mma_run<kJVadOut, 1>(r, fcur, tiles, 1, lane, acc);
        mma_pre<kJVadOut>(r, acc[0], 0, lane, x);  // column 0 lives in the lanes with lane % 4 == 0
        vad[0] = activate(tab, act_vadout, x[0]);
        vad[1] = activate(tab, act_vadout, x[2]);
      }
      Simt::cta_sync();
      if (warp < 6) {  // noise_gru candidate
        float acc[1][2][4];
        const int tiles[1] = {warp};
        mma_run<kJNoiseC, 1>(r, fcur, tiles, 1, lane, acc);
        mma_pre<kJNoiseC>(r, acc[0], warp, lane, x);
        gru_update(hn, z[0], x, act_noise, sil);
        store_frag(r, kPosNoiseH + warp * 8, lane, hn);
      }
      Simt::cta_sync();
      const int nown = warp < 4 ? 2 : 1;  // denoise_gru: warp w owns neuron tiles w and (w < 4) w + 8
      {
        float acc[4][2][4];
        const int tiles[4] = {warp, 12 + warp, warp + 8, 12 + warp + 8};
        mma_run<kJDenZR, 4>(r, fcur, tiles, 2 * nown, lane, acc);
#pragma unroll
        for (int o = 0; o < 2; o++) {
          if (o < nown) {
            float rh[4];
            mma_pre<kJDenZR>(r, acc[2 * o], tiles[2 * o], lane, x);
#pragma unroll
            for (int e = 0; e < 4; e++) z[o][e] = sigmoid_approx(tab, x[e]);
            mma_pre<kJDenZR>(r, acc[2 * o + 1], tiles[2 * o + 1], lane, x);
#pragma unroll
            for (int e = 0; e < 4; e++) rh[e] = hd[o][e] * sigmoid_approx(tab, x[e]);
            store_frag(r, kPosDenR + tiles[2 * o] * 8, lane, rh);
          }
        }
      }
      Simt::cta_sync();
      {
        float acc[2][2][4];
        const int tiles[2] = {warp, warp + 8};
        mma_run<kJDenC, 2>(r, fcur, tiles, nown, lane, acc);
#pragma unroll
        for (int o = 0; o < 2; o++) {
          if (o < nown) {
            mma_pre<kJDenC>(r, acc[o], tiles[o], lane, x);
            gru_update(hd[o], z[o], x, act_den, sil);
            store_frag(r, kPosDenH + tiles[o] * 8, lane, hd[o]);
          }
        }
      }
      Simt::cta_sync();
      if (warp < 3) {  // denoise_output -> band gains; g = max(g, 0.6 lastg)
        float acc[1][2][4];
        const int tiles[1] = {warp};
        mma_run<kJOut, 1>(r, fcur, tiles, 1, lane, acc);
        mma_pre<kJOut>(r, acc[0], warp, lane, x);
        float gact[4];
        activate_n<4>(tab, act_out, x, gact);
#pragma unroll
        for (int e = 0; e < 4; e++) {
          if (!sil[e >> 1]) {
            graw[e] = gact[e];
            gout[e] = fmaxf(graw[e], .6f * lastg[e]);
            lastg[e] = gout[e];
          }
        }
      }
    }
    if (warp < 3) {  // band gains of this frame -> record (zeros on silent frames)
      const int band = warp * 8 + c2;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        if (live[h] && band < kBands) {
          float *rec = p.rec + ((long long)srow[h] * p.chunk_cap + t) * kRecFloats;
          *reinterpret_cast<cf *>(rec + kRecGRaw + band) = cf{graw[2 * h], graw[2 * h + 1]};
          *reinterpret_cast<cf *>(rec + kRecG + band) = cf{gout[2 * h], gout[2 * h + 1]};
        }
      }
    } else if (gate_lane) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        if (live[h]) {
          const float v = sil[h] ? 0.f : vad[h];
          float *rec = p.rec + ((long long)srow[h] * p.chunk_cap + t) * kRecFloats;
          rec[kRecVad] = v;
          gate_step(gate[h], v, rec);
          if (p.vad) p.vad[(long long)srow[h] * p.vad_stride + p.frame0 + t] = v;
        }
      }
    }
    Simt::cp_async_wait<0>();
    Simt::cta_sync();
  }
  save4(hv, kStHVad, warp * 8 + c2, warp < 3 ? 24 : 0);
  save4(hn, kStHNoise, warp * 8 + c2, warp < 6 ? 48 : 0);
  save4(hd[0], kStHDen, warp * 8 + c2, 96);
  save4(hd[1], kStHDen, (warp + 8) * 8 + c2, warp < 4 ? 96 : 0);
  save4(lastg, kStLastG, warp * 8 + c2, warp < 3 ? kBands : 0);
#pragma unroll
  for (int h = 0; h < 2; h++)
    if (gate_lane && live[h]) gate_save(gate[h], p.state + (long long)srow[h] * kStateFloats);
}

// =================================================================================================
// K5: a15 pitch filter + gain interpolation, a16 synthesis; one 128-thread group per stream walks
// the chunk's frames carrying synthesis_mem in shared memory
// =================================================================================================
// min_gain (crispy_ns_controls): floor on the applied band gains; lastg and the pitch filter keep the unfloored ones
NS_DEV void pitch_filter_and_gains(const Grp &g, const Tab &T, SpecSmem &s, cf *X, const cf *P, const float *rc, float min_gain) {
  if (g.tid < kBands) {
    const int i = g.tid;
    const float e = rc[kRecExp + i], gi = rc[kRecGRaw + i];
    float r;
    if (e > gi)
      r = 1.f;
    else
      r = (e * e) * (1.f - gi * gi) / (.001f + (gi * gi) * (1.f - e * e));
    r = sqrtf(fminf(1.f, fmaxf(0.f, r)));
    r *= (float)sqrt((double)rc[kRecEx + i] / (1e-8 + (double)rc[kRecEp + i]));
    s.r[i] = r;
  }
  gsync(g);
  // slot pass (four bins of one band interval per thread): X += rf P, and the filtered spectrum's band
  // energy partials in the same sweep
  if (g.tid < kSlots) {
    const int k0 = 4 * g.tid, b = T.bin_band(k0);
    const f4 fr4 = T.bin_frac4(k0);
    const float fr[4] = {fr4.x, fr4.y, fr4.z, fr4.w};
    const float r0 = s.r[b], r1 = s.r[b + 1];
    const bool sw = (g.tid & 4) != 0;
    f4 xq[2], pq[2];
    ld_slot(X + k0, sw, xq[0], xq[1]);
    ld_slot(P + k0, sw, pq[0], pq[1]);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      f4 x = xq[h];
      const f4 pp = pq[h];
      const float rfa = (1.f - fr[2 * h]) * r0 + fr[2 * h] * r1, rfb = (1.f - fr[2 * h + 1]) * r0 + fr[2 * h + 1] * r1;
      x.x += rfa * pp.x;
      x.y += rfa * pp.y;
      x.z += rfb * pp.z;
      x.w += rfb * pp.w;
      xq[h] = x;
      const float va = fmaf(x.x, x.x, x.y * x.y), vb = fmaf(x.z, x.z, x.w * x.w);
      s0 += va;
      s1 = fmaf(fr[2 * h], va, s1);
      s0 += vb;
      s1 = fmaf(fr[2 * h + 1], vb, s1);
    }
    st_slot(X + k0, sw, xq[0], xq[1]);
    s.part[g.tid] = s0 - s1;
    s.part[kPartStride + g.tid] = s1;
  }
  gsync(g);
  {
    float e[1];
    band_reduce<1>(g, T, s.part, e);
    if (g.tid < 4 * kBands && (g.tid & 3) == 0) {
      const int i = g.tid >> 2;
      s.nrm[i] = (float)sqrt((double)rc[kRecEx + i] / (1e-8 + (double)e[0]));
    }
  }
  gsync(g);
  if (g.tid < kSlots) {
    const int k0 = 4 * g.tid, b = T.bin_band(k0);
    const f4 fr4 = T.bin_frac4(k0);
    const float fr[4] = {fr4.x, fr4.y, fr4.z, fr4.w};
    const float n0 = s.nrm[b], n1 = s.nrm[b + 1];
    float g0 = rc[kRecG + b], g1 = rc[kRecG + b + 1];
    if (min_gain > 0.f) {  // uniform per stream: the default path skips it
      g0 = fmaxf(g0, min_gain);
      g1 = fmaxf(g1, min_gain);
    }
    const bool sw = (g.tid & 4) != 0;
    f4 xq[2];
    ld_slot(X + k0, sw, xq[0], xq[1]);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      f4 x = xq[h];
      const float fa = fr[2 * h], fb = fr[2 * h + 1];
      const float nfa = (1.f - fa) * n0 + fa * n1, gfa = (1.f - fa) * g0 + fa * g1;
      const float nfb = (1.f - fb) * n0 + fb * n1, gfb = (1.f - fb) * g0 + fb * g1;
      x.x = (x.x * nfa) * gfa;
      x.y = (x.y * nfa) * gfa;
      x.z = (x.z * nfb) * gfb;
      x.w = (x.w * nfb) * gfb;
      xq[h] = x;
    }
    st_slot(X + k0, sw, xq[0], xq[1]);
  } else {
    for (int k = 400 + (g.tid - kSlots); k < kFreq; k += kGroupThreads - kSlots) X[k] = cf{0.f, 0.f};
  }
  gsync(g);
}

// a16 tail + the fused output conversions.  Thread i handles samples 4i..4i+3 (one 16-byte shared-memory
// access per operand); the caller's buffers are written with 16 / 8-byte stores when their base and
// stride allow it (any torch tensor does), else sample by sample.
NS_DEV float out_unit(const Params &p, float o) { return fminf(1.f, fmaxf(-1.f, o / 32768.0f)) * p.volume; }
NS_DEV int16_t out_i16(float o) {
  float v = rintf(o);
  v = fminf(32767.f, fmaxf(-32768.f, v));
  return (int16_t)(int)v;
}
NS_DEV int16_t out_mix(const Params &p, float o, float app) {
  float mixed = out_unit(p, o) + app;
  mixed = fminf(1.f, fmaxf(-1.f, mixed));
  return (int16_t)(int)(mixed * 32767.0f);  // truncation toward zero, as Rust `as i16`
}
NS_DEV uint32_t pack16(int16_t lo, int16_t hi) { return (uint32_t)(uint16_t)lo | ((uint32_t)(uint16_t)hi << 16); }

NS_DEV void store_frame(const Grp &g, const Tab &T, const Params &p, SpecSmem &s, const cf *X, const float *rc, int stream,
                        int t_call) {
  // X holds z[m] with x[2m] = z.x, x[2m+1] = -z.y.  out[i] = x[i] w[i] + synth[i]; synth = x[480+i] w[479-i]
  const int slot = t_call + p.out_frame_offset;
  const float *zb = reinterpret_cast<const float *>(X);
  if (g.tid >= kFrame / 4) return;
  const int i = 4 * g.tid;
  const f4 za = ld4(zb + i), zc = ld4(zb + kFrame + i), wa = T.win4(i), wr = T.win4(kFrame - 4 - i);
  const f4 sy = ld4(s.synth + i);
  float o[4] = {za.x * wa.x + sy.x, (-za.y) * wa.y + sy.y, za.z * wa.z + sy.z, (-za.w) * wa.w + sy.w};
  *reinterpret_cast<f4 *>(s.synth + i) = f4{zc.x * wr.w, (-zc.y) * wr.z, zc.z * wr.y, (-zc.w) * wr.x};
  if (slot < 0) return;
  const float gp = rc[kRecGatePrev], gc = rc[kRecGate];
  if (gp != 1.f || gc != 1.f) {  // the voice gate's ramp from G of the previous frame to G of this one; uniform per frame
#pragma unroll
    for (int u = 0; u < 4; u++) o[u] = o[u] * (gp + (gc - gp) * ((float)(i + u + 1) / 480.0f));
  }
  const long long o_off = (long long)stream * p.out_stride + (long long)slot * kFrame + i;
  const bool vec_out = ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0) && ((p.out_stride & 3) == 0);
  if (p.flags & kFlagMixStereoI16) {
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.app) {
      const float *ap = p.app + (long long)stream * p.app_stride + (long long)slot * kFrame + i;
      if (((reinterpret_cast<uintptr_t>(p.app) & 15) == 0) && ((p.app_stride & 3) == 0)) {
        const f4 a4 = ld4(ap);
        a[0] = a4.x, a[1] = a4.y, a[2] = a4.z, a[3] = a4.w;
      } else {
#pragma unroll
        for (int u = 0; u < 4; u++) a[u] = ap[u];
      }
    }
    int16_t q[4];
#pragma unroll
    for (int u = 0; u < 4; u++) q[u] = out_mix(p, o[u], a[u]);
    int16_t *dst = reinterpret_cast<int16_t *>(p.out) + 2 * o_off;
    if (vec_out) {
      *reinterpret_cast<u4 *>(dst) = u4{pack16(q[0], q[0]), pack16(q[1], q[1]), pack16(q[2], q[2]), pack16(q[3], q[3])};
    } else {
#pragma unroll
      for (int u = 0; u < 4; u++) dst[2 * u] = dst[2 * u + 1] = q[u];
    }
  } else if (p.flags & kFlagOutI16) {
    int16_t *dst = reinterpret_cast<int16_t *>(p.out) + o_off;
    if (vec_out) {
      *reinterpret_cast<u2 *>(dst) = u2{pack16(out_i16(o[0]), out_i16(o[1])), pack16(out_i16(o[2]), out_i16(o[3]))};
    } else {
#pragma unroll
      for (int u = 0; u < 4; u++) dst[u] = out_i16(o[u]);
    }
  } else {
    float *dst = reinterpret_cast<float *>(p.out) + o_off;
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = (p.flags & kFlagUnitScale) ? out_unit(p, o[u]) : o[u];
    if (vec_out) {
      *reinterpret_cast<f4 *>(dst) = f4{v[0], v[1], v[2], v[3]};
    } else {
#pragma unroll
      for (int u = 0; u < 4; u++) dst[u] = v[u];
    }
  }
}

// One task = p.syn_run consecutive frames of one stream.  A run that does not start the chunk first
// re-synthesises the frame before it to recover synthesis_mem (the overlap-add halo); the result does not
// depend on the run length.  pick_syn_run (host): fewest task-loop rounds x frames per task, halo included.
inline int pick_syn_run(int n_streams, int n_frames, int resident_ctas) {
  int best = n_frames < 1 ? 1 : n_frames;
  long long best_cost = -1;
  for (int run = 1; run <= n_frames; run++) {
    const long long tasks = (long long)n_streams * ((n_frames + run - 1) / run);
    const long long rounds = (tasks + resident_ctas - 1) / resident_ctas;
    const long long cost = rounds * (run + (run < n_frames ? 1 : 0));
    if (best_cost < 0 || cost < best_cost || (cost == best_cost && run > best)) {
      best_cost = cost;
      best = run;
    }
  }
  return best;
}

// The kernel forms a model's numerics select (crispy_ns_model_set_numerics; host only).  K1 is instantiated per sum
// order (pitch_body<R, NT, SP>), K0's single recursion warp per biquad arithmetic (highpass_body<F32>).  K0's
// time-parallel form speculates the f64 expression only, so under kBiquadF32 the single recursion warp runs.
constexpr uint32_t kSumMask = 3u, kBiquadF32 = 1u << 4;  // CRISPY_NS_SUM_MASK, CRISPY_NS_BIQUAD_F32
#ifndef NS_PITCH_V7
constexpr int kSumOrders = 3;
#else
constexpr int kSumOrders = 1;  // ns_pitch7.cuh sums in the sequential order only
#endif
inline bool numerics_valid(uint32_t numerics) {  // known bits, and sum order 3 is none
  return !(numerics & ~(kSumMask | kBiquadF32)) && (numerics & kSumMask) != kSumMask;
}
inline bool biquad_f32(uint32_t numerics) { return (numerics & kBiquadF32) != 0; }
inline bool hp_par_form(uint32_t numerics, bool par) { return par && !biquad_f32(numerics); }
// f(std::integral_constant<int, SP>()) for the sum order of numerics; orders this build does not have run as 0
template <class F>
inline auto with_sum_order(uint32_t numerics, F &&f) {
  if constexpr (kSumOrders > 1) {
    if ((numerics & kSumMask) == 1) return f(std::integral_constant<int, 1>());
    if ((numerics & kSumMask) == 2) return f(std::integral_constant<int, 2>());
  }
  return f(std::integral_constant<int, 0>());
}

// one thread stages a frame's spectra (X | P, 7,712 B) and record (592 B) into buffer b: two bulk copies on s.mbar
NS_DEV void synth_stage(const Grp &g, const Params &p, SpecSmem &s, int stream, int t, int b) {
  static_assert((2 * kSpecStride * sizeof(cf)) % 16 == 0 && (kRecFloats * sizeof(float)) % 16 == 0, "bulk copy sizes");
  if (g.tid == 0) {
    const long long fidx = (long long)stream * p.chunk_cap + t;
    Simt::fence_async_proxy();
    Simt::mbar_expect_tx(&s.mbar, (unsigned)(2 * kSpecStride * sizeof(cf) + kRecFloats * sizeof(float)));
    Simt::bulk_g2s(s.spec[b], p.spec + fidx * (2 * kSpecStride), (unsigned)(2 * kSpecStride * sizeof(cf)), &s.mbar);
    Simt::bulk_g2s(s.rec_s[b], p.rec + fidx * kRecFloats, (unsigned)(kRecFloats * sizeof(float)), &s.mbar);
  }
}

NS_DEV void synth_frame(const Grp &g, const Tab &T, const Params &p, SpecSmem &s, int stream, int t, bool halo, int b,
                        float min_gain) {
  cf *X = s.spec[b], *P = X + kSpecStride;
  const float *rc = s.rec_s[b];
  const bool silent = reinterpret_cast<const int *>(rc)[kRecSilence] != 0;
  if (!silent) pitch_filter_and_gains(g, T, s, X, P, rc, min_gain);
  if (p.dbg && !halo) {
    float *d = p.dbg + ((long long)stream * p.n_frames_call + p.frame0 + t) * kDbgFloats;
    if (g.tid < kBands) d[kDbgGains + g.tid] = rc[kRecG + g.tid];
    if (g.tid < kBands) d[kDbgGRaw + g.tid] = rc[kRecGRaw + g.tid];
    if (g.tid == 0) {
      d[kDbgPitchGain] = rc[kRecPitchGain];
      d[kDbgVad] = rc[kRecVad];
      d[kDbgPitchIndex] = (float)reinterpret_cast<const int *>(rc)[kRecPitchIndex];
      d[kDbgSilence] = silent ? 1.f : 0.f;
    }
  }
  irfft960_inplace(g, T, X, P);  // P is dead after the pitch filter
  if (halo) {
    const float *zb = reinterpret_cast<const float *>(X);
    for (int i = g.tid; i < kFrame; i += kGroupThreads) {
      const float x1 = (i & 1) ? -zb[kFrame + i] : zb[kFrame + i];
      s.synth[i] = x1 * T.win(kFrame - 1 - i);
    }
  } else {
    store_frame(g, T, p, s, X, rc, stream, p.frame0 + t);
  }
  gsync(g);
}

NS_DEV void synthesis_body(const Params &p, SpecSmem &s) {
  Grp g;
  g.tid = Simt::tid();
  g.lane = g.tid & 31;
  g.warp = g.tid >> 5;
  g.bar = 1;
  load_twiddles(p, s.tw, g.tid, kGroupThreads);
  if (g.tid == 0) Simt::mbar_init(&s.mbar, 1);
  Simt::cta_sync();
  const Tab T{&s.tw, p.tables};
  unsigned parity = 0;
  const int run = p.syn_run;
  const int runs = (p.n_frames + run - 1) / run;
  const int n_tasks = p.n_streams * runs;  // < 2^31: checked on the host
  for (int task = Simt::cta(); task < n_tasks; task += Simt::n_ctas()) {
    const int stream = task / runs, t0 = (task - stream * runs) * run;
    const int t1 = (t0 + run < p.n_frames) ? t0 + run : p.n_frames;
    float *st = p.state + (long long)stream * kStateFloats;
    const float min_gain = st[kStCtlMinGain];  // set between calls only: no kernel of this call writes it
    // a run that does not start the chunk re-synthesises the frame before it (the overlap-add halo)
    const int first = (t0 == 0) ? 0 : t0 - 1;
    synth_stage(g, p, s, stream, first, 0);
    if (t0 == 0)
      for (int i = g.tid; i < kFrame; i += kGroupThreads) s.synth[i] = st[kStSynth + p.synth_sel * kFrame + i];
    for (int t = first; t < t1; t++) {
      const int b = (t - first) & 1;
      Simt::mbar_wait(&s.mbar, parity);
      parity ^= 1u;
      gsync(g);  // frame t has landed in buffer b; everyone is done with buffer b ^ 1
      if (t + 1 < t1) synth_stage(g, p, s, stream, t + 1, b ^ 1);  // in flight while frame t is worked on
      synth_frame(g, T, p, s, stream, t, t < t0, b, min_gain);
    }
    if (t1 == p.n_frames) {
      for (int i = g.tid; i < kFrame; i += kGroupThreads) st[kStSynth + (1 - p.synth_sel) * kFrame + i] = s.synth[i];
      if (g.tid == 0) reinterpret_cast<int *>(st)[kStFrameCount] += p.n_frames;
    }
    gsync(g);
  }
}

}  // namespace ns
