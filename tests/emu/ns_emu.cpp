// ns_emu.cpp -- host SIMT emulation of the pipeline kernels (TEST PLUMBING, never shipped).
// Compiles crispy_b200/csrc/ns_pipe.cuh with NS_HOST_EMU: one OS thread per CUDA thread,
// pthread barriers for bar.sync / __syncthreads, a per-warp exchange buffer for shuffles.
// Lets `pytest -m "not gpu"` run the kernels' exact control flow against the oracle.
// Build with -ffp-contract=off: the kernels' exactness contract (ns_pipe.cuh) relies on it.
#define NS_HOST_EMU 1
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <functional>
#include <string>
#include <vector>

#include "../../crispy_b200/csrc/ns_host.h"
#include "../../crispy_b200/csrc/ns_pipe.cuh"
#include "../../crispy_b200/csrc/ns_pitch7.cuh"

namespace ns {
thread_local EmuThread g_emu;
}

namespace {
struct ThreadArg {
  ns::EmuCta *cta;
  int tid;
  const std::function<void()> *body;
};
void *thread_main(void *a) {
  ThreadArg *ta = (ThreadArg *)a;
  ns::g_emu.cta = ta->cta;
  ns::g_emu.tid = ta->tid;
  (*ta->body)();
  return nullptr;
}

// run `n_ctas` CTAs of `n_threads` threads one after another; `body(smem)` is the kernel body
int launch(int n_ctas, int n_threads, size_t smem_bytes, const std::function<void(void *)> &kernel) {
  std::vector<unsigned char> smem(smem_bytes + 64);
  void *sm = (void *)(((uintptr_t)smem.data() + 63) & ~(uintptr_t)63);
  for (int c = 0; c < n_ctas; c++) {
    ns::EmuCta cta;
    std::vector<ns::EmuWarp> warps((n_threads + 31) / 32);
    cta.warps = warps.data();
    cta.cta_index = c;
    cta.n_ctas = n_ctas;
    pthread_barrier_init(&cta.cta_bar, nullptr, n_threads);
    for (int i = 0; i < 16; i++) pthread_barrier_init(&cta.group_bar[i], nullptr, ns::kGroupThreads);
    for (size_t w = 0; w < warps.size(); w++) {
      const int in_warp = (n_threads - (int)w * 32) < 32 ? (n_threads - (int)w * 32) : 32;
      pthread_barrier_init(&warps[w].bar, nullptr, in_warp);
    }
    memset(sm, 0xCD, smem_bytes);  // shared memory is not zeroed on a GPU either
    const std::function<void()> body = [&]() { kernel(sm); };
    std::vector<pthread_t> th(n_threads);
    std::vector<ThreadArg> args(n_threads);
    pthread_attr_t attr;
    pthread_attr_init(&attr);
    pthread_attr_setstacksize(&attr, 256 * 1024);
    for (int t = 0; t < n_threads; t++) {
      args[t] = ThreadArg{&cta, t, &body};
      if (pthread_create(&th[t], &attr, thread_main, &args[t]) != 0) return -2;
    }
    for (int t = 0; t < n_threads; t++) pthread_join(th[t], nullptr);
    pthread_attr_destroy(&attr);
    pthread_barrier_destroy(&cta.cta_bar);
    for (int i = 0; i < 16; i++) pthread_barrier_destroy(&cta.group_bar[i]);
    for (auto &w : warps) pthread_barrier_destroy(&w.bar);
  }
  return 0;
}

constexpr int kPitchRun = 8;
#ifndef NS_PITCH_V7
constexpr int kPitchThreads = 352;  // as the device build: warp f < 8 replays frame f's coarse insertion, chain warps follow
using PitchShared = ns::PitchSmem<kPitchRun>;
#else
constexpr int kPitchThreads = ns::kP7Threads;  // warp w < 8 owns frame w, three chain warps follow
using PitchShared = ns::PitchSmem7<kPitchRun>;
#endif
constexpr int kScanWarps = 1;
}  // namespace

extern "C" {
int ns_emu_state_floats(void) { return ns::kStateFloats; }
int ns_emu_dbg_floats(void) { return ns::kDbgFloats; }
int ns_emu_state_hp_offset(void) { return ns::kStHp; }
int ns_emu_hp_spec(void) { return NS_HP_PAR; }
// groups the speculative biquad recomputed with upstream's f64 expression since the last call (K0, ns_pipe.cuh)
long long ns_emu_hp_respeculated(void) { return __atomic_exchange_n(&ns::g_hp_respeculated, 0, __ATOMIC_RELAXED); }

// in/out/app use the same strides the device path uses; state is in/out ([n_streams][kStateFloats]).
// The call is cut into chunks of `chunk_cap` frames exactly as libcrispy_ns.so does.  numerics: the model's setting
// (crispy_ns_model_set_numerics); -3 for one the library refuses, a nonzero sum order in the NS_PITCH_V7 build included.
int ns_emu_process(const void *model_blob, size_t model_len, const void *in, void *out, float *vad,
                   const float *app, float *state, float *dbg, int n_streams, int n_frames,
                   long long in_stride, long long out_stride, long long app_stride, int chunk_cap,
                   unsigned flags, float volume, int out_frame_offset, unsigned numerics) {
  if (!ns::numerics_valid(numerics) || (int)(numerics & ns::kSumMask) >= ns::kSumOrders) return -3;
  ns::Model m;
  std::string err;
  if (!ns::model_from_bytes(m, model_blob, model_len, err)) {
    fprintf(stderr, "ns_emu: %s\n", err.c_str());
    return -1;
  }
  ns::PackedRnn pk;
  ns::pack_rnn(m, pk);
  static ns::Tables tab;
  ns::make_tables(tab);
  if (chunk_cap < 1) chunk_cap = 8;
  ns::Params p = ns::call_params(in, out, vad, app, dbg, state, &tab, &pk.hdr, pk.words.data(), pk.bias.data(), in_stride,
                                 out_stride, n_frames, app_stride, n_streams, n_frames, chunk_cap, out_frame_offset, flags,
                                 volume);
  std::vector<float> hp((size_t)n_streams * p.hp_stride, 0.f);
  std::vector<uint32_t> tabw((size_t)n_streams * chunk_cap * ns::kTabWords, 0u);
  std::vector<float> rec((size_t)n_streams * chunk_cap * ns::kRecFloats, 0.f);
  std::vector<ns::cf> spec((size_t)n_streams * chunk_cap * 2 * ns::kSpecStride);
  const int groups = (n_streams + ns::kMmaStreams - 1) / ns::kMmaStreams;
  std::vector<uint32_t> featq((size_t)groups * chunk_cap * ns::kFeatBlockWords, 0xCDCDCDCDu);
  // both forms of K0 (the library picks by batch size; here $CRISPY_NS_HP_PAR = 0 selects the single recursion warp)
  const char *hpp = getenv("CRISPY_NS_HP_PAR");
  const bool hp_par = ns::hp_par_form(numerics, hpp ? atoi(hpp) != 0 : NS_HP_PAR != 0);
  const bool f32 = ns::biquad_f32(numerics);
  for (int f0 = 0; f0 < n_frames; f0 += chunk_cap) {
    const int nf = (n_frames - f0) < chunk_cap ? (n_frames - f0) : chunk_cap;
    // the library keeps its chunk counter in the batch handle; the emulation keeps it in stream 0's
    // state block (host side) so that chained calls see the same synthesis_mem buffer parity
    int *chunk_counter = reinterpret_cast<int *>(state) + ns::kStateFloats - 1;
    ns::set_chunk(p, f0, nf, hp.data(), tabw.data(), rec.data(), spec.data(), featq.data(), *chunk_counter & 1);
    *chunk_counter += 1;
    int rc = hp_par ? launch((n_streams + 31) / 32, ns::kHpParThreads, sizeof(ns::HpParSmem),
                             [&](void *sm) { ns::highpass_par_body(p, *(ns::HpParSmem *)sm); })
                    : launch((n_streams + 31) / 32, ns::kHpThreads, sizeof(ns::HpSmem), [&](void *sm) {
                        if (f32)
                          ns::highpass_body<true>(p, *(ns::HpSmem *)sm);
                        else
                          ns::highpass_body<false>(p, *(ns::HpSmem *)sm);
                      });
    if (rc) return rc;
    const int runs = (nf + kPitchRun - 1) / kPitchRun;
    rc = launch(n_streams * runs, kPitchThreads, sizeof(PitchShared), [&](void *sm) {
      ns::with_sum_order(numerics, [&](auto sp) {
#ifndef NS_PITCH_V7
        ns::pitch_body<kPitchRun, kPitchThreads, decltype(sp)::value>(p, *(PitchShared *)sm);
#else
        ns::pitch_body7<kPitchRun, kPitchThreads>(p, *(PitchShared *)sm);
#endif
      });
    });
    if (rc) return rc;
    rc = launch((n_streams + kScanWarps - 1) / kScanWarps, 32 * kScanWarps, 16,
                [&](void *) { ns::pitchscan_body(p, kScanWarps); });
    if (rc) return rc;
    const int spec_ctas = n_streams * nf < 4 ? n_streams * nf : 4;
    rc = launch(spec_ctas, ns::kGroupThreads, sizeof(ns::SpecSmem),
                [&](void *sm) { ns::spectrum_body(p, *(ns::SpecSmem *)sm); });
    if (rc) return rc;
    rc = launch((groups * ns::kMmaStreams + ns::kFeatWarps - 1) / ns::kFeatWarps, 32 * ns::kFeatWarps, sizeof(ns::FeatSmem),
                [&](void *sm) { ns::features_body(p, *(ns::FeatSmem *)sm); });
    if (rc) return rc;
    rc = launch(groups, ns::kMmaThreads, sizeof(ns::RnnSmem), [&](void *sm) { ns::rnn_body(p, *(ns::RnnSmem *)sm); });
    if (rc) return rc;
    p.syn_run = nf > 5 ? 5 : nf;  // a run length that leaves a ragged last run and exercises the halo path
    const int syn_tasks = n_streams * ((nf + p.syn_run - 1) / p.syn_run);
    rc = launch(syn_tasks < 3 ? syn_tasks : 3, ns::kGroupThreads, sizeof(ns::SpecSmem),
                [&](void *sm) { ns::synthesis_body(p, *(ns::SpecSmem *)sm); });
    if (rc) return rc;
  }
  return 0;
}

// the per-stream suppression controls (crispy_ns_controls) on row `stream` of a state as ns_emu_process takes it, word
// for word as libcrispy_ns.so's ns_set_controls_kernel writes them; the gate's carry is left alone
void ns_emu_set_controls(float *state, int stream, float min_gain, float gate_threshold, int gate_hold, float gate_gain) {
  float *row = state + (size_t)stream * ns::kStateFloats;
  row[ns::kStCtlMinGain] = min_gain;
  row[ns::kStCtlGateThr] = gate_threshold;
  memcpy(&row[ns::kStCtlGateHold], &gate_hold, 4);
  row[ns::kStCtlGateGain] = gate_gain;
}
}
