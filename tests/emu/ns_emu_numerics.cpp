// ns_emu_numerics.cpp -- the host SIMT emulation (ns_emu.cpp, included whole) plus an entry point that runs K0 and K1
// under a model's numerics (crispy_ns_model_set_numerics: CRISPY_NS_SUM_* | CRISPY_NS_BIQUAD_F32).  TEST PLUMBING.
// Build as ns_emu.cpp: -ffp-contract=off.
#include "ns_emu.cpp"

extern "C" {
// as ns_emu_process, with the numerics of the batch: K1 sums in order (numerics & 3), K0 runs the f32 biquad when
// bit 4 is set (always on the single recursion warp: the time-parallel form speculates the f64 expression only)
int ns_emu_process_numerics(const void *model_blob, size_t model_len, const void *in, void *out, float *vad,
                            const float *app, float *state, float *dbg, int n_streams, int n_frames,
                            long long in_stride, long long out_stride, long long app_stride, int chunk_cap,
                            unsigned flags, float volume, int out_frame_offset, unsigned numerics) {
  const int sp = (int)(numerics & 3u);
  const bool biquad_f32 = (numerics & (1u << 4)) != 0;
  if (sp == 3 || (numerics & ~0x13u)) return -3;
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
  ns::Params p;
  memset(&p, 0, sizeof(p));
  const long long hp_stride = ns::kHist + (long long)chunk_cap * ns::kFrame;
  std::vector<float> hp((size_t)n_streams * hp_stride, 0.f);
  std::vector<uint32_t> tabw((size_t)n_streams * chunk_cap * ns::kTabWords, 0u);
  std::vector<float> rec((size_t)n_streams * chunk_cap * ns::kRecFloats, 0.f);
  std::vector<ns::cf> spec((size_t)n_streams * chunk_cap * 2 * ns::kSpecStride);
  const int groups = (n_streams + ns::kMmaStreams - 1) / ns::kMmaStreams;
  std::vector<uint32_t> featq((size_t)groups * chunk_cap * ns::kFeatBlockWords, 0xCDCDCDCDu);
  p.in = in;
  p.out = out;
  p.vad = vad;
  p.app = app;
  p.dbg = dbg;
  p.state = state;
  p.hp = hp.data();
  p.tab = tabw.data();
  p.rec = rec.data();
  p.spec = spec.data();
  p.featq = featq.data();
  p.tables = &tab;
  p.rnn_hdr = &pk.hdr;
  p.rnn_words = pk.words.data();
  p.rnn_bias = pk.bias.data();
  p.in_stride = in_stride;
  p.out_stride = out_stride;
  p.vad_stride = n_frames;
  p.app_stride = app_stride;
  p.hp_stride = hp_stride;
  p.n_streams = n_streams;
  p.n_frames_call = n_frames;
  p.chunk_cap = chunk_cap;
  p.out_frame_offset = out_frame_offset;
  p.flags = flags;
  p.volume = volume;
  for (int f0 = 0; f0 < n_frames; f0 += chunk_cap) {
    const int nf = (n_frames - f0) < chunk_cap ? (n_frames - f0) : chunk_cap;
    p.frame0 = f0;
    p.n_frames = nf;
    int *chunk_counter = reinterpret_cast<int *>(state) + ns::kStateFloats - 1;  // as ns_emu_process
    p.synth_sel = *chunk_counter & 1;
    *chunk_counter += 1;
    const bool hp_par = !biquad_f32 && NS_HP_PAR != 0;
    int rc = hp_par ? launch((n_streams + 31) / 32, ns::kHpParThreads, sizeof(ns::HpParSmem),
                             [&](void *sm) { ns::highpass_par_body(p, *(ns::HpParSmem *)sm); })
                    : launch((n_streams + 31) / 32, ns::kHpThreads, sizeof(ns::HpSmem), [&](void *sm) {
                        if (biquad_f32)
                          ns::highpass_body<true>(p, *(ns::HpSmem *)sm);
                        else
                          ns::highpass_body<false>(p, *(ns::HpSmem *)sm);
                      });
    if (rc) return rc;
    const int runs = (nf + kPitchRun - 1) / kPitchRun;
    rc = launch(n_streams * runs, kPitchThreads, sizeof(PitchShared), [&](void *sm) {
      if (sp == 2)
        ns::pitch_body<kPitchRun, kPitchThreads, 2>(p, *(PitchShared *)sm);
      else if (sp == 1)
        ns::pitch_body<kPitchRun, kPitchThreads, 1>(p, *(PitchShared *)sm);
      else
        ns::pitch_body<kPitchRun, kPitchThreads, 0>(p, *(PitchShared *)sm);
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
    p.syn_run = nf > 5 ? 5 : nf;
    const int syn_tasks = n_streams * ((nf + p.syn_run - 1) / p.syn_run);
    rc = launch(syn_tasks < 3 ? syn_tasks : 3, ns::kGroupThreads, sizeof(ns::SpecSmem),
                [&](void *sm) { ns::synthesis_body(p, *(ns::SpecSmem *)sm); });
    if (rc) return rc;
  }
  return 0;
}
}
