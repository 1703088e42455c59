// ns_emu_controls.cpp -- the host SIMT emulation (ns_emu.cpp, included whole) plus an entry point that sets the
// per-stream suppression controls (crispy_ns_controls) on state rows, word for word as libcrispy_ns.so's
// ns_set_controls_kernel does.  TEST PLUMBING.  Build as ns_emu.cpp: -ffp-contract=off.
#include "ns_emu.cpp"

extern "C" {
// state: [n_streams][kStateFloats] as ns_emu_process takes it; the gate's carry is left alone
void ns_emu_set_controls(float *state, int stream, float min_gain, float gate_threshold, int gate_hold, float gate_gain) {
  float *row = state + (size_t)stream * ns::kStateFloats;
  row[ns::kStCtlMinGain] = min_gain;
  row[ns::kStCtlGateThr] = gate_threshold;
  memcpy(&row[ns::kStCtlGateHold], &gate_hold, 4);
  row[ns::kStCtlGateGain] = gate_gain;
}
}
