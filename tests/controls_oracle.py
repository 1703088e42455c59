"""Test plumbing: the oracle under the per-stream suppression controls of the library (crispy_ns_controls).

The oracle (oracle/rnnoise_oracle.c) has no controls.  The same source is compiled a second time, once per process into
a temporary directory, with two edits and one addition:
  - the band gains handed to interp_band_gain for the spectrum become max(g, min_gain) when min_gain > 0 (lastg keeps
    g, the pitch filter g_raw, silent frames never get there);
  - the branch margin counts a band as audible when the floor makes it so;
  - rno_controls_process_frame runs rno_process_frame under a stream's controls and applies the voice gate to its
    16-bit-scale output: the recursion over the returned VAD and the ramp G_{t-1} + (G_t - G_{t-1}) * ((i + 1) / 480),
    in C float arithmetic with every operation rounded (-ffp-contract=off, as the oracle's own build).
Nothing else of the oracle changes, and the build refuses to proceed if the source no longer has what it edits.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import pyoracle as po
from tests.util import patched_oracle

INCLUDE = "#include <string.h>\n"
APPLY = "    interp_band_gain(gf, g);\n"
APPLY_FLOORED = """    if (g_ctl_min_gain > 0.f) {
      float ga[NB_BANDS]; /* the applied gains; lastg keeps the unfloored ones */
      for (i = 0; i < NB_BANDS; i++) ga[i] = fmaxf(g[i], g_ctl_min_gain);
      interp_band_gain(gf, ga);
    } else {
      interp_band_gain(gf, g);
    }
"""
AUDIBLE = "if (audible > 1e-3f && d < st->branch_margin)"
AUDIBLE_FLOORED = "if (fmaxf(audible, g_ctl_min_gain) > 1e-3f && d < st->branch_margin)"
GLOBAL = "static _Thread_local float g_ctl_min_gain; /* the floor of the frame being processed */\n"
ENTRY = r"""
typedef struct {
  float min_gain, gate_threshold;
  int gate_hold;
  float gate_gain;
  int left, shut;   /* the gate's carry: hold frames left, whether G of the last frame was a closed gate's */
  float shut_gain;  /* that G */
} rno_controls;

float rno_controls_process_frame(rno_state *st, rno_controls *c, float *out, const float *in) {
  float v, gp, gc;
  int i, open = 1;
  g_ctl_min_gain = c->min_gain;
  v = rno_process_frame(st, out, in); /* the returned VAD: 0 on silent frames */
  g_ctl_min_gain = 0.f;
  gp = c->shut ? c->shut_gain : 1.f;
  if (!(v < c->gate_threshold)) /* voiced (a NaN VAD counts as voiced) */
    c->left = c->gate_hold;
  else if (c->left > 0)
    c->left -= 1;
  else
    open = 0;
  gc = open ? 1.f : c->gate_gain;
  c->shut = !open;
  c->shut_gain = open ? 0.f : c->gate_gain;
  if (gp != 1.f || gc != 1.f)
    for (i = 0; i < FRAME_SIZE; i++) out[i] = out[i] * (gp + (gc - gp) * ((float)(i + 1) / 480.0f));
  return v;
}

float rno_controls_branch_margin(const rno_state *st) { return st->branch_margin; }
"""


class Controls(C.Structure):
    _fields_ = [("min_gain", C.c_float), ("gate_threshold", C.c_float), ("gate_hold", C.c_int),
                ("gate_gain", C.c_float), ("left", C.c_int), ("shut", C.c_int), ("shut_gain", C.c_float)]


_lib = None


def lib() -> C.CDLL:
    """the oracle with the controls (pyoracle's bindings, plus rno_controls_*)"""
    global _lib
    if _lib is None:
        L = patched_oracle([(INCLUDE, INCLUDE + GLOBAL), (APPLY, APPLY_FLOORED), (AUDIBLE, AUDIBLE_FLOORED)], ENTRY)
        f32p = C.POINTER(C.c_float)
        L.rno_controls_process_frame.argtypes = [C.c_void_p, C.POINTER(Controls), f32p, f32p]
        L.rno_controls_process_frame.restype = C.c_float
        L.rno_controls_branch_margin.argtypes = [C.c_void_p]
        L.rno_controls_branch_margin.restype = C.c_float
        _lib = L
    return _lib


def process_streams(model_blob: bytes, x: np.ndarray, controls):
    """Frame by frame, stream s under controls[s] = (min_gain, gate_threshold, gate_hold, gate_gain), 16-bit scale:
    (out, vad, pitch_index, pitch_gain, silence, branch margin), each [n_streams, n_frames] but out."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    n_streams, n = x.shape
    n_frames = n // po.FRAME_SIZE
    out = np.zeros_like(x)
    vad, pg, mg = (np.zeros((n_streams, n_frames), np.float32) for _ in range(3))
    pi, sil = (np.zeros((n_streams, n_frames), np.int32) for _ in range(2))
    m = L.rno_model_from_bytes(model_blob, len(model_blob))
    assert m, "the oracle refused the model blob"
    try:
        for s in range(n_streams):
            st = L.rno_create(m)
            c = Controls(*controls[s], 0, 0, 0.0)
            d = po.Debug()
            fo = np.empty(po.FRAME_SIZE, np.float32)
            for t in range(n_frames):
                fi = np.ascontiguousarray(x[s, t * po.FRAME_SIZE:(t + 1) * po.FRAME_SIZE])
                vad[s, t] = L.rno_controls_process_frame(st, C.byref(c), po._fp(fo), po._fp(fi))
                out[s, t * po.FRAME_SIZE:(t + 1) * po.FRAME_SIZE] = fo
                L.rno_get_debug(st, C.byref(d))
                pi[s, t], pg[s, t], sil[s, t] = d.pitch_index, d.pitch_gain, d.silence
                mg[s, t] = L.rno_controls_branch_margin(st)
            L.rno_destroy(st)
    finally:
        L.rno_model_free(m)
    return out, vad, pi, pg, sil, mg
