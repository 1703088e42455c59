"""Test plumbing: the oracle under every numerics setting of the library (crispy_ns_model_set_numerics).

The oracle (oracle/rnnoise_oracle.c) already switches the pitch path's summation order (rno_set_sum_policy).  For the
biquad in f32 arithmetic (CRISPY_NS_BIQUAD_F32) the same source is compiled a second time, once per process into a
temporary directory, with the a6 high-pass call redirected to the f32 form

    yi = xi + mem[0];  mem[0] = mem[1] + (b[0]*xi - a[0]*yi);  mem[1] = b[1]*xi - a[1]*yi;

all float, every product and sum rounded separately (-ffp-contract=off, as the oracle's own build).  Nothing else of
the oracle changes, and the build refuses to proceed if the source no longer has the one call it redirects.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from oracle import pyoracle as po
from tests.util import patched_oracle

CALL = "biquad(x, st->mem_hp_x, in, b_hp, a_hp, FRAME_SIZE);"
DEF = "static void biquad(float *y, float mem[2], const float *x, const float *b, const float *a, int N) {"
F32_BIQUAD = """static void biquad_f32(float *y, float mem[2], const float *x, const float *b, const float *a, int N) {
  int i;
  for (i = 0; i < N; i++) {
    float xi = x[i];
    float yi = xi + mem[0];
    mem[0] = mem[1] + (b[0] * xi - a[0] * yi);
    mem[1] = b[1] * xi - a[1] * yi;
    y[i] = yi;
  }
}
"""
HIGHPASS = """
void rno_numerics_highpass_f32(float *y, float mem[2], const float *x, int n) {
  static const float a_hp[2] = {-1.99599f, 0.99600f};
  static const float b_hp[2] = {-2, 1};
  biquad_f32(y, mem, x, b_hp, a_hp, n);
}
"""

_lib = None


def lib_f32() -> C.CDLL:
    """the oracle with the f32 biquad (pyoracle's bindings, plus rno_numerics_highpass_f32)"""
    global _lib
    if _lib is None:
        L = patched_oracle([(DEF, F32_BIQUAD + DEF), (CALL, "biquad_f32" + CALL[len("biquad"):])], HIGHPASS)
        f32p = C.POINTER(C.c_float)
        L.rno_numerics_highpass_f32.argtypes = [f32p, f32p, f32p, C.c_int]
        L.rno_numerics_highpass_f32.restype = None
        _lib = L
    return _lib


def highpass_f32(x: np.ndarray, mem=(0.0, 0.0)):
    """the f32 biquad alone on one signal: (y, final (mem0, mem1))"""
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.zeros_like(x)
    m = np.array(mem, dtype=np.float32)
    lib_f32().rno_numerics_highpass_f32(po._fp(y), po._fp(m), po._fp(x), x.size)
    return y, (m[0], m[1])


def process_streams_trace(model_blob: bytes, x: np.ndarray, numerics: int, unit_scale: bool = False,
                          n_threads: int = 1, native: bool = False, margin: bool = False):
    """po.process_streams_trace under a library numerics setting (sum order = numerics & 3, bit 4 = f32 biquad); the
    f32 build has no -march=native variant, so `native` applies to the f64 biquad only"""
    if not numerics & 16:
        model = po.Model.from_bytes(model_blob)
        return po.process_streams_trace(model, x, unit_scale=unit_scale, n_threads=n_threads, native=native,
                                        sum_policy=numerics & 3, margin=margin)
    L = lib_f32()
    x = np.ascontiguousarray(x, dtype=np.float32)
    n_streams, n = x.shape
    n_frames = n // po.FRAME_SIZE
    out = np.zeros_like(x)
    vad = np.zeros((n_streams, n_frames), dtype=np.float32)
    pi = np.zeros((n_streams, n_frames), dtype=np.int32)
    pg = np.zeros((n_streams, n_frames), dtype=np.float32)
    sil = np.zeros((n_streams, n_frames), dtype=np.int32)
    mg = np.zeros((n_streams, n_frames), dtype=np.float32) if margin else None
    m = L.rno_model_from_bytes(model_blob, len(model_blob))
    assert m, "the oracle refused the model blob"
    L.rno_set_sum_policy(numerics & 3)
    try:
        L.rno_process_streams_trace(m, po._fp(x), po._fp(out), po._fp(vad), n_streams, n_frames, n, n,
                                    1 if unit_scale else 0, 1.0, n_threads, pi.ctypes.data_as(C.POINTER(C.c_int32)),
                                    po._fp(pg), sil.ctypes.data_as(C.POINTER(C.c_int32)), po._fp(mg) if margin else None)
    finally:
        L.rno_set_sum_policy(0)
        L.rno_model_free(m)
    return (out, vad, pi, pg, sil, mg) if margin else (out, vad, pi, pg, sil)
