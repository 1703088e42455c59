"""NumPy float32 transliteration of the voice gate of crispy_ns_controls (include/crispy_ns.h), test plumbing: the gate
recursion over a stream's returned VAD and the per-sample ramp it multiplies the 16-bit-scale output with."""
from __future__ import annotations

import numpy as np

FRAME = 480


def gate_gains(vad, threshold, hold, gate_gain, left=0, g_prev=1.0):
    """G_t of every frame of one stream, and the carry (left, G of the last frame).  A frame is voiced if its VAD >=
    threshold; a voiced frame opens the gate for `hold` more frames; G = 1 while open, else gate_gain."""
    thr, gg = np.float32(threshold), np.float32(gate_gain)
    g = np.empty(len(vad), np.float32)
    for t, v in enumerate(np.asarray(vad, np.float32)):
        if not (v < thr):
            left, g[t] = hold, 1.0
        elif left > 0:
            left, g[t] = left - 1, 1.0
        else:
            g[t] = gg
    return g, left, (np.float32(g[-1]) if len(g) else np.float32(g_prev))


def ramp(g, g_prev=1.0):
    """[n_frames * 480] factors: G_{t-1} + (G_t - G_{t-1}) * ((float)(i + 1) / 480.0f), each operation rounded"""
    g = np.asarray(g, np.float32)
    prev = np.concatenate([[np.float32(g_prev)], g[:-1]]).astype(np.float32)
    frac = (np.arange(1, FRAME + 1, dtype=np.float32) / np.float32(FRAME)).astype(np.float32)
    r = prev[:, None] + ((g - prev)[:, None] * frac[None, :]).astype(np.float32)
    return r.astype(np.float32).reshape(-1)


def gated(out16, vad, threshold, hold, gate_gain):
    """what the gate makes of one stream's ungated 16-bit-scale output"""
    g, _, _ = gate_gains(vad, threshold, hold, gate_gain)
    return (np.asarray(out16, np.float32) * ramp(g)).astype(np.float32)
