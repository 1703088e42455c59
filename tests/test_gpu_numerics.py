"""GPU: the model's numerics setting (crispy_ns_model_set_numerics) on the CUDA path.  Under every combination of the
pitch path's summation order and the biquad's arithmetic, the kernels name the same pitch index, pitch gain and silence
gate as the oracle under the same combination, bit for bit, and meet north_star's tolerances on the samples; every
entry point inherits the setting through its batch; stream records carry it."""
import ctypes as C
import itertools
import os
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import crispy_b200 as cb  # noqa: E402
from crispy_b200 import _lib  # noqa: E402
from crispy_b200.synth import synth_chunk  # noqa: E402
from tests import numerics_oracle as no  # noqa: E402
from tests.util import (TOL_MAX_ABS, TOL_SNR_DB, TOL_VAD, assert_parity, long_run_parity, make_signal,  # noqa: E402
                        parity_report)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORES = os.cpu_count() or 1
EINVAL = -1
SUMS = (_lib.SUM_SEQUENTIAL, _lib.SUM_DOT4, _lib.SUM_DOT4_XCORR)
COMBOS = [s | b for s, b in itertools.product(SUMS, (0, _lib.BIQUAD_F32))]
TAP_GAIN, TAP_INDEX, TAP_SILENCE = 130, 132, 133


def model_with(numerics: int) -> "cb.Model":
    m = cb.Model.synthetic(0)
    m.numerics = numerics
    return m


def oracle_trace(model_blob, x, numerics, **kw):
    """the oracle under the same numerics (tests/numerics_oracle.py)"""
    return no.process_streams_trace(model_blob, x, numerics, n_threads=CORES, native=True, **kw)


def bits_differ(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """float32 identity with NaN equal to NaN (a signal decaying through the denormals can give a NaN pitch gain in
    the oracle and the kernels alike; their payloads need not match)"""
    return (a.view(np.uint32) != b.view(np.uint32)) & ~(np.isnan(a) & np.isnan(b))


def decisions(taps, rpi, rpg, rsil) -> dict:
    return {"pitch_index_flips": int((taps[:, :, TAP_INDEX].astype(np.int32) != rpi).sum()),
            "pitch_gain_bit_differences": int(bits_differ(taps[:, :, TAP_GAIN], rpg).sum()),
            "silence_gate_flips": int((taps[:, :, TAP_SILENCE].astype(np.int32) != rsil).sum())}


# ---- long runs: 16 streams of a 1,024-stream batch over 60 s, per combination -----------------------------------------
C2_IDS = [0, 3, 19, 64, 127, 200, 255, 256, 333, 511, 512, 640, 777, 900, 1003, 1023]
_c2_gains = {}  # numerics -> (GPU pitch gains, oracle pitch gains) of the 16 streams


@pytest.fixture(scope="module")
def c2_input():
    n_streams, n_frames = 1024, 6000
    return torch.cat([synth_chunk(n_streams, min(100, n_frames - f) * 480, start_sample=f * 480, device="cuda")
                      for f in range(0, n_frames, 100)], 1)


@pytest.mark.parametrize("numerics", COMBOS)
def test_c2_sixteen_streams_of_the_full_batch_match_the_oracle_under_the_same_numerics(model_blob, c2_input, numerics):
    x = c2_input
    model = model_with(numerics)
    den = cb.BatchDenoiser(x.shape[0], model)
    out, vad = den.process_streams(x, unit_scale=True)
    xs = x[C2_IDS].contiguous()
    ref, rvad, rpi, rpg, rsil, rmargin = oracle_trace(model_blob, xs.cpu().numpy(), numerics, unit_scale=True,
                                                      margin=True)
    den16 = cb.BatchDenoiser(16, model)
    o16, v16, taps = den16.process_streams(xs, unit_scale=True, return_taps=True)
    assert torch.equal(o16, out[C2_IDS]) and torch.equal(v16, vad[C2_IDS]), "a stream's result must not depend on its batch"
    taps = taps.cpu().numpy()
    d = decisions(taps, rpi, rpg, rsil)
    assert d == {"pitch_index_flips": 0, "pitch_gain_bit_differences": 0, "silence_gate_flips": 0}, (numerics, d)
    r = long_run_parity(ref, out[C2_IDS].cpu().numpy(), rvad, vad[C2_IDS].cpu().numpy(), rmargin, f"c2 numerics {numerics}")
    print(f"c2 numerics {numerics}:", {**d, **r})
    _c2_gains[numerics] = (taps[:, :, TAP_GAIN].copy(), rpg)


def test_c2_pitch_gains_move_with_the_sum_order_where_the_oracles_do():
    """Non-vacuity: against the sequential order, the GPU's pitch gains under DOT4 and DOT4_XCORR change in exactly the
    frames where the oracle's change (most frames: the gain is a ratio of the changed inner products)."""
    for bq in (0, _lib.BIQUAD_F32):
        for pol in (_lib.SUM_DOT4, _lib.SUM_DOT4_XCORR):
            if bq not in _c2_gains or (pol | bq) not in _c2_gains:
                pytest.skip("the per-combination runs above did not all complete")
            g0, r0 = _c2_gains[bq]
            g1, r1 = _c2_gains[pol | bq]
            moved, moved_ref = bits_differ(g1, g0), bits_differ(r1, r0)
            assert np.array_equal(moved, moved_ref), (pol | bq)
            assert moved.mean() > 0.5, (pol | bq, float(moved.mean()))
    assert bits_differ(_c2_gains[_lib.BIQUAD_F32][0], _c2_gains[0][0]).any()


# ---- small batches: where the default picks the time-parallel biquad ---------------------------------------------------
def test_small_batch_runs_the_f32_biquad_on_the_single_warp(model_blob, monkeypatch):
    """256 streams: without the setting the time-parallel K0 runs, which speculates the f64 expression.  Under
    BIQUAD_F32 the single recursion warp runs whatever the stream count or $CRISPY_NS_HP_PAR says."""
    n, nf, ids = 256, 300, [0, 1, 77, 255]
    x = torch.from_numpy(make_signal(n, nf, seed=31)).cuda()
    nm = _lib.SUM_DOT4 | _lib.BIQUAD_F32
    out, vad, taps = cb.BatchDenoiser(n, model_with(nm)).process_streams(x, unit_scale=False, return_taps=True)
    ref, rvad, rpi, rpg, rsil = oracle_trace(model_blob, x[ids].cpu().numpy(), nm)
    taps = taps[ids].cpu().numpy()
    assert decisions(taps, rpi, rpg, rsil) == {"pitch_index_flips": 0, "pitch_gain_bit_differences": 0,
                                               "silence_gate_flips": 0}
    assert_parity(ref, out[ids].cpu().numpy(), rvad, vad[ids].cpu().numpy(), "256 streams, f32 biquad")
    monkeypatch.setenv("CRISPY_NS_HP_PAR", "1")
    monkeypatch.setenv("CRISPY_NS_HP_EXCLUSIVE", "1")
    o2, v2 = cb.BatchDenoiser(n, model_with(nm)).process_streams(x, unit_scale=False)
    assert torch.equal(o2, out) and torch.equal(v2, vad)
    # and the setting is not ignored: the f64 biquad gives other samples
    o0, _ = cb.BatchDenoiser(n, model_with(_lib.SUM_DOT4)).process_streams(x, unit_scale=False)
    assert not torch.equal(o0, out)


# ---- other cores and entry points under a nonzero setting --------------------------------------------------------------
def test_tcgen05_core_under_dot4(model_blob, monkeypatch):
    monkeypatch.setenv("CRISPY_NS_RNN", "tc5")
    n, nf = 130, 120  # two tcgen05 CTAs, the second mostly empty
    x = torch.from_numpy(make_signal(n, nf, seed=32)).cuda()
    den = cb.BatchDenoiser(n, model_with(_lib.SUM_DOT4))
    assert den.info["rnn_streams_per_cta"] == 128
    out, vad, taps = den.process_streams(x, unit_scale=False, return_taps=True)
    ids = [0, 1, 64, 129]
    ref, rvad, rpi, rpg, rsil = oracle_trace(model_blob, x[ids].cpu().numpy(), _lib.SUM_DOT4)
    assert decisions(taps[ids].cpu().numpy(), rpi, rpg, rsil) == {"pitch_index_flips": 0, "pitch_gain_bit_differences": 0,
                                                                  "silence_gate_flips": 0}
    assert_parity(ref, out[ids].cpu().numpy(), rvad, vad[ids].cpu().numpy(), "tc5 core, DOT4")


def test_process_frame_equals_a_one_stream_batch(model_blob):
    nm = _lib.SUM_DOT4_XCORR | _lib.BIQUAD_F32
    model = model_with(nm)
    x = make_signal(1, 40, seed=33)
    want, wvad = cb.BatchDenoiser(1, model).process_streams(torch.from_numpy(x).cuda(), unit_scale=False)
    want, wvad = want.cpu().numpy()[0], wvad.cpu().numpy()[0]
    st = cb.DenoiseState.new(model)
    model.numerics = 0  # the handle copied the setting when it was created
    o = np.zeros(480, np.float32)
    for t in range(40):
        v = st.process_frame(o, x[0, t * 480:(t + 1) * 480])
        assert np.array_equal(o, want[t * 480:(t + 1) * 480]) and np.float32(v) == wvad[t], t
    ref, rvad = oracle_trace(model_blob, x, nm)[:2]
    assert_parity(ref, want[None, :], rvad, wvad[None, :], "process_frame, DOT4_XCORR + f32 biquad")


def test_random_subset_schedule_equals_batches_of_their_own(monkeypatch):
    from tests.test_gpu_streams import CHUNK, Variant, make_schedule, reference, run_schedule
    monkeypatch.setenv("CRISPY_NS_CHUNK_FRAMES", str(CHUNK))
    model = model_with(_lib.SUM_DOT4 | _lib.BIQUAD_F32)
    n = 21
    sched = make_schedule(n, 10, seed=41)
    var = Variant("f32", n, sum(nf for _, nf in sched))
    outs, vads, pos = run_schedule(cb.BatchDenoiser(n, model), var, sched, n)
    for s in range(n):
        o, v, _ = reference(model, var, s, int(pos[s]))
        assert torch.equal(outs[s], o) and torch.equal(vads[s], v), s


def test_stream_records_carry_the_numerics():
    """A record saved under numerics 1 continues bit-identically in another numerics-1 batch and is refused by a
    numerics-0 batch, whose state stays untouched.  At numerics 0 the header word stays 0."""
    x = make_signal(5, 60, seed=51)
    one = model_with(_lib.SUM_DOT4)
    a = cb.BatchDenoiser(5, one)
    a.process_streams(torch.from_numpy(x[:, :25 * 480]).cuda(), unit_scale=False)
    blob = a.save_streams([2])
    assert struct.unpack_from("<8sII", blob) == (b"CRNSSTR1", (len(blob) - 16) // 4, _lib.SUM_DOT4)
    b = cb.BatchDenoiser(3, one)
    b.load_streams([1], blob)
    got, gv = b.process_streams_subset([1], torch.from_numpy(x[2:3, 25 * 480:]).cuda(), unit_scale=False)
    whole, wv = cb.BatchDenoiser(1, one).process_streams(torch.from_numpy(x[2:3]).cuda(), unit_scale=False)
    assert torch.equal(got[0], whole[0, 25 * 480:]) and torch.equal(gv[0], wv[0, 25:])
    zero = cb.BatchDenoiser(3, cb.Model.synthetic(0))
    zero.process_streams(torch.from_numpy(x[:3, :10 * 480]).cuda(), unit_scale=False)
    snap = zero.save_state()
    ids = (C.c_int * 1)(1)
    assert _lib.lib().crispy_ns_batch_load_streams(zero._h, ids, 1, blob, len(blob)) == EINVAL
    assert b"numerics" in _lib.lib().crispy_ns_last_error()
    assert zero.save_state() == snap
    assert struct.unpack_from("<I", zero.save_streams([0]), 12)[0] == 0


def test_multi_gpu_handle_inherits_the_setting():
    """crispy_ns_multi_create over one device: its batch takes the model's numerics"""
    nm = _lib.SUM_DOT4_XCORR
    x = make_signal(4, 30, seed=61)
    m = cb.MultiDenoiser(4, devices=[0], model=model_with(nm))
    out, vad = m.process_streams_host(torch.from_numpy(x).pin_memory(), unit_scale=False)
    want, wvad = cb.BatchDenoiser(4, model_with(nm)).process_streams(torch.from_numpy(x).cuda(), unit_scale=False)
    assert torch.equal(out, want.cpu()) and torch.equal(vad, wvad.cpu())


# ---- the real reference ------------------------------------------------------------------------------------------------
GOLDEN = os.environ.get("CRISPY_NNNOISELESS_GOLDEN", os.path.join(ROOT, "tests", "golden", "nnnoiseless_c1.npz"))
WEIGHTS = os.environ.get("CRISPY_NS_REAL_WEIGHTS", os.path.join(ROOT, "weights", "rnnoise_default.crnsmdl"))
HAVE = os.path.exists(GOLDEN) and os.path.exists(WEIGHTS)
WHY = ("PARITY UNPINNED: no nnnoiseless 0.5.2 output / weights in the tree (" + os.path.relpath(GOLDEN, ROOT) + ", "
       + os.path.relpath(WEIGHTS, ROOT) + "), so no numerics setting can be checked against the crate; make them with "
       "tools/nnnoiseless_golden/README.md")


@pytest.mark.skipif(not HAVE, reason=WHY)
def test_which_numerics_match_nnnoiseless():
    """The crate's clip under every combination; reports which meet north_star against the crate's own output."""
    g = np.load(GOLDEN)
    x = torch.from_numpy(g["x"].astype(np.float32)[None, :]).cuda()
    blob = open(WEIGHTS, "rb").read()
    results = {}
    for nm in COMBOS:
        model = cb.Model.from_bytes(blob)
        model.numerics = nm
        out, vad = cb.BatchDenoiser(1, model).process_streams(x, unit_scale=False)
        r = parity_report(g["out"][None, :], out.cpu().numpy(), g["vad"][None, :], vad.cpu().numpy())
        r["meets_north_star"] = r["max_abs"] <= TOL_MAX_ABS and r["snr_db"] >= TOL_SNR_DB and r["vad_max"] <= TOL_VAD
        results[nm] = r
    print("numerics vs nnnoiseless 0.5.2:", results)
    assert any(r["meets_north_star"] for r in results.values()), results
