"""GPU: per-stream suppression controls (crispy_ns_controls: attenuation limit and voice gate with hold).  The gate is
checked bit for bit against the run without controls times the NumPy ramp of the returned VAD (tests/controls_ref.py),
the floor against the oracle under the same controls; a stream's bits do not depend on who shares its batch or call."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import crispy_b200 as cb  # noqa: E402
from crispy_b200 import _lib  # noqa: E402
from tests import controls_oracle as co  # noqa: E402
from tests import controls_ref as cr  # noqa: E402
from tests.test_gpu_streams import make_schedule  # noqa: E402
from tests.util import BRANCH_EPS, TOL_MAX_ABS, TOL_SNR_DB, TOL_VAD, make_signal, snr_db  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 16  # engine chunk: a hold of 20 frames crosses chunk boundaries
EINVAL = -1
OFF = dict(min_gain=0.0, vad_threshold=0.0, hold_frames=0, gate_gain=0.0)
# per stream: off, gate only (mute, hold across chunks), floor only, both, gate with a partial gain and no hold
MIXED = [OFF, dict(min_gain=0.0, vad_threshold=0.55, hold_frames=20, gate_gain=0.0),
         dict(min_gain=0.1, vad_threshold=0.0, hold_frames=0, gate_gain=0.0),
         dict(min_gain=1e-3, vad_threshold=0.6, hold_frames=3, gate_gain=0.25),
         dict(min_gain=0.0, vad_threshold=0.5, hold_frames=0, gate_gain=0.5)]
TAP_PITCH = (130, 131, 132, 133)  # ns_common.h: pitch gain, VAD, pitch index, silence


@pytest.fixture(scope="module")
def model():
    return cb.Model.synthetic(0)


@pytest.fixture(autouse=True)
def small_chunks(monkeypatch):
    monkeypatch.setenv("CRISPY_NS_CHUNK_FRAMES", str(CHUNK))


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _set(den, controls):
    for s, c in enumerate(controls):
        den.set_controls([s], **c)


def _run(model, x, controls=None, rnn=None, monkeypatch=None, taps=True, **kw):
    if rnn:
        monkeypatch.setenv("CRISPY_NS_RNN", rnn)
    den = cb.BatchDenoiser(x.shape[0], model)
    if controls:
        _set(den, controls)
    r = den.process_streams(_dev(x), unit_scale=False, return_taps=taps, **kw)
    return [_np(t) for t in r]


def _gate_of(c):
    return c["vad_threshold"], c["hold_frames"], c["gate_gain"]


# ---- the gate: bit for bit against the ungated run ---------------------------------------------------------------------
@pytest.mark.parametrize("rnn", ["mma", "tc5"])
def test_gate_is_the_ungated_output_times_the_ramp(model, monkeypatch, rnn):
    gates = [dict(OFF, vad_threshold=t, hold_frames=h, gate_gain=g)
             for t, h, g in [(0.55, 20, 0.0), (0.6, 0, 0.25), (0.5, 3, 1.0), (1.0, 0, 0.0), (0.0, 5, 0.0), (0.58, 7, 0.1)]]
    x = make_signal(len(gates), 3 * CHUNK + 5)
    out0, vad0, taps0 = _run(model, x, None, rnn, monkeypatch)
    out1, vad1, taps1 = _run(model, x, gates, rnn, monkeypatch)
    assert np.array_equal(vad0, vad1) and np.array_equal(taps0.view(np.uint32), taps1.view(np.uint32))
    for s, c in enumerate(gates):
        want = cr.gated(out0[s], vad0[s], *_gate_of(c))
        assert np.array_equal(out1[s].view(np.uint32), want.view(np.uint32)), (rnn, s)


def test_controls_never_set_and_set_to_zero_give_the_same_bits(model):
    x = make_signal(5, 2 * CHUNK + 3)
    out0, vad0, taps0 = _run(model, x, None)
    out1, vad1, taps1 = _run(model, x, [OFF] * 5)
    assert np.array_equal(out0.view(np.uint32), out1.view(np.uint32)) and np.array_equal(taps0, taps1)


# ---- the floor: against the oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("min_gain", [1e-3, 0.1, 1.0])
def test_floor_matches_the_oracle(model, model_blob, min_gain):
    x = make_signal(4, 30)
    c = dict(OFF, min_gain=min_gain)
    out, vad, taps = _run(model, x, [c] * 4)
    ref, rvad, rpi, rpg, rsil, margin = co.process_streams(model_blob, x, [(min_gain, 0.0, 0, 0.0)] * 4)
    assert np.array_equal(taps[:, :, 132].astype(np.int32), rpi)
    assert np.array_equal(taps[:, :, 130].view(np.uint32), rpg.view(np.uint32))
    assert np.array_equal(taps[:, :, 133].astype(np.int32), rsil)
    assert np.abs(vad - rvad).max() <= TOL_VAD
    risky = margin < BRANCH_EPS
    risky[:, 1:] |= risky[:, :-1].copy()
    err = np.abs(out.astype(np.float64) - ref).reshape(4, 30, 480).max(2)
    assert err[~risky].max() <= TOL_MAX_ABS and risky.mean() < 0.1, (err[~risky].max(), risky.mean())
    assert snr_db(ref, out) >= TOL_SNR_DB
    _, _, taps0 = _run(model, x, None)
    for tap in TAP_PITCH:
        assert np.array_equal(taps[:, :, tap].view(np.uint32), taps0[:, :, tap].view(np.uint32))


def test_controls_are_not_vacuous_on_the_synthetic_workload(model):
    from crispy_b200.synth import synth_chunk
    x = (synth_chunk(16, 200 * 480, seed=5).numpy() * 32768.0).astype(np.float32)
    out0, vad0, taps0 = _run(model, x, None)
    g = np.stack([cr.gate_gains(vad0[s], 0.5, 20, 0.0)[0] for s in range(16)])
    assert (g == 0).sum() > 0 and (g == 1).mean() > 0.2, ((g == 0).mean(), (g == 1).mean())  # oracle: 0.9 % closed
    out1, _, _ = _run(model, x, [dict(OFF, min_gain=0.1)] * 16)
    changed = (out1 != out0).reshape(16, 200, 480).any(2)
    assert changed[taps0[:, :, 133] == 0].mean() > 0.5


# ---- per-stream independence -------------------------------------------------------------------------------------------
def test_mixed_controls_equal_batches_of_their_own(model):
    x = make_signal(len(MIXED), 2 * CHUNK + 7)
    out, vad = _run(model, x, MIXED, taps=False)
    for s, c in enumerate(MIXED):
        o1, v1 = _run(model, x[s:s + 1], [c], taps=False)
        assert np.array_equal(out[s].view(np.uint32), o1[0].view(np.uint32)) and np.array_equal(vad[s], v1[0]), s


@pytest.mark.parametrize("seed", [3, 8])
def test_subset_schedules_equal_single_stream_batches(model, seed):
    n = len(MIXED)
    sched = make_schedule(n, 10, seed)
    total = sum(nf for _, nf in sched)
    x = make_signal(n, total, seed=77)
    den = cb.BatchDenoiser(n, model)
    _set(den, MIXED)
    singles = []
    for s in range(n):
        d1 = cb.BatchDenoiser(1, model)
        d1.set_controls([0], **MIXED[s])
        singles.append(d1)
    f = 0
    for ids, nf in sched:
        ids = list(range(n)) if ids is None else ids
        xs = x[ids, f * 480:(f + nf) * 480]
        o, v = den.process_streams_subset(ids, _dev(xs), unit_scale=False)
        o, v = _np(o), _np(v)
        for i, s in enumerate(ids):
            o1, v1 = singles[s].process_streams(_dev(xs[i:i + 1]), unit_scale=False)
            assert np.array_equal(o[i].view(np.uint32), _np(o1)[0].view(np.uint32)), (ids, nf, s)
            assert np.array_equal(v[i], _np(v1)[0])
        f += nf


def test_new_controls_take_effect_at_the_next_call(model):
    x = make_signal(2, 2 * CHUNK + 9)
    a, b = 20 * 480, x.shape[1]
    ref = cb.BatchDenoiser(2, model)
    den = cb.BatchDenoiser(2, model)
    ca, cb_ = dict(OFF, vad_threshold=0.55, hold_frames=6, gate_gain=0.0), dict(OFF, vad_threshold=0.6, hold_frames=2, gate_gain=0.3)
    den.set_controls([0, 1], **ca)
    outs, refs = [], []
    for lo, hi, c in ((0, a, None), (a, b, cb_)):
        if c:
            den.set_controls([0, 1], **c)
        o, _ = den.process_streams(_dev(x[:, lo:hi]), unit_scale=False)
        r, v = ref.process_streams(_dev(x[:, lo:hi]), unit_scale=False)
        outs.append(_np(o))
        refs.append((_np(r), _np(v)))
    for s in range(2):
        g1, left, g_last = cr.gate_gains(refs[0][1][s], *_gate_of(ca))
        g2, _, _ = cr.gate_gains(refs[1][1][s], *_gate_of(cb_), left=left, g_prev=g_last)
        want1 = (refs[0][0][s] * cr.ramp(g1)).astype(np.float32)
        want2 = (refs[1][0][s] * cr.ramp(g2, g_prev=g_last)).astype(np.float32)
        assert np.array_equal(outs[0][s].view(np.uint32), want1.view(np.uint32))
        assert np.array_equal(outs[1][s].view(np.uint32), want2.view(np.uint32))
    assert den.get_controls([1])[0] == {"min_gain": 0.0, "vad_threshold": np.float32(0.6), "hold_frames": 2,
                                        "gate_gain": np.float32(0.3)}


# ---- lifecycle -------------------------------------------------------------------------------------------------------
def test_controls_travel_in_records_and_states_and_resets_clear_them(model):
    n = len(MIXED)
    x = make_signal(n, 3 * CHUNK)
    h = CHUNK + 5
    den = cb.BatchDenoiser(n, model)
    _set(den, MIXED)
    den.process_streams(_dev(x[:, :h * 480]), unit_scale=False)
    rec = den.save_streams([3, 1])
    whole = den.save_state()
    o_cont, _ = den.process_streams(_dev(x[:, h * 480:]), unit_scale=False)
    o_cont = _np(o_cont)
    # a stream record: into other slots of another batch
    other = cb.BatchDenoiser(n, model)
    other.load_streams([0, 4], rec)
    assert other.get_controls([0, 4]) == den.get_controls([3, 1])
    o2, _ = other.process_streams_subset([0, 4], _dev(x[[3, 1], h * 480:]), unit_scale=False)
    assert np.array_equal(_np(o2), o_cont[[3, 1]])
    # a whole-batch state
    third = cb.BatchDenoiser(n, model)
    third.load_state(whole)
    assert third.get_controls(range(n)) == den.get_controls(range(n))
    o3, _ = third.process_streams(_dev(x[:, h * 480:]), unit_scale=False)
    assert np.array_equal(_np(o3), o_cont)
    # per-stream reset clears only the listed streams; a whole reset clears all
    before = den.get_controls(range(n))
    den.reset_streams([1, 3])
    after = den.get_controls(range(n))
    zero = den.get_controls([0])[0]
    assert after[1] == zero and after[3] == zero and [after[i] for i in (0, 2, 4)] == [before[i] for i in (0, 2, 4)]
    den.reset()
    assert den.get_controls(range(n)) == [zero] * n
    assert zero == {"min_gain": 0.0, "vad_threshold": 0.0, "hold_frames": 0, "gate_gain": 0.0}


def test_records_without_controls_load_with_the_controls_off(model):
    """a stream that never had controls leaves every new word of its record zero -- the bytes a record saved before
    the controls existed holds there -- and such a record loads with the controls off"""
    x = make_signal(2, CHUNK + 3)
    den = cb.BatchDenoiser(2, model)
    den.process_streams(_dev(x), unit_scale=False)
    rec = den.save_streams([0])
    words = np.frombuffer(rec[16:], np.uint32)
    assert not words[2772:2779].any()
    other = cb.BatchDenoiser(2, model)
    other.set_controls([1], min_gain=0.5, vad_threshold=0.5, hold_frames=4, gate_gain=0.1)
    other.load_streams([1], rec)
    assert other.get_controls([1])[0] == den.get_controls([0])[0]


def test_bad_arguments_are_refused_and_change_nothing(model):
    den = cb.BatchDenoiser(3, model)
    den.set_controls([0, 1, 2], min_gain=0.25, vad_threshold=0.5, hold_frames=9, gate_gain=0.5)
    before = den.get_controls(range(3))
    L = _lib.lib()
    bad = [dict(min_gain=-0.1), dict(min_gain=1.5), dict(min_gain=float("nan")), dict(vad_threshold=1.01),
           dict(vad_threshold=float("nan")), dict(gate_gain=-1e-9), dict(gate_gain=float("inf")), dict(hold_frames=-1),
           dict(hold_frames=(1 << 20) + 1)]
    for b in bad:
        with pytest.raises(cb.CrispyNsError, match="error -1"):
            den.set_controls([0, 2], **b)
        assert den.get_controls(range(3)) == before, b
    c = (_lib.Controls * 2)(_lib.Controls(0.0, 0.0, 0, 0.0), _lib.Controls(0.0, 0.0, 0, 0.0))
    for ids in ([0, 0], [0, 3], [-1, 1]):
        arr = (C.c_int * 2)(*ids)
        assert L.crispy_ns_batch_set_controls(den._h, arr, 2, c, None) == EINVAL
        assert L.crispy_ns_batch_get_controls(den._h, arr, 2, c) == EINVAL
    assert L.crispy_ns_batch_set_controls(den._h, (C.c_int * 1)(0), 1, None, None) == EINVAL
    assert den.get_controls(range(3)) == before
    assert den.get_controls([2])[0]["hold_frames"] == 9
    den.set_controls([1], hold_frames=1 << 20, vad_threshold=1.0, gate_gain=1.0, min_gain=1.0)  # the closed ends


# ---- coverage: process_frame, host pointers, PCM16 and the dual-mono mix, the multi handle -----------------------------
def test_process_frame_follows_its_controls(model):
    x = make_signal(1, 24)
    c = dict(min_gain=0.05, vad_threshold=0.55, hold_frames=4, gate_gain=0.2)
    want, _ = _run(model, x, [c], taps=False)
    st = cb.DenoiseState(model)
    st.set_controls(**c)
    assert st.get_controls() == {"min_gain": np.float32(0.05), "vad_threshold": np.float32(0.55), "hold_frames": 4,
                                 "gate_gain": np.float32(0.2)}
    out = np.zeros(480, np.float32)
    got = []
    for t in range(24):
        st.process_frame(out, x[0, t * 480:(t + 1) * 480])
        got.append(out.copy())
    assert np.array_equal(np.concatenate(got), want[0])
    st.reset()
    assert st.get_controls()["vad_threshold"] == 0.0


def test_host_path_pcm16_and_the_dual_mono_mix(model):
    n = len(MIXED)
    x = np.clip(np.rint(make_signal(n, 2 * CHUNK + 1)), -32768, 32767).astype(np.int16)
    app = (make_signal(n, 2 * CHUNK + 1, seed=99) / np.float32(65536.0)).astype(np.float32)
    d = cb.BatchDenoiser(n, model)
    _set(d, MIXED)
    o16, _ = d.process_streams(_dev(x), unit_scale=False)
    o16 = _np(o16)
    h = cb.BatchDenoiser(n, model)
    _set(h, MIXED)
    oh, _ = h.process_streams_host(torch.from_numpy(x), unit_scale=False)
    assert np.array_equal(oh.numpy(), o16)
    m = cb.BatchDenoiser(n, model)
    _set(m, MIXED)
    mix, _ = m.process_streams(_dev(x), unit_scale=False, mix_stereo_i16=True, app=_dev(app))
    mix = _np(mix)
    u = np.clip(o16 / np.float32(32768.0), -1, 1).astype(np.float32)  # the gated microphone; the app audio is not gated
    want = np.trunc(np.clip((u + app).astype(np.float32), -1, 1) * np.float32(32767.0)).astype(np.int16)
    assert np.array_equal(mix[:, :, 0], want) and np.array_equal(mix[:, :, 1], want)


def test_multi_handle_over_two_blocks_of_one_device(model):
    n = 6
    x = (make_signal(n, 2 * CHUNK + 2) / np.float32(32768.0)).astype(np.float32)
    ctl = {1: MIXED[1], 4: MIXED[3], 5: MIXED[4]}
    md = cb.MultiDenoiser(n, [0, 0], model)
    assert [r[2] for r in md.ranges] == [3, 3]
    for s, c in ctl.items():
        md.set_controls([s], **c)
    ref = cb.BatchDenoiser(n, model)
    for s, c in ctl.items():
        ref.set_controls([s], **c)
    assert md.get_controls(range(n)) == ref.get_controls(range(n))
    o, v = md.process_streams_host(torch.from_numpy(x))
    r, rv = ref.process_streams_host(torch.from_numpy(x))
    assert np.array_equal(o.numpy(), r.numpy()) and np.array_equal(v.numpy(), rv.numpy())
    with pytest.raises(cb.CrispyNsError):
        md.set_controls([2, 5], min_gain=2.0)
    assert md.get_controls([5])[0] == ref.get_controls([5])[0]


def test_c_consumer_of_the_controls(tmp_path):
    exe = str(tmp_path / "controls_smoke")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c_abi", "controls_smoke.c"), "-L" + lib_dir, "-lcrispy_ns", "-lm",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "controls_smoke: ok" in r.stdout, r.stdout + r.stderr
