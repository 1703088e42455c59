"""CPU: the per-stream suppression controls (crispy_ns_controls: attenuation limit and voice gate).  The C boundary's
contract without a device, the oracle under the controls (tests/controls_oracle.py) against a NumPy float32
transliteration of the gate (tests/controls_ref.py), and K4 / K5 under the host SIMT emulation
(tests/emu/ns_emu.cpp) with different controls per stream against that oracle under the same controls."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import crispy_b200 as cb
from crispy_b200 import _lib, build
from oracle import pyoracle as po
from tests import controls_oracle as co
from tests import controls_ref as cr
from tests.util import BRANCH_EPS, TOL_MAX_ABS, TOL_SNR_DB, TOL_VAD, emu_lib, emu_process, make_signal, snr_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL, ENODEV = -1, -2
TAP_GAIN, TAP_VAD, TAP_INDEX, TAP_SILENCE = 130, 131, 132, 133  # ns_common.h debug taps
# (min_gain, gate_threshold, gate_hold, gate_gain) per stream: off, gate only, floor only, both (hold across chunks)
CONTROLS = [(0.0, 0.0, 0, 0.0), (0.0, 0.55, 3, 0.0), (0.1, 0.0, 0, 0.0), (1e-3, 0.6, 10, 0.25)]
NF, CHUNK = 30, 8
ST_CTL = 2772  # ns_common.h kStCtlMinGain: min_gain, threshold, hold, gate gain, then left, shut, shut gain


@pytest.fixture(scope="module", autouse=True)
def built():
    build.build()


# ---- the C ABI -------------------------------------------------------------------------------------------------------
def test_controls_struct_matches_the_header():
    h = open(os.path.join(ROOT, "include", "crispy_ns.h")).read()
    body = re.search(r"typedef struct \{(.*?)\} crispy_ns_controls;", h, flags=re.S).group(1)
    fields = re.findall(r"^\s*(float|int32_t)\s+(\w+);", body, flags=re.M)
    assert [(f, t) for t, f in fields] == [(n, "float" if t is C.c_float else "int32_t") for n, t in _lib.Controls._fields_]
    assert C.sizeof(_lib.Controls) == 16


def test_new_symbols_are_exported():
    new = {"crispy_ns_batch_set_controls", "crispy_ns_batch_get_controls", "crispy_ns_set_controls",
           "crispy_ns_get_controls", "crispy_ns_multi_set_controls", "crispy_ns_multi_get_controls"}
    assert new <= set(_lib.SYMBOLS)
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert new <= set(re.findall(r"\b(crispy_ns_\w+)$", nm, flags=re.M))


def test_null_handles_are_refused():
    L = _lib.lib()
    ids = (C.c_int * 1)(0)
    c = _lib.Controls(0.5, 0.5, 3, 0.0)
    assert L.crispy_ns_batch_set_controls(None, ids, 1, C.byref(c), None) == EINVAL
    assert L.crispy_ns_batch_get_controls(None, ids, 1, C.byref(c)) == EINVAL
    assert L.crispy_ns_set_controls(None, C.byref(c)) == EINVAL
    assert L.crispy_ns_get_controls(None, C.byref(c)) == EINVAL
    assert L.crispy_ns_multi_set_controls(None, ids, 1, C.byref(c)) == EINVAL
    assert L.crispy_ns_multi_get_controls(None, ids, 1, C.byref(c)) == EINVAL
    assert b"null handle" in L.crispy_ns_last_error()
    assert (c.min_gain, c.gate_threshold, c.gate_hold, c.gate_gain) == (0.5, 0.5, 3, 0.0)


def test_handles_follow_the_enodev_contract_without_a_device():
    if cb.device_count() > 0:
        pytest.skip("a CUDA device is present: the controls are exercised by tests/test_gpu_controls.py")
    with pytest.raises(cb.CrispyNsError, match="error -2"):
        cb.BatchDenoiser(4)
    with pytest.raises(cb.CrispyNsError, match="error -2"):
        cb.DenoiseState()


def test_python_arguments_map_onto_the_struct():
    from crispy_b200.denoise import _controls
    c = _controls(2, None, 20.0, [0.25, 0.5], 7, 0.125)
    assert [(x.min_gain, x.gate_threshold, x.gate_hold, x.gate_gain) for x in c] == \
        [(np.float32(0.1), 0.25, 7, 0.125), (np.float32(0.1), 0.5, 7, 0.125)]
    assert _controls(1, None, None, 0.0, 0, 0.0)[0].min_gain == 0.0
    assert _controls(1, None, None, 0.0, 2**40, 0.0)[0].gate_hold == -1  # refused by the library, not wrapped
    with pytest.raises(cb.CrispyNsError):
        _controls(1, 0.5, 6.0, 0.0, 0, 0.0)


def test_c_consumer_compiles_against_the_header(tmp_path):
    exe = str(tmp_path / "controls_smoke")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c_abi", "controls_smoke.c"), "-L" + lib_dir, "-lcrispy_ns", "-lm",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    if cb.device_count() == 0:
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 0 and "ENODEV contract ok" in r.stdout, r.stdout + r.stderr


def test_cpp_layer_exposes_the_controls(tmp_path):
    src = tmp_path / "controls.cpp"
    src.write_text(r"""
#include <crispy_ns.hpp>
#include <cstdio>
int main() {
  crispy::Controls c{};
  if (c.min_gain != 0.f || c.gate_threshold != 0.f || c.gate_hold != 0 || c.gate_gain != 0.f) return 1;
  try {
    crispy::BatchDenoiser b(2);
    b.set_controls({0}, {crispy::Controls{0.1f, 0.5f, 3, 0.f}});
    if (b.controls({0})[0].gate_hold != 3) return 2;
    try {
      b.set_controls({0}, {crispy::Controls{2.f, 0.f, 0, 0.f}});
      return 3;
    } catch (const crispy::Error &e) {
      if (e.code() != CRISPY_NS_EINVAL) return 4;
    }
  } catch (const crispy::Error &e) {
    if (e.code() != CRISPY_NS_ENODEV) return 5;
  }
  std::printf("controls ok\n");
  return 0;
}
""")
    exe = str(tmp_path / "controls")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                           "-L" + lib_dir, "-lcrispy_ns", "-Wl,-rpath," + lib_dir, "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "controls ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


# ---- the oracle's gate -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sig():
    return make_signal(len(CONTROLS), NF)


@pytest.fixture(scope="module")
def oracle_off(model_blob, sig):
    return co.process_streams(model_blob, sig, [(0.0, 0.0, 0, 0.0)] * len(CONTROLS))


@pytest.fixture(scope="module")
def oracle_on(model_blob, sig):
    return co.process_streams(model_blob, sig, CONTROLS)


def test_oracle_without_controls_is_the_plain_oracle(oracle_model, sig, oracle_off):
    plain = po.process_streams_trace(oracle_model, sig, margin=True)
    for a, b in zip(plain, oracle_off):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("thr,hold,gain", [(0.55, 0, 0.0), (0.55, 3, 0.0), (0.6, 10, 0.25), (1.0, 0, 0.5), (0.5, 2, 1.0)])
def test_oracle_gate_is_the_numpy_transliteration(model_blob, sig, oracle_off, thr, hold, gain):
    """gate only: the oracle's output is its ungated output times the NumPy ramp of its own VAD, bit for bit"""
    out, vad = co.process_streams(model_blob, sig, [(0.0, thr, hold, gain)] * len(CONTROLS))[:2]
    ref, rvad = oracle_off[:2]
    assert np.array_equal(vad, rvad)
    for s in range(len(CONTROLS)):
        want = cr.gated(ref[s], rvad[s], thr, hold, gain)
        assert np.array_equal(out[s].view(np.uint32), want.view(np.uint32)), s


def test_gate_and_floor_are_not_vacuous(oracle_off, oracle_on):
    ref, rvad = oracle_off[:2]
    g1, _, _ = cr.gate_gains(rvad[1], *CONTROLS[1][1:])
    g3, _, _ = cr.gate_gains(rvad[3], *CONTROLS[3][1:])
    assert (g1 == 0).sum() >= 3 and (g1 == 1).sum() >= 3, g1  # stream 1 closes and opens
    assert (g3 != 1).sum() >= 1 and (g3 == 1).sum() >= 3, g3
    out, _, _, _, sil = oracle_on[:5]
    frames = np.abs(out[2] - ref[2]).reshape(NF, 480).max(1) > 0
    assert frames[sil[2] == 0].mean() > 0.5  # the floor changes most non-silent frames


# ---- K4 / K5 under the host emulation --------------------------------------------------------------------------------
def emu_run(blob, x, controls, chunk=CHUNK):
    L = emu_lib()
    state = np.zeros((x.shape[0], L.ns_emu_state_floats()), np.float32)
    for s, c in enumerate(controls):
        L.ns_emu_set_controls(state.ctypes.data, s, *c)
    return emu_process(blob, x, chunk=chunk, state=state)


@pytest.fixture(scope="module")
def emu_off(model_blob, sig):
    return emu_run(model_blob, sig, [(0.0, 0.0, 0, 0.0)] * len(CONTROLS))


@pytest.fixture(scope="module")
def emu_on(model_blob, sig):
    return emu_run(model_blob, sig, CONTROLS)


def test_emulated_controls_leave_every_decision_alone(emu_off, emu_on):
    """pitch index, pitch gain, silence gate and VAD are those of the run without controls, bit for bit"""
    for tap in (TAP_INDEX, TAP_GAIN, TAP_SILENCE, TAP_VAD):
        assert np.array_equal(emu_on[2][:, :, tap].view(np.uint32), emu_off[2][:, :, tap].view(np.uint32)), tap
    assert np.array_equal(emu_on[1], emu_off[1])
    assert np.array_equal(emu_on[0][0], emu_off[0][0])  # the stream without controls


def test_emulated_gate_is_the_numpy_transliteration(emu_off, emu_on):
    """stream 1 (gate only, hold across the 8-frame chunks): its ungated output times the NumPy ramp, bit for bit"""
    want = cr.gated(emu_off[0][1], emu_off[1][1], *CONTROLS[1][1:])
    assert np.array_equal(emu_on[0][1].view(np.uint32), want.view(np.uint32))


def test_emulated_gate_carry_is_in_the_state(emu_on):
    """the controls and the gate's carry sit in the state row (ns_common.h kStCtl*, kStGate*) after the last chunk"""
    st = emu_on[3]
    for s, c in enumerate(CONTROLS):
        g, left, g_last = cr.gate_gains(emu_on[1][s], *c[1:])
        closed = bool(g[-1] != 1)  # the gate gains of CONTROLS are below 1
        sti = st[s].view(np.int32)
        assert st[s, ST_CTL:ST_CTL + 4].tolist() == [np.float32(c[0]), np.float32(c[1]), st[s, ST_CTL + 2], np.float32(c[3])]
        assert sti[ST_CTL + 2] == c[2]
        assert (sti[ST_CTL + 4], sti[ST_CTL + 5], st[s, ST_CTL + 6]) == (left, int(closed), g_last if closed else 0.0)


def test_emulated_controls_match_the_oracle(oracle_on, emu_on):
    """every stream under its own controls: gate decisions as the oracle's, samples within the tolerances"""
    ref, rvad, rpi, rpg, rsil, margin = oracle_on
    out, vad, dbg, _ = emu_on
    assert np.array_equal(dbg[:, :, TAP_INDEX].astype(np.int32), rpi)
    assert np.array_equal(dbg[:, :, TAP_GAIN].view(np.uint32), rpg.view(np.uint32))
    assert np.array_equal(dbg[:, :, TAP_SILENCE].astype(np.int32), rsil)
    assert np.abs(vad - rvad).max() <= TOL_VAD
    for s, c in enumerate(CONTROLS):
        near = np.flatnonzero(np.abs(rvad[s] - np.float32(c[1])) <= TOL_VAD) if c[1] > 0 else []
        upto = near[0] if len(near) else NF  # decisions after a frame at the threshold may differ
        assert np.array_equal(cr.gate_gains(vad[s], *c[1:])[0][:upto], cr.gate_gains(rvad[s], *c[1:])[0][:upto]), s
    risky = margin < BRANCH_EPS
    risky[:, 1:] |= risky[:, :-1].copy()
    err = np.abs(out.astype(np.float64) - ref).reshape(len(CONTROLS), NF, 480).max(2)
    assert err[~risky].max() <= TOL_MAX_ABS, err[~risky].max()
    assert snr_db(ref, out) >= TOL_SNR_DB
