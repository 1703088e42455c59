"""CPU: the model's numerics setting (crispy_ns_model_set_numerics) at the C boundary, the oracle's f32 biquad
(tests/numerics_oracle.py), and the pitch and biquad kernels under every combination of sum order and biquad form, run
under the host SIMT emulation (tests/emu/ns_emu_numerics.cpp) against the oracle under the same combination."""
import atexit
import ctypes as C
import itertools
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import crispy_b200 as cb
from crispy_b200 import _lib, build
from tests import numerics_oracle as no
from tests.util import CSRC, EMU_DIR, assert_parity, make_signal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL, ENODEV = -1, -2
COMBOS = [s | b for s, b in itertools.product((_lib.SUM_SEQUENTIAL, _lib.SUM_DOT4, _lib.SUM_DOT4_XCORR), (0, _lib.BIQUAD_F32))]
TAP_GAIN, TAP_INDEX, TAP_SILENCE = 130, 132, 133  # ns_common.h debug taps


@pytest.fixture(scope="module", autouse=True)
def built():
    build.build()


# ---- the C ABI -------------------------------------------------------------------------------------------------------
def test_numerics_constants_match_the_header():
    h = open(os.path.join(ROOT, "include", "crispy_ns.h")).read()
    for name in ("SUM_SEQUENTIAL", "SUM_DOT4", "SUM_DOT4_XCORR", "SUM_MASK", "BIQUAD_F32"):
        expr = re.search(r"CRISPY_NS_%s\s*=\s*([^,/\n]+)" % name, h).group(1).strip().replace("u", "")
        assert eval(expr) == getattr(_lib, name), name


def test_default_is_zero_and_null_models_give_zero():
    L = _lib.lib()
    assert cb.Model.synthetic(3).numerics == 0
    assert L.crispy_ns_model_numerics(None) == 0
    assert L.crispy_ns_model_set_numerics(None, 0) == EINVAL
    blob = cb.Model.synthetic(3).to_bytes()
    assert cb.Model.from_bytes(blob).numerics == 0


@pytest.mark.parametrize("numerics", COMBOS)
def test_set_and_get_round_trip_and_the_blob_does_not_carry_it(numerics):
    m = cb.Model.synthetic(5)
    plain = m.to_bytes()
    m.numerics = numerics
    assert m.numerics == numerics
    assert m.to_bytes() == plain
    assert cb.Model.from_bytes(m.to_bytes()).numerics == 0


@pytest.mark.parametrize("bad", [3, 3 | _lib.BIQUAD_F32, 4, 8, 1 << 5, 1 << 8, 1 << 31, 0xFFFFFFFF])
def test_unknown_bits_and_sum_order_3_are_refused_and_change_nothing(bad):
    m = cb.Model.synthetic(0)
    m.numerics = _lib.SUM_DOT4
    assert _lib.lib().crispy_ns_model_set_numerics(m._h, bad) == EINVAL
    assert b"model_set_numerics" in _lib.lib().crispy_ns_last_error()
    assert m.numerics == _lib.SUM_DOT4
    with pytest.raises(cb.CrispyNsError):
        m.numerics = bad


def test_new_symbols_are_exported():
    assert {"crispy_ns_model_set_numerics", "crispy_ns_model_numerics"} <= set(_lib.SYMBOLS)
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\b(crispy_ns_\w+)$", nm, flags=re.M))
    assert set(_lib.SYMBOLS) <= exported


def test_handles_from_a_numerics_model_follow_the_enodev_contract_without_a_device():
    if cb.device_count() > 0:
        pytest.skip("a CUDA device is present: the handles are exercised by tests/test_gpu_numerics.py")
    L = _lib.lib()
    m = cb.Model.synthetic(0)
    m.numerics = _lib.SUM_DOT4_XCORR | _lib.BIQUAD_F32
    h = C.c_void_p()
    assert L.crispy_ns_batch_create(m._h, 0, 4, C.byref(h)) == ENODEV
    assert L.crispy_ns_create(m._h, 0, C.byref(h)) == ENODEV
    devs = (C.c_int * 1)(0)
    assert L.crispy_ns_multi_create(m._h, devs, 1, 4, C.byref(h)) == ENODEV
    assert not h.value


def test_cpp_model_exposes_the_setting(tmp_path):
    src = tmp_path / "numerics.cpp"
    src.write_text(r"""
#include <crispy_ns.hpp>
#include <cstdio>
int main() {
  crispy::Model m = crispy::Model::synthetic(1);
  if (m.numerics() != 0) return 1;
  m.set_numerics(CRISPY_NS_SUM_DOT4 | CRISPY_NS_BIQUAD_F32);
  if (m.numerics() != (CRISPY_NS_SUM_DOT4 | CRISPY_NS_BIQUAD_F32)) return 2;
  try {
    m.set_numerics(3);
    return 3;
  } catch (const std::exception &) {
  }
  std::printf("numerics ok\n");
  return m.numerics() == (CRISPY_NS_SUM_DOT4 | CRISPY_NS_BIQUAD_F32) ? 0 : 4;
}
""")
    exe = str(tmp_path / "numerics")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                           "-L" + lib_dir, "-lcrispy_ns", "-Wl,-rpath," + lib_dir, "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "numerics ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


# ---- the oracle's f32 biquad -----------------------------------------------------------------------------------------
def _biquad_f32_numpy(x, m0=0.0, m1=0.0):
    """the oracle's biquad in f32 arithmetic (tests/numerics_oracle.py), in NumPy float32: every product and sum rounded"""
    b0, b1 = np.float32(-2.0), np.float32(1.0)
    a0, a1 = np.float32(-1.99599), np.float32(0.99600)
    m0, m1 = np.float32(m0), np.float32(m1)
    y = np.empty(len(x), np.float32)
    for i, xi in enumerate(x.astype(np.float32)):
        yi = np.float32(xi + m0)
        m0 = np.float32(m1 + np.float32(np.float32(b0 * xi) - np.float32(a0 * yi)))
        m1 = np.float32(np.float32(b1 * xi) - np.float32(a1 * yi))
        y[i] = yi
    return y, m0, m1


def test_oracle_f32_biquad_is_the_float32_transliteration_and_not_the_f64_form():
    x = make_signal(1, 6)[0]
    x[700:900] = 0.0
    y32, (m0, m1) = no.highpass_f32(x, mem=(1.5, -0.75))
    want, w0, w1 = _biquad_f32_numpy(x, 1.5, -0.75)
    assert np.array_equal(y32.view(np.uint32), want.view(np.uint32))
    assert (np.float32(m0), np.float32(m1)) == (w0, w1)
    from tests.test_emu_parity import _biquad_reference  # upstream's f64-intermediate biquad, line for line
    y64, _, _ = _biquad_reference(x, 1.5, -0.75)
    differ = float(np.mean(y64 != y32))
    assert differ > 0.3, differ  # the two forms part within a few samples and never meet again (ns_pipe.cuh K0)


# ---- the kernels under the host emulation ----------------------------------------------------------------------------
_emu = None


def emu_lib():
    """tests/emu/ns_emu_numerics.cpp (the emulation of tests/emu/ns_emu.cpp plus a numerics entry point), built once per
    process into a temporary directory"""
    global _emu
    if _emu is None:
        d = tempfile.mkdtemp(prefix="crispy_emu_numerics_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libns_emu_numerics.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, os.path.join(EMU_DIR, "ns_emu_numerics.cpp"),
                               os.path.join(CSRC, "ns_host.cpp")])
        _emu = C.CDLL(so)
    return _emu


def emu_run(blob, x, numerics, chunk=8):
    L = emu_lib()
    L.ns_emu_process_numerics.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                          C.c_longlong, C.c_int, C.c_uint, C.c_float, C.c_int, C.c_uint]
    x = np.ascontiguousarray(x, dtype=np.float32)
    ns, n = x.shape
    nf = n // 480
    out = np.zeros_like(x)
    vad = np.zeros((ns, nf), np.float32)
    dbg = np.zeros((ns, nf, L.ns_emu_dbg_floats()), np.float32)
    state = np.zeros((ns, L.ns_emu_state_floats()), np.float32)
    rc = L.ns_emu_process_numerics(blob, len(blob), x.ctypes.data, out.ctypes.data, vad.ctypes.data, None,
                                   state.ctypes.data, dbg.ctypes.data, ns, nf, n, n, 0, chunk, 0, 1.0, 0, numerics)
    assert rc == 0, rc
    return out, vad, dbg, state


@pytest.fixture(scope="module")
def sig():
    return make_signal(3, 28)


@pytest.fixture(scope="module")
def oracle_runs(model_blob, sig):
    return {nm: no.process_streams_trace(model_blob, sig, nm, n_threads=3) for nm in COMBOS}


@pytest.fixture(scope="module")
def emu_runs(model_blob, sig):
    return {nm: emu_run(model_blob, sig, nm) for nm in COMBOS}


@pytest.mark.parametrize("numerics", COMBOS)
def test_emulated_kernels_match_the_oracle_under_the_same_numerics(oracle_runs, emu_runs, numerics):
    """pitch index, pitch gain and silence gate bit for bit; samples within north_star"""
    ref, rvad, rpi, rpg, rsil = oracle_runs[numerics]
    out, vad, dbg, _ = emu_runs[numerics]
    assert np.array_equal(dbg[:, :, TAP_INDEX].astype(np.int32), rpi)
    assert np.array_equal(dbg[:, :, TAP_GAIN].view(np.uint32), rpg.view(np.uint32))
    assert np.array_equal(dbg[:, :, TAP_SILENCE].astype(np.int32), rsil)
    assert rsil.sum() > 0  # stream 1's digital silence reaches the gate
    assert_parity(ref, out, rvad, vad, f"numerics {numerics}")


def test_numerics_zero_entry_point_is_the_existing_one(model_blob, sig, emu_runs):
    from tests.util import emu_process
    out, vad, dbg, st = emu_process(model_blob, sig, chunk=8)
    o0, v0, d0, s0 = emu_runs[0]
    assert np.array_equal(out, o0) and np.array_equal(vad, v0) and np.array_equal(dbg, d0) and np.array_equal(st, s0)


def test_the_switches_are_not_vacuous(oracle_runs, emu_runs):
    """The changed inner products feed every frame's pitch gain, so dot4 moves the gain's last bits in most frames even
    where no index flips: a kernel that ignored the switch would fail the bit-exact comparison above.  Measured on this
    input (3 streams x 28 frames, no index flips): 89 % of frames under DOT4, 93 % under DOT4_XCORR."""
    g0 = oracle_runs[0][3]
    for pol in (_lib.SUM_DOT4, _lib.SUM_DOT4_XCORR):
        share = float(np.mean(oracle_runs[pol][3].view(np.uint32) != g0.view(np.uint32)))
        assert share > 0.8, (pol, share)
        emu_share = float(np.mean(emu_runs[pol][2][:, :, TAP_GAIN].view(np.uint32) !=
                                  emu_runs[0][2][:, :, TAP_GAIN].view(np.uint32)))
        assert emu_share == share
    # DOT4_XCORR changes the autocorrelation and the coarse search as well: their sums differ from DOT4's
    assert not np.array_equal(oracle_runs[_lib.SUM_DOT4][3], oracle_runs[_lib.SUM_DOT4_XCORR][3])
    # the f32 biquad changes every sample after the first few, hence the output
    assert not np.array_equal(emu_runs[_lib.BIQUAD_F32][0], emu_runs[0][0])


def test_emulated_f32_biquad_is_the_float32_transliteration(model_blob):
    x = (2500.0 * np.random.default_rng(4).standard_normal((2, 4 * 480))).astype(np.float32)
    hp = emu_lib().ns_emu_state_hp_offset()
    _, _, _, st = emu_run(model_blob, x, _lib.BIQUAD_F32, chunk=3)
    for s in range(2):
        y, m0, m1 = _biquad_f32_numpy(x[s])
        assert st[s, hp:hp + 2].view(np.uint32).tolist() == [np.float32(m0).view(np.uint32), np.float32(m1).view(np.uint32)]
        assert np.array_equal(st[s, :1440].view(np.uint32), y[-1440:].view(np.uint32))  # the high-passed history
