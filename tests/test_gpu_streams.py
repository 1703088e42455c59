"""GPU: streams of a batch that advance independently -- subset calls, per-stream reset, save and load of single streams
(include/crispy_ns.h, the per-stream section).  Every check is bit-exact except the one against the oracle: a stream's
bits in a subset call are those of the same stream in a batch of its own, whoever else shares the call."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import crispy_b200 as cb  # noqa: E402
from crispy_b200 import _lib  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from tests.util import assert_parity, make_signal  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 16  # engine chunk for these tests: calls of 1, 15, 16, 17, 33 ... frames are 1, 2, 3 chunks, odd and even
EINVAL = -1


@pytest.fixture(scope="module")
def model():
    return cb.Model.synthetic(0)


@pytest.fixture(autouse=True)
def small_chunks(monkeypatch):
    monkeypatch.setenv("CRISPY_NS_CHUNK_FRAMES", str(CHUNK))


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _rows(state: bytes, n: int):
    """save_state payload (after its 16-byte header) as one bytes object per stream"""
    row = (len(state) - 16) // n
    return [state[16 + i * row:16 + (i + 1) * row] for i in range(n)]


def make_schedule(n_streams: int, n_calls: int, seed: int):
    """[(ids or None for a full call, n_frames)]: random subsets in random order, frame counts at and around the chunk"""
    rng = np.random.default_rng(seed)
    lengths = [1, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK, 2 * CHUNK + 1, 3 * CHUNK, 5]
    sched = []
    for c in range(n_calls):
        nf = lengths[c % len(lengths)] if c < len(lengths) else int(rng.choice(lengths))
        if c % 4 == 3:
            sched.append((None, nf))
        else:
            m = int(rng.integers(1, n_streams + 1))
            sched.append((rng.permutation(n_streams)[:m].tolist(), nf))
    return sched


class Variant:
    """input / output formats of one run: 'f32' (16-bit scale), 'unit' (UNIT_SCALE + volume), 'i16_mix' (PCM16 in,
    MIX_STEREO_I16 + app out)"""

    def __init__(self, kind: str, n_streams: int, n_frames: int):
        self.kind = kind
        x = make_signal(n_streams, n_frames, seed=1234)
        self.app = None
        if kind == "f32":
            self.x, self.kw = x, {"unit_scale": False}
        elif kind == "unit":
            self.x, self.kw = (x / np.float32(32768.0)).astype(np.float32), {"unit_scale": True, "volume": 0.7}
        else:
            self.x = np.clip(np.rint(x), -32768, 32767).astype(np.int16)
            self.app = (make_signal(n_streams, n_frames, seed=99) / np.float32(65536.0)).astype(np.float32)
            self.kw = {"unit_scale": False, "mix_stereo_i16": True}

    def args(self, ids, a, b):
        kw = dict(self.kw)
        if self.app is not None:
            kw["app"] = _dev(self.app[ids, a * 480:b * 480])
        return _dev(self.x[ids, a * 480:b * 480]), kw


def run_schedule(den, var: Variant, sched, n_streams: int, host: bool = False):
    """Feed every stream its next frames per the schedule; returns per-stream concatenated (out, vad) and positions."""
    pos = np.zeros(n_streams, np.int64)
    outs = [[] for _ in range(n_streams)]
    vads = [[] for _ in range(n_streams)]
    for ids, nf in sched:
        full = ids is None
        ids = list(range(n_streams)) if full else ids
        x = np.stack([var.x[s, pos[s] * 480:(pos[s] + nf) * 480] for s in ids])
        kw = dict(var.kw)
        if var.app is not None:
            kw["app"] = np.stack([var.app[s, pos[s] * 480:(pos[s] + nf) * 480] for s in ids])
        if host:
            if "app" in kw:
                kw["app"] = torch.from_numpy(kw["app"]).pin_memory()
            xt = torch.from_numpy(x).pin_memory()
            o, v = (den.process_streams_host(xt, **kw) if full else den.process_streams_subset_host(ids, xt, **kw))
        else:
            if "app" in kw:
                kw["app"] = _dev(kw["app"])
            o, v = den.process_streams(_dev(x), **kw) if full else den.process_streams_subset(ids, _dev(x), **kw)
        o, v = o.cpu(), v.cpu()
        for i, s in enumerate(ids):
            outs[s].append(o[i])
            vads[s].append(v[i])
            pos[s] += nf
    return [torch.cat(o) for o in outs], [torch.cat(v) for v in vads], pos


def reference(model, var: Variant, s: int, n_frames: int):
    """stream s fed alone, in one call, to a batch of its own"""
    ref = cb.BatchDenoiser(1, model)
    x, kw = var.args([s], 0, n_frames)
    o, v = ref.process_streams(x, **kw)
    return o[0].cpu(), v[0].cpu(), ref.save_streams([0])


# ---- 1. random schedule against separate batches ---------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["f32", "unit", "i16_mix"])
def test_random_schedule_equals_separate_batches(model, kind):
    n = 37
    sched = make_schedule(n, 12, seed={"f32": 1, "unit": 2, "i16_mix": 3}[kind])
    assert {nf for _, nf in sched} >= {1, CHUNK - 1, CHUNK + 1, 2 * CHUNK + 1, 3 * CHUNK}
    var = Variant(kind, n, sum(nf for _, nf in sched))
    den = cb.BatchDenoiser(n, model)
    launches0 = den.info["launches"]
    outs, vads, pos = run_schedule(den, var, sched, n)
    assert den.frames_done == sum(nf for ids, nf in sched if ids is None)
    chunks = sum(-(-nf // CHUNK) for _, nf in sched)
    assert den.info["launches"] - launches0 == 7 * chunks
    saved = den.save_streams(range(n))
    rec = cb.stream_state_size()
    for s in range(n):
        o, v, st = reference(model, var, s, int(pos[s]))
        assert torch.equal(outs[s], o), (kind, s)
        assert torch.equal(vads[s], v), (kind, s)
        assert saved[s * rec:(s + 1) * rec] == st, (kind, s)


# ---- 2. identity subset -----------------------------------------------------------------------------------------------
def test_identity_subset_equals_full_call(model):
    """ids 0..n-1 in order: same output and VAD as a full call.  After an even number of chunks the state rows are the
    same bytes too; after an odd number the subset call has advanced the chunk counter once more (parity invariant), so
    the two copies of synthesis_mem sit swapped and the stream records are compared instead.  frames_done moves only
    for the full call."""
    n = 9
    x = make_signal(n, 7 * CHUNK + 1, seed=5)
    a, b = cb.BatchDenoiser(n, model), cb.BatchDenoiser(n, model)
    f0 = 0
    for nf, even in ((2 * CHUNK, True), (CHUNK + 1, True), (CHUNK, False), (3 * CHUNK, False)):
        oa, va = a.process_streams(_dev(x[:, f0 * 480:(f0 + nf) * 480]), unit_scale=False)
        ob, vb = b.process_streams_subset(list(range(n)), _dev(x[:, f0 * 480:(f0 + nf) * 480]), unit_scale=False)
        f0 += nf
        assert torch.equal(oa, ob) and torch.equal(va, vb), nf
        assert a.save_streams(range(n)) == b.save_streams(range(n))
        if even and f0 == 3 * CHUNK + 1:
            assert a.save_state()[16:] == b.save_state()[16:]
    assert b.frames_done == 0 and a.frames_done == f0


# ---- 3. bystanders ----------------------------------------------------------------------------------------------------
def test_streams_outside_a_subset_keep_their_state_bits(model):
    n = 12
    x = make_signal(n, 200, seed=6)
    den = cb.BatchDenoiser(n, model)
    den.process_streams(_dev(x[:, :20 * 480]), unit_scale=False)
    active = [3, 7, 1]
    f0 = 20
    for nf in (CHUNK, 2 * CHUNK, 1, CHUNK + 1):  # odd, even, odd, even chunk counts
        before = _rows(den.save_state(), n)
        den.process_streams_subset(active, _dev(x[active, f0 * 480:(f0 + nf) * 480]), unit_scale=False)
        f0 += nf
        after = _rows(den.save_state(), n)
        for s in range(n):
            if s in active:
                assert before[s] != after[s], (nf, s)
            else:
                assert before[s] == after[s], (nf, s)


# ---- 4. reset_streams -------------------------------------------------------------------------------------------------
def test_reset_streams_gives_a_fresh_stream_and_leaves_the_neighbours(model):
    n = 6
    x = make_signal(n, 60, seed=7)
    y = make_signal(1, 40, seed=8)
    den = cb.BatchDenoiser(n, model)
    den.process_streams(_dev(x[:, :CHUNK * 480]), unit_scale=False)
    before = _rows(den.save_state(), n)
    den.reset_streams([2, 4])
    after = _rows(den.save_state(), n)
    assert all(before[s] == after[s] for s in (0, 1, 3, 5))
    assert after[2] == after[4] == bytes(len(after[2]))
    ref = cb.BatchDenoiser(1, model)
    want, wv = ref.process_streams(_dev(y), unit_scale=False)
    got, gv = den.process_streams_subset([2], _dev(y), unit_scale=False)
    assert torch.equal(got, want) and torch.equal(gv, wv)
    # a neighbour continues as if nothing had happened
    alone = cb.BatchDenoiser(1, model)
    w0, _ = alone.process_streams(_dev(x[:1, :(CHUNK + 20) * 480]), unit_scale=False)
    g0, _ = den.process_streams_subset([0], _dev(x[:1, CHUNK * 480:(CHUNK + 20) * 480]), unit_scale=False)
    assert torch.equal(g0[0], w0[0, CHUNK * 480:])


def test_reset_streams_is_ordered_before_a_call_on_another_cuda_stream(model):
    """The reset is enqueued on one CUDA stream behind a long sleep; the next call is made at once on another stream.
    It must still see the fresh state."""
    n = 5
    x = make_signal(n, 40, seed=9)
    y = make_signal(1, 30, seed=10)
    den = cb.BatchDenoiser(n, model)
    den.process_streams(_dev(x[:, :20 * 480]), unit_scale=False)
    want, _ = cb.BatchDenoiser(1, model).process_streams(_dev(y), unit_scale=False)
    yd = _dev(y)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(100_000_000)
        den.reset_streams([3])
    with torch.cuda.stream(s2):
        got, _ = den.process_streams_subset([3], yd, unit_scale=False)
    s2.synchronize()
    assert torch.equal(got, want)


# ---- 5. save_streams / load_streams -----------------------------------------------------------------------------------
def test_a_stream_moves_to_another_batch_at_the_other_parity(model):
    x = make_signal(11, 2 * CHUNK + 40, seed=11)
    a = cb.BatchDenoiser(11, model)
    a.process_streams(_dev(x[:, :CHUNK * 480]), unit_scale=False)  # one chunk: odd
    b = cb.BatchDenoiser(20, model)
    b.process_streams(_dev(make_signal(20, 2 * CHUNK, seed=12)), unit_scale=False)  # two chunks: even
    blob = a.save_streams([3])
    assert len(blob) == cb.stream_state_size()
    others = _rows(b.save_state(), 20)
    b.load_streams([7], blob)
    after = _rows(b.save_state(), 20)
    assert all(others[s] == after[s] for s in range(20) if s != 7)
    assert b.save_streams([7]) == blob
    cont = _dev(x[3:4, CHUNK * 480:])
    got, gv = b.process_streams_subset([7], cont, unit_scale=False)
    whole, wv = cb.BatchDenoiser(1, model).process_streams(_dev(x[3:4]), unit_scale=False)
    assert torch.equal(got[0], whole[0, CHUNK * 480:]) and torch.equal(gv[0], wv[0, CHUNK:])
    # truncated, foreign and mis-sized blobs: refused, state untouched
    L = _lib.lib()
    snap = b.save_state()
    ids = (C.c_int * 1)(7)
    for bad in (blob[:-1], b"X" + blob[1:], blob + blob, bytes(len(blob))):
        assert L.crispy_ns_batch_load_streams(b._h, ids, 1, bad, len(bad)) == EINVAL
    assert b.save_state() == snap


# ---- 6. host and device -----------------------------------------------------------------------------------------------
def test_host_subset_path_equals_device_subset_path(model, monkeypatch):
    n = 13
    sched = make_schedule(n, 10, seed=21)
    var = Variant("unit", n, sum(nf for _, nf in sched))
    dev = cb.BatchDenoiser(n, model)
    od, vd, _ = run_schedule(dev, var, sched, n)
    monkeypatch.setenv("CRISPY_NS_HOST_CHUNK_FRAMES", "7")  # several host chunks per call, not a multiple of the chunk
    host = cb.BatchDenoiser(n, model)
    oh, vh, _ = run_schedule(host, var, sched, n, host=True)
    for s in range(n):
        assert torch.equal(od[s], oh[s]) and torch.equal(vd[s], vh[s]), s
    assert dev.save_streams(range(n)) == host.save_streams(range(n))  # chunked differently: records, not raw rows


# ---- 7. both biquad forms ---------------------------------------------------------------------------------------------
def test_both_forms_of_the_biquad_kernel_give_the_same_bits_on_subset_calls(model, monkeypatch):
    """K0's form follows the call's stream count (exclusive + parallel in time up to 768 streams, one recursion warp
    above); $CRISPY_NS_HP_EXCLUSIVE / $CRISPY_NS_HP_PAR force each form, which covers both sides of 768 at this size."""
    n = 40
    sched = make_schedule(n, 8, seed=31)
    var = Variant("f32", n, sum(nf for _, nf in sched))
    res = []
    for excl, par in (("1", "1"), ("1", "0"), ("0", "0"), ("0", "1")):
        monkeypatch.setenv("CRISPY_NS_HP_EXCLUSIVE", excl)
        monkeypatch.setenv("CRISPY_NS_HP_PAR", par)
        den = cb.BatchDenoiser(n, model)
        o, v, _ = run_schedule(den, var, sched, n)
        res.append((o, v, den.save_state()))
    for o, v, st in res[1:]:
        assert all(torch.equal(a, b) for a, b in zip(o, res[0][0]))
        assert all(torch.equal(a, b) for a, b in zip(v, res[0][1]))
        assert st == res[0][2]


# ---- 8. tcgen05 recurrent core ----------------------------------------------------------------------------------------
def test_tc5_core_subset_calls_equal_tc5_separate_batches(model, monkeypatch):
    monkeypatch.setenv("CRISPY_NS_RNN", "tc5")
    n = 19
    sched = make_schedule(n, 8, seed=41)
    var = Variant("f32", n, sum(nf for _, nf in sched))
    den = cb.BatchDenoiser(n, model)
    assert den.info["rnn_streams_per_cta"] == 128
    outs, vads, pos = run_schedule(den, var, sched, n)
    for s in range(n):
        o, v, _ = reference(model, var, s, int(pos[s]))
        assert torch.equal(outs[s], o) and torch.equal(vads[s], v), s


# ---- 9. oracle --------------------------------------------------------------------------------------------------------
def test_subset_schedule_matches_the_oracle(oracle_model, model):
    n = 37
    sched = make_schedule(n, 12, seed=1)
    var = Variant("f32", n, sum(nf for _, nf in sched))
    den = cb.BatchDenoiser(n, model)
    outs, vads, pos = run_schedule(den, var, sched, n)
    for s in (0, 5, 18, 36):
        ref, rvad = po.process_streams(oracle_model, var.x[s:s + 1, :pos[s] * 480])
        assert_parity(ref, outs[s].numpy()[None, :], rvad, vads[s].numpy()[None, :], f"subset stream {s}")


# ---- 10. argument errors ----------------------------------------------------------------------------------------------
def test_bad_arguments_are_refused_and_change_nothing(model):
    n = 8
    den = cb.BatchDenoiser(n, model)
    x = make_signal(n, 40, seed=51)
    den.process_streams(_dev(x[:, :CHUNK * 480]), unit_scale=False)
    L = _lib.lib()
    buf = torch.zeros((n, 4 * 480), device="cuda")
    out = torch.zeros_like(buf)
    ip = lambda *v: (C.c_int * max(len(v), 1))(*v)  # noqa: E731
    snap, fd = den.save_state(), den.frames_done
    rec = cb.stream_state_size()

    def sub(ids, m, flags=0, h=den._h):
        return L.crispy_ns_process_streams_subset(h, ids, m, buf.data_ptr(), out.data_ptr(), None, None, 4, 1920, 1920,
                                                  0, 0, flags, 1.0, None)
    assert sub(ip(0), 1, h=None) == EINVAL
    assert sub(ip(0), -1) == EINVAL
    assert sub(ip(*range(n + 1)), n + 1) == EINVAL
    assert sub(ip(0, n), 2) == EINVAL
    assert sub(ip(0, -1), 2) == EINVAL
    assert sub(ip(2, 5, 2), 3) == EINVAL
    assert sub(None, 2) == EINVAL
    assert sub(ip(1), 1, flags=_lib.DROP_FIRST_FRAME) == EINVAL
    assert L.crispy_ns_process_streams_subset_host(den._h, ip(1, 1), 2, buf.cpu().data_ptr(), None, None, None, 4, 1920,
                                                   1920, 0, 0, 0, 1.0) == EINVAL
    assert L.crispy_ns_batch_reset_streams(den._h, ip(9), 1, None) == EINVAL
    assert L.crispy_ns_batch_reset_streams(None, ip(1), 1, None) == EINVAL
    assert L.crispy_ns_batch_reset_streams(den._h, ip(3, 3), 2, None) == EINVAL
    small = C.create_string_buffer(2 * rec)
    assert L.crispy_ns_batch_save_streams(den._h, ip(1, 2), 2, small, 2 * rec - 1) == EINVAL
    assert L.crispy_ns_batch_save_streams(den._h, ip(1, 1), 2, small, 2 * rec) == EINVAL
    good = den.save_streams([1, 2])
    assert L.crispy_ns_batch_load_streams(den._h, ip(1, 2), 2, good, len(good) - rec) == EINVAL
    assert L.crispy_ns_batch_load_streams(den._h, ip(1, 1), 2, good, len(good)) == EINVAL
    assert L.crispy_ns_batch_load_streams(den._h, ip(1, 2), 2, good[:rec] + b"Y" + good[rec + 1:], len(good)) == EINVAL
    # empty calls touch nothing, null pointers included
    assert sub(None, 0) == 0
    assert L.crispy_ns_process_streams_subset(den._h, ip(1), 1, None, None, None, None, 0, 0, 0, 0, 0, 0, 1.0, None) == 0
    assert L.crispy_ns_batch_reset_streams(den._h, None, 0, None) == 0
    torch.cuda.synchronize()
    assert den.save_state() == snap and den.frames_done == fd
    # after a per-stream operation a full call cannot drop "the" first frame; a whole-batch reset lifts that
    den.process_streams_subset([1], _dev(x[1:2, :480]), unit_scale=False)
    with pytest.raises(cb.CrispyNsError, match="DROP_FIRST_FRAME"):
        den.process_streams(_dev(x[:, :480]), unit_scale=False, drop_first_frame=True)
    den.reset()
    o, _ = den.process_streams(_dev(x[:, :2 * 480]), unit_scale=False, drop_first_frame=True)
    assert o.shape[1] == 480


# ---- 11. C consumer ---------------------------------------------------------------------------------------------------
def test_c_consumer_of_the_per_stream_calls(tmp_path):
    exe = str(tmp_path / "streams_smoke")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c_abi", "streams_smoke.c"), "-L" + lib_dir, "-lcrispy_ns", "-lm",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "streams_smoke: ok" in r.stdout, r.stdout + r.stderr
