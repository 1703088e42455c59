"""CPU: the per-stream calls of include/crispy_ns.h at the boundary (no batch handle can exist without a device, so the
argument rules that need none), the stream record size against the header, and the continuous-batching scheduler."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import crispy_b200 as cb
from crispy_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL = -1


@pytest.fixture(scope="module", autouse=True)
def built():
    build.build()


def test_per_stream_calls_refuse_a_null_handle_and_bad_arguments():
    L = _lib.lib()
    ids = (C.c_int * 2)(0, 1)
    buf = C.create_string_buffer(4 * 480 * 4)
    assert L.crispy_ns_process_streams_subset(None, ids, 2, buf, buf, None, None, 1, 480, 480, 0, 0, 0, 1.0, None) == EINVAL
    assert L.crispy_ns_process_streams_subset_host(None, ids, 2, buf, buf, None, None, 1, 480, 480, 0, 0, 0, 1.0) == EINVAL
    assert L.crispy_ns_batch_reset_streams(None, ids, 2, None) == EINVAL
    assert L.crispy_ns_batch_save_streams(None, ids, 2, buf, len(buf)) == EINVAL
    assert L.crispy_ns_batch_load_streams(None, ids, 2, buf, len(buf)) == EINVAL
    assert b"null handle" in L.crispy_ns_last_error()


def test_stream_record_size_matches_the_header_and_the_state_layout():
    h = open(os.path.join(ROOT, "include", "crispy_ns.h")).read()
    stated = int(re.search(r"([\d,]+) bytes in this build", h).group(1).replace(",", ""))
    common = open(os.path.join(ROOT, "crispy_b200", "csrc", "ns_common.h")).read()
    floats = int(re.search(r"kStateFloats = (\d+);", common).group(1))
    assert cb.stream_state_size() == stated == 16 + 4 * floats


def test_c_consumer_of_the_per_stream_calls_compiles_and_checks_arguments(tmp_path):
    exe = str(tmp_path / "streams_smoke")
    lib_dir = os.path.join(ROOT, "crispy_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c_abi", "streams_smoke.c"), "-L" + lib_dir, "-lcrispy_ns", "-lm",
                           "-Wl,-rpath," + lib_dir, "-o", exe])
    if cb.device_count() == 0:
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 0 and "argument checks ok" in r.stdout, r.stdout + r.stderr


def _sched():
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import continuous_batching as cbat
    return cbat


def test_scheduler_dry_run_counts():
    cbat = _sched()
    lengths = cbat.recording_lengths(300, 1.0, 20.0, 7)
    assert lengths.min() >= 6000 - 1 and lengths.max() <= 120000 + 1
    # arm A: every group runs to its longest recording
    groups, proc_a, useful = cbat.padded_schedule(lengths, 64, 1000)
    assert useful == lengths.sum()
    assert proc_a == sum(len(lengths[g:g + 64]) * lengths[g:g + 64].max() for g in range(0, 300, 64))
    assert [sum(c) for _, c in groups] == [lengths[g:g + 64].max() for g in range(0, 300, 64)]
    # arm B: every recording runs in its own slot to the end of the call it ends in, nothing more
    calls, proc_b, _ = cbat.continuous_schedule(lengths, 64, 1000)
    assert proc_b == sum((64 if ids is None else len(ids)) * 1000 for ids, _ in calls)
    assert useful <= proc_b < useful + 300 * 1000
    assert sum(len(r) for _, r in calls) == 300 - 64  # every recording after the first 64 refills a slot
    assert calls[-1][0] is not None  # the tail runs as subset calls
    # a by-hand case: two slots, recordings of 3, 1 and 0.5 calls: the third refills slot 1 after the first call and
    # is padded to the end of the second; the third call runs slot 0 alone
    calls, proc, useful = cbat.continuous_schedule(np.array([3000, 1000, 500]), 2, 1000)
    assert [c[0] for c in calls] == [None, None, [0]] and [c[1] for c in calls] == [[1], [], []]
    assert (proc, useful) == (5000, 4500)


def test_scheduler_dry_run_prints_its_utilisation():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "continuous_batching.py"), "--dry-run",
                        "--recordings", "500", "--slots", "128"], capture_output=True, text=True, check=True)
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["continuous_utilisation"] == res["useful_frames"] / res["continuous_processed_frames"]
    assert res["padded_utilisation"] == res["useful_frames"] / res["padded_processed_frames"]
    assert 0 < res["padded_utilisation"] < res["continuous_utilisation"] <= 1
