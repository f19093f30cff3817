"""The reference's own test-suite, as seen from the native library: every call its unmodified Python layer makes while
the suite runs, replayed against another library with the reference ABI.

tests/golden/reference_suite_abi.json holds each hyperscan() and check_patterns() call the reference's
hypergrep/test/test_hypergrep.py made (arguments as passed through ctypes) and the answer that let the suite pass:
return code and every callback batch of (id, line_number, line), batch boundaries included.  A library that gives the
same answers to the same calls passes the reference's suite under the reference's own Python layer.  The CPU legs pin
the oracle and the host logic to those answers; the GPU leg is the drop-in acceptance test for libgpugrep.so.
tools/record_reference_abi.py regenerates the file from a reference checkout.
"""

import ctypes
import json
import os

import pytest

from oracle_api import CALLBACK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "reference_suite_abi.json"), encoding="utf-8") as _handle:
    _RECORDED = json.load(_handle)


def _set(call: dict):
    n = len(call["patterns"])
    return ((ctypes.c_char_p * n)(*[p.encode("latin-1") for p in call["patterns"]]), (ctypes.c_uint * n)(*call["flags"]),
            (ctypes.c_uint * n)(*call["ids"]), n)


def _replay(lib: ctypes.CDLL, fixture_dir: str) -> None:
    assert _RECORDED["suite_result"] == "75 passed"
    for call in _RECORDED["calls"]:
        where = f"{call['fn']} call of {call['tests']}"
        if call["fn"] == "check_patterns":
            assert lib.check_patterns(*_set(call)) == call["rc"], where
            continue
        batches = []

        def on_event(results, count, batches=batches):
            batches.append([[results[i].id, results[i].line_number, results[i].line.decode("latin-1")] for i in range(count)])

        path = os.path.join(fixture_dir, call["file"]["fixture"]).encode()
        rc = lib.hyperscan(path, *_set(call), CALLBACK(on_event), call["buffer_size"], call["buffer_count"],
                           ctypes.c_ulonglong(call["max_match_count"]))
        assert rc == call["rc"], where
        assert batches == call["batches"], where


def test_oracle_passes_reference_suite(oracle_lib, fixture_dir):
    _replay(oracle_lib, fixture_dir)


def test_host_logic_passes_reference_suite(hostmock_lib, fixture_dir):
    _replay(hostmock_lib, fixture_dir)


@pytest.mark.gpu
def test_libgpugrep_passes_reference_suite(gpu_lib, fixture_dir):
    _replay(gpu_lib, fixture_dir)
