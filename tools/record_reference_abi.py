#!/usr/bin/env python3
"""Record what the reference's own test-suite asks of the native library into tests/golden/reference_suite_abi.json.

    python tools/record_reference_abi.py REFERENCE_CHECKOUT

Runs the reference's unmodified hypergrep/test/test_hypergrep.py with its loader hook (`_get_hyperscanner_lib`) pointed
at a recording proxy of the CPU oracle (oracle/_build/liboracle_hyperscanner.so).  Every hyperscan() and check_patterns()
call the reference's Python layer makes is stored with its arguments and what the oracle answered: return code and
every callback batch of (id, line_number, line).  The suite must pass on top of the oracle, so these answers are what
the reference's layer needs from a native library to pass its own tests; tests/test_reference_suite.py replays the
calls against the oracle, the host-logic build and libgpugrep.so and requires identical answers.  Fixture paths are
stored by name: the files themselves are in tests/golden/reference_cases.json (tools/make_golden.py).

Also loaded by that pytest run as the plugin `-p record_reference_abi` (the fixture below).
"""

from __future__ import annotations

import ctypes
import io
import json
import os
import subprocess
import sys
import tempfile
import threading

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle", "_build", "liboracle_hyperscanner.so")
OUT = os.path.join(ROOT, "tests", "golden", "reference_suite_abi.json")


class _Recorder:
    """Stands in for the reference's ctypes handle: forwards to the oracle, appends one JSON line per call to $RECORD_TO
    (a file, because parallel_grep runs some calls in forked worker processes)."""

    def __init__(self, lib: ctypes.CDLL, out_path: str, fixture_root: str, test_id: str) -> None:
        self.lib, self.out_path, self.fixture_root, self.test_id = lib, out_path, fixture_root, test_id
        self.lock = threading.Lock()

    def _write(self, entry: dict) -> None:
        entry["test"] = self.test_id
        # io.open: the suite replaces builtins.open with a mock in most of its tests
        with self.lock, io.open(self.out_path, "a", encoding="utf-8") as handle:
            handle.write(json.dumps(entry) + "\n")

    @staticmethod
    def _set(patterns, flags, ids, count: int) -> dict:
        return {"patterns": [patterns[i].decode("latin-1") for i in range(count)], "flags": [flags[i] for i in range(count)],
                "ids": [ids[i] for i in range(count)]}

    def check_patterns(self, patterns, flags, ids, count):
        rc = self.lib.check_patterns(patterns, flags, ids, count)
        self._write({"fn": "check_patterns", **self._set(patterns, flags, ids, count), "rc": rc})
        return rc

    def hyperscan(self, path, patterns, flags, ids, count, callback, buffer_size, buffer_count, max_match_count):  # pylint: disable=too-many-arguments
        batches = []

        def record(results, n):
            batches.append([[results[i].id, results[i].line_number, results[i].line.decode("latin-1")] for i in range(n)])
            callback(results, n)

        hook = type(callback)(record)
        rc = self.lib.hyperscan(path, patterns, flags, ids, count, hook, buffer_size, buffer_count, max_match_count)
        name = path.decode()
        rel = os.path.relpath(name, self.fixture_root)
        file = {"fixture": rel} if not rel.startswith("..") else {"path": name}
        self._write({"fn": "hyperscan", "file": file, **self._set(patterns, flags, ids, count), "buffer_size": buffer_size,
                     "buffer_count": buffer_count, "max_match_count": max_match_count.value, "rc": rc, "batches": batches})
        return rc


@pytest.fixture(autouse=True)
def _record_native_calls(request: pytest.FixtureRequest, monkeypatch: pytest.MonkeyPatch) -> None:
    from hypergrep import utils  # the reference package, from the checkout on PYTHONPATH

    fixture_root = os.path.dirname(str(request.node.path))
    recorder = _Recorder(ctypes.CDLL(ORACLE), os.environ["RECORD_TO"], fixture_root, request.node.nodeid.split("::", 1)[-1])
    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: recorder)


def main() -> None:
    reference = os.path.abspath(sys.argv[1])
    suite = os.path.join(reference, "hypergrep", "test", "test_hypergrep.py")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    raw = os.path.join(tempfile.mkdtemp(), "calls.jsonl")
    env = dict(os.environ, RECORD_TO=raw, PYTHONPATH=os.pathsep.join([reference, os.path.join(ROOT, "tools")]))
    proc = subprocess.run([sys.executable, "-m", "pytest", suite, "-p", "record_reference_abi", "-p", "no:cacheprovider", "-q"],
                          cwd=reference, env=env, capture_output=True, text=True, check=False)
    summary = proc.stdout.strip().splitlines()[-1].split(" in ")[0]   # "75 passed"
    if proc.returncode != 0:
        sys.exit(proc.stdout[-3000:] + proc.stderr[-2000:])
    # one entry per distinct call, in a stable order; the tests that made it are kept for the reader
    calls: dict = {}
    with open(raw, encoding="utf-8") as handle:
        for line in handle:
            entry = json.loads(line)
            test = entry.pop("test")
            key = json.dumps(entry, sort_keys=True)
            calls.setdefault(key, {**entry, "tests": []})["tests"].append(test)
    os.unlink(raw)
    os.rmdir(os.path.dirname(raw))
    for entry in calls.values():
        entry["tests"] = sorted(set(entry["tests"]))
    doc = {
        "source": "pyranha-labs/hypergrep v3.2.0 hypergrep/test/test_hypergrep.py, run unmodified on the CPU oracle",
        "generator": "tools/record_reference_abi.py",
        "suite_result": summary,
        "calls": [calls[key] for key in sorted(calls)],
    }
    with open(OUT, "w", encoding="utf-8") as handle:
        json.dump(doc, handle, indent=1, sort_keys=True)
    print(OUT, summary, f"{len(calls)} distinct calls")


if __name__ == "__main__":
    main()
