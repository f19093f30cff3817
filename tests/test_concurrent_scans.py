"""Concurrent scans in one process: what two scans running at the same time do to each other.

The product runs scans concurrently (multiscanner.parallel_grep: one hyperscan() per file on a thread pool; utils.scan/grep
on worker threads), and the engine shares state between them: per-device slot pools with grow-only scratch, compiled-database,
device-table and tuned-prefilter caches, decode and read helpers, device load accounting, and kernel attributes that belong to
the process (a kernel's dynamic shared-memory limit).  Each concurrent answer here is compared with the same call made
serially earlier in the same process - return code, every record, batch sizes, stats.matches and stats.lines - and each
serial answer once with the oracle, so that a test cannot pass by agreeing with a wrong serial answer.

  a. mixed stress on one device: every entry point, input kind and scan mode, pattern sets that take every fast-path kernel
     (including 64 and 128 KiB tables of one k_stream instantiation, and k_verify_smem with two table sizes over 48 KiB);
  b. pooled scratch is not read stale: small scans in a fresh process, then scans that grow every buffer, then the small
     scans again;
  c. the caller's stream: device text written on a torch stream and scanned on it without a host synchronisation;
  d. the Python layer: parallel_grep over many files and utils.grep from several threads;
  e. several GPUs: (a) spread by the least-loaded choice, with a sharded scan at the same time;
  f. the host pipeline under ThreadSanitizer, over the CPU engine stand-in (tests/tsan_driver).
"""

from __future__ import annotations

import ctypes
import gzip
import os
import random
import re
import subprocess
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

# pylint: disable=wrong-import-position
import fast_path_cases as fpc
from dfa_sim import CompiledDb
from event_cases import match_ends, oracle_ends
from gpu_api import Stats, marshal
from k1_model import K1Tables
from oracle_api import CALLBACK, load_oracle, run_scan
from parity import gz_members, zstd_frame
from test_context_lines import CONTEXT_ID, oracle_context
from test_invert_match import _short_lines, oracle_invert

HOST, DEVICE = 0, 1
SMALL_BYTES = 3000          # under the 4 KiB below which scans keep the database's untuned prefilter table
CHUNK_BYTES = 256 << 10     # GPUGREP_CHUNK_BYTES of the stress: many segments per call
SAMPLE_BYTES = 512 << 10    # head of an input that the prefilter is tuned on (capi.cpp kSampleBytes)
MAX_SHARED_TABLE = 112 << 10   # engine.cu kMaxSharedTableBytes


def _words(seed: int, count: int, length: int) -> list[str]:
    rng = random.Random(seed)
    return ["".join(rng.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(length)) for _ in range(count)]


# ---- pattern sets -------------------------------------------------------------------------------------------------------------
# GRAM: 129-256 prefilter grams, so the untuned table (inputs under 4 KiB) is a 64 KiB bloom table and the tuned one 128 KiB,
# of the same k_stream instantiation.  VERIFY_A / VERIFY_B: one DFA group each whose class-compressed tables for
# k_verify_smem are over 48 KiB and differ in size.  The preconditions are asserted (test_stress_sets_reach_their_kernels).
GRAM = _words(11, 45, 24)
VERIFY_A = _words(12, 60, 24)
VERIFY_B = _words(13, 80, 24)
NFA_PATTERNS = ["alpha.*x.{14}omega", "kilo.*q.{16}gram"]
GAP_INSTANCES = [b"alpha " + b"x" * 30 + b"omega", b"kilo" + b"q" * 20 + b"gram"]


def _c3():
    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    return synth.c3_patterns()


def pattern_sets() -> dict:
    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    multi = ["ERROR", "port [0-9]+", "sshd", "fail(ed|ure)", "timeout"]
    return {
        "c1": (synth.C1_PATTERNS, [14], [0]),
        "c2": (synth.C2_PATTERNS, [14] * len(synth.C2_PATTERNS), [0] * len(synth.C2_PATTERNS)),
        # several ids, every other pattern without SINGLEMATCH: the general path and match events
        "multi": (multi, [6, 14, 6, 14, 6], [1, 2, 3, 4, 5]),
        # patterns whose DFA would need 2^15 and 2^17 states: NFA fallbacks, which ride the fast path through k_confirm
        "nfa": (NFA_PATTERNS + GRAM[:8], [14] * 10, [0] * 10),
        "c3": (_c3()[0], [14] * 1000, [0] * 1000),
        "gram": (GRAM, [14] * len(GRAM), [0] * len(GRAM)),
        "verify_a": (VERIFY_A, [14] * len(VERIFY_A), [0] * len(VERIFY_A)),
        "verify_b": (VERIFY_B, [14] * len(VERIFY_B), [0] * len(VERIFY_B)),
    }


# ---- texts ----------------------------------------------------------------------------------------------------------------------

def _planted(size: int, seed: int, plants: list[str]) -> bytes:
    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    data = synth.syslog_bytes(size, seed=seed, plants=plants, plant_ppm=30000)
    return data[:data.rfind(b"\n") + 1]


def _small(big: bytes, seed: int, words: list[str]) -> bytes:
    """Under SMALL_BYTES: lines of `big`, every third one carrying a word of the set."""
    rng = random.Random(seed)
    lines = big.splitlines(keepends=True)[:400]
    out = b""
    for k, line in enumerate(lines):
        if k % 3 == 0:
            w = rng.choice(words).encode()
            at = rng.randrange(len(line))
            line = line[:at] + w + line[at:]
        if len(out) + len(line) > SMALL_BYTES:
            break
        out += line
    return out


def texts() -> dict:
    plants = GRAM + VERIFY_A[::2] + VERIFY_B[::3] + [g.decode() for g in GAP_INSTANCES] + _c3()[1][:40]
    big = _planted(4 << 20, 21, plants)
    return {
        "big": big,
        "mid": big[:big.rfind(b"\n", 0, 1 << 20) + 1],
        "small": _small(big, 5, GRAM),
        "small_a": _small(big, 6, VERIFY_A),
        "small_b": _small(big, 7, VERIFY_B),
    }


# ---- calls ----------------------------------------------------------------------------------------------------------------------
# A call: (set, text, entry, input).  entry: scan | count | invert | invert_count | context | ends.  input: file | gzip |
# gzip_members | zstd_frames | host | pinned | device.

_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
_CONTEXT_BUFFER_ARGS = _BUFFER_ARGS[:11] + [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
              ctypes.c_ulonglong, ctypes.c_void_p]
_CONTEXT_FILE_ARGS = _FILE_ARGS[:9] + [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
CONTEXT = (2, 1)   # -B2 -A1
BUFFER_COUNT = 7


def bind(lib) -> None:
    for name, args in (("gpugrep_scan_buffer", _BUFFER_ARGS), ("gpugrep_invert_scan_buffer", _BUFFER_ARGS),
                       ("gpugrep_context_scan_buffer", _CONTEXT_BUFFER_ARGS), ("gpugrep_scan_file", _FILE_ARGS),
                       ("gpugrep_invert_scan_file", _FILE_ARGS), ("gpugrep_context_scan_file", _CONTEXT_FILE_ARGS)):
        entry = getattr(lib, name)
        entry.restype, entry.argtypes = ctypes.c_int, args


class Inputs:
    """Every text in every input form: files (plain, gzip, gzip members, zstd frames), pageable, pinned and device memory."""

    def __init__(self, data: dict, directory: str, torch=None):
        self.data = data
        self.paths, self.host, self.pinned, self.device = {}, {}, {}, {}
        for name, blob in data.items():
            lines = blob.splitlines(keepends=True)
            pieces = [b"".join(lines[k:k + 500]) for k in range(0, len(lines), 500)]
            forms = {"file": blob, "gzip": gzip.compress(blob, 1), "gzip_members": gz_members(pieces),
                     "zstd_frames": b"".join(zstd_frame(p) for p in pieces)}
            for form, payload in forms.items():
                path = os.path.join(directory, f"{name}.{form}")
                with open(path, "wb") as handle:
                    handle.write(payload)
                self.paths[(name, form)] = path
            self.host[name] = np.frombuffer(blob + bytes(64), dtype=np.uint8).copy()
            if torch is not None:
                pinned = torch.empty(len(blob) + 64, dtype=torch.uint8, pin_memory=True)
                pinned.numpy()[:] = self.host[name]
                self.pinned[name] = pinned
                self.device[name] = torch.from_numpy(self.host[name]).cuda()
        if torch is not None:
            torch.cuda.synchronize()

    def buffer(self, text: str, form: str) -> tuple[int, int]:
        if form == "host":
            return self.host[text].ctypes.data, HOST
        if form == "pinned":
            return self.pinned[text].data_ptr(), HOST
        return self.device[text].data_ptr(), DEVICE


class _Sink:
    def __init__(self, collect: bool):
        self.records, self.batches = [], []

        def cb(results, count):
            self.batches.append(count)
            for i in range(count):
                r = results[i]
                self.records.append((r.id, r.line_number, r.line))

        self.c_callback = CALLBACK(cb) if collect else None

    def pointer(self):
        return ctypes.cast(self.c_callback, ctypes.c_void_p) if self.c_callback else None


def run_call(lib, call: tuple, sets: dict, inputs: Inputs, stream: int = 0, text_override: tuple | None = None) -> tuple:
    """One call -> (rc, records, batches, stats.matches, stats.lines, stats.path).  `text_override`: (pointer, size) of a device
    buffer holding the call's text (the stream tests)."""
    set_name, text, entry, form = call
    patterns, flags, ids = sets[set_name]
    pa, fa, ia, n = marshal(patterns, flags, ids)
    size = len(inputs.data[text])
    stats = Stats()
    if entry == "ends":
        ptr, loc = (text_override[0], DEVICE) if text_override else inputs.buffer(text, form)
        rc, ends, found = match_ends(lib, ptr, size, loc, patterns, flags, ids, 262140, stats=stats)
        return rc, tuple(ends), (found,), stats.matches, stats.lines, stats.path
    sink = _Sink(entry in ("scan", "invert", "context"))
    cb = sink.pointer()
    if form in ("file", "gzip", "gzip_members", "zstd_frames"):
        path = inputs.paths[(text, form)].encode()
        if entry in ("scan", "count"):
            rc = lib.gpugrep_scan_file(path, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, ctypes.byref(stats))
        elif entry in ("invert", "invert_count"):
            rc = lib.gpugrep_invert_scan_file(path, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, ctypes.byref(stats))
        else:
            rc = lib.gpugrep_context_scan_file(path, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, CONTEXT[0], CONTEXT[1], 0, ctypes.byref(stats))
    else:
        ptr, loc = (text_override[0], DEVICE) if text_override else inputs.buffer(text, form)
        st = stream or None
        if entry in ("scan", "count"):
            rc = lib.gpugrep_scan_buffer(ptr, size, loc, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, st, ctypes.byref(stats))
        elif entry in ("invert", "invert_count"):
            rc = lib.gpugrep_invert_scan_buffer(ptr, size, loc, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, st, ctypes.byref(stats))
        else:
            rc = lib.gpugrep_context_scan_buffer(ptr, size, loc, pa, fa, ia, n, cb, 262140, BUFFER_COUNT, 0, CONTEXT[0], CONTEXT[1], 0, st,
                                                 ctypes.byref(stats))
    return rc, tuple(sink.records), tuple(sink.batches), stats.matches, stats.lines, stats.path


def same_answer(got: tuple, want: tuple) -> str | None:
    """None if the answers agree (the path may differ: a drifted table may send a segment the other way), else what differs."""
    names = ("return code", "records", "batches", "stats.matches", "stats.lines")
    for name, a, b in zip(names, got[:5], want[:5]):
        if a != b:
            if name == "records":
                k = next((k for k, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
                return f"records: {len(a)} vs {len(b)}, first difference at {k}: {a[k] if k < len(a) else None} vs {b[k] if k < len(b) else None}"
            return f"{name}: {a if not isinstance(a, tuple) else a[:8]} vs {b if not isinstance(b, tuple) else b[:8]}"
    return None


def check_with_oracle(oracle, call: tuple, answer: tuple, sets: dict, inputs: Inputs, cache: dict) -> None:
    """A serial answer against the oracle.  Compressed inputs hold the text of the plain file: their answers must equal the
    plain file's, which `cache` holds once it has been checked."""
    set_name, text, entry, form = call
    patterns, flags, ids = sets[set_name]
    path = inputs.paths[(text, "file")]
    rc, records, batches, matches, lines, _ = answer
    label = str(call)
    assert rc == 0, f"{label}: return code {rc}"
    key = (set_name, text, entry)
    if key in cache:
        assert same_answer(answer, cache[key]) is None, f"{label}: {same_answer(answer, cache[key])}"
        return
    if entry == "ends":
        exp_rc, exp, found = oracle_ends(oracle, inputs.data[text], patterns, flags, ids, 262140)
        assert (rc, list(records), batches[0]) == (exp_rc, exp, found), label
    elif entry in ("scan", "count"):
        exp_rc, exp, exp_batches = run_scan(oracle, path, patterns, flags=flags, ids=ids, buffer_count=BUFFER_COUNT)
        if entry == "scan":
            assert (rc, list(records), list(batches)) == (exp_rc, exp, exp_batches), label
        else:
            assert records == () and rc == exp_rc, label
        assert matches == len(exp), f"{label}: stats.matches {matches} != {len(exp)}"
    elif entry in ("invert", "invert_count"):
        exp_rc, exp, exp_batches = oracle_invert(oracle, path, patterns, flags=flags, ids=ids, buffer_count=BUFFER_COUNT)
        if entry == "invert":
            assert (rc, list(records), list(batches)) == (exp_rc, exp, exp_batches), label
        assert matches == len(exp), f"{label}: stats.matches {matches} != {len(exp)}"
    else:
        exp_rc, exp, exp_batches = oracle_context(oracle, path, patterns, flags=flags, ids=ids, buffer_count=BUFFER_COUNT,
                                                  before=CONTEXT[0], after=CONTEXT[1])
        assert (rc, list(records), list(batches)) == (exp_rc, exp, exp_batches), label
        assert matches == sum(1 for r in exp if r[0] != CONTEXT_ID), label
    assert lines == inputs.data[text].count(b"\n"), f"{label}: stats.lines {lines}"
    cache[key] = answer


def stress_calls(with_device: bool = True) -> list[tuple]:
    calls = [
        ("c1", "big", "scan", "file"), ("c1", "big", "scan", "host"), ("c1", "big", "count", "device"), ("c1", "big", "invert", "device"),
        ("c1", "big", "context", "pinned"),
        ("c2", "big", "scan", "gzip_members"), ("c2", "big", "scan", "pinned"), ("c2", "big", "invert", "file"),
        ("c2", "big", "context", "device"), ("c2", "big", "count", "host"), ("c2", "big", "invert_count", "device"),
        ("multi", "big", "scan", "zstd_frames"), ("multi", "big", "scan", "device"), ("multi", "mid", "ends", "host"),
        ("multi", "big", "count", "device"),
        ("nfa", "big", "scan", "device"), ("nfa", "big", "scan", "gzip"), ("nfa", "mid", "ends", "device"), ("nfa", "big", "invert", "host"),
        ("c3", "mid", "scan", "device"), ("c3", "mid", "scan", "gzip"), ("c3", "mid", "count", "host"),
        ("gram", "small", "scan", "host"), ("gram", "small", "scan", "device"), ("gram", "small", "count", "device"),
        ("gram", "small", "invert", "device"), ("gram", "small", "context", "host"), ("gram", "small", "scan", "pinned"),
        ("gram", "big", "scan", "device"), ("gram", "big", "scan", "host"), ("gram", "big", "scan", "file"),
        ("gram", "big", "scan", "zstd_frames"), ("gram", "big", "count", "device"), ("gram", "big", "invert", "pinned"),
        ("gram", "big", "context", "device"),
        ("verify_a", "big", "scan", "device"), ("verify_a", "big", "scan", "host"), ("verify_a", "big", "count", "device"),
        ("verify_a", "small_a", "scan", "device"),
        ("verify_b", "big", "scan", "device"), ("verify_b", "big", "scan", "file"), ("verify_b", "big", "context", "device"),
        ("verify_b", "small_b", "scan", "host"),
    ]
    if not with_device:
        calls = [c for c in calls if c[3] not in ("device", "pinned")]
    return calls


def run_concurrently(worker, count: int) -> list:
    """Runs worker(k) on `count` threads, joins them all, returns what each raised (None for none)."""
    errors = [None] * count

    def body(k):
        try:
            worker(k)
        except BaseException as exc:  # pylint: disable=broad-except
            errors[k] = exc

    threads = [threading.Thread(target=body, args=(k,)) for k in range(count)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    return errors


def stress(lib, calls: list, serial: dict, sets: dict, inputs: Inputs, threads: int = 12, per_thread: int = 40, seed: int = 1) -> None:
    """`threads` threads, each working through a shuffled list of `per_thread` calls; every answer must equal the serial one."""
    rng = random.Random(seed)
    lists = [[calls[rng.randrange(len(calls))] for _ in range(per_thread)] for _ in range(threads)]
    failures = []

    def worker(k):
        for call in lists[k]:
            diff = same_answer(run_call(lib, call, sets, inputs), serial[call])
            if diff:
                failures.append(f"{call}: {diff}")

    errors = run_concurrently(worker, threads)
    assert not [e for e in errors if e], [repr(e) for e in errors if e]
    assert not failures, failures[:10]


# ---- preconditions ---------------------------------------------------------------------------------------------------------------

def verify_smem_bytes(db: CompiledDb) -> int:
    """The shared memory k_verify_smem takes for a database (engine_upload: class-compressed table and depths, each rounded up
    to 16 bytes, plus 256), or 0 when the database does not take that kernel."""
    if db.info.groups != 1 or not db.info.simple:
        return 0
    gi = db.groups[0][0]
    ncls = gi.classes + 2
    ctab = gi.states * ncls * 2
    if ncls > 255 or ctab + gi.states + 32 > MAX_SHARED_TABLE:
        return 0
    return 256 + (ctab + 15) // 16 * 16 + (gi.states + 15) // 16 * 16


def bloom_false_rate(db: CompiledDb, tables: K1Tables) -> float:
    """engine_upload_prefilter's bloom_false_rate: above 0.005 the fast path confirms candidates (k_confirm) first."""
    return db.info.prefilter_grams * (16.0 / tables.stride) / (1 << tables.log2_bits)


def stress_preconditions(lib, sets: dict, data: dict) -> dict:
    """The sets reach the kernels the stress is about; returns what was found (for the messages)."""
    found = {}
    gram = CompiledDb(lib, *sets["gram"])
    assert 129 <= gram.info.prefilter_grams <= 256, gram.info.prefilter_grams
    untuned = K1Tables(gram)
    gram.retune(data["big"][:SAMPLE_BYTES])
    tuned = K1Tables(gram)
    assert untuned.bitmap.size == 64 << 10 and tuned.bitmap.size == 128 << 10, (untuned.bitmap.size, tuned.bitmap.size)
    assert fpc.instantiation(untuned, {}) == fpc.instantiation(tuned, {}), "tuned and untuned inputs take different k_stream instantiations"
    found["gram"] = (gram.info.prefilter_grams, fpc.instantiation(tuned, {}))
    sizes = []
    for name in ("verify_a", "verify_b"):
        db = CompiledDb(lib, *sets[name])
        assert db.info.prefilter and db.info.prefilter_lookback <= 64, name
        for sample in (None, data["big"][:SAMPLE_BYTES]):
            if sample is not None:
                db.retune(sample)
            # k_verify_smem is taken only without candidate confirmation: one group, no NFA, few bloom collisions
            assert bloom_false_rate(db, K1Tables(db)) <= 0.005, name
        size = verify_smem_bytes(db)
        assert size > 48 << 10, (name, size)
        sizes.append(size)
    assert sizes[0] != sizes[1], sizes
    found["verify"] = sizes
    c3 = CompiledDb(lib, *sets["c3"])
    assert c3.info.groups >= 2 and c3.info.simple, "the 1,000-pattern set must compile to several DFA groups (k_confirm)"
    nfa = CompiledDb(lib, *sets["nfa"])
    assert sum(g[0].members for g in nfa.groups) == len(GRAM[:8]) and nfa.info.simple, "the gap patterns must be NFA fallbacks"
    multi = CompiledDb(lib, *sets["multi"])
    assert not multi.info.simple
    return found


# ---- a. mixed stress on one device ----------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    assert module.cuda.is_available()
    return module


@pytest.fixture(scope="module")
def stress_state(gpu_lib, oracle_lib, torch, tmp_path_factory):
    """Inputs, the serial answer of every stress call (checked with the oracle) - made with small segments."""
    bind(gpu_lib)
    sets, data = pattern_sets(), texts()
    found = stress_preconditions(gpu_lib, sets, data)
    inputs = Inputs(data, str(tmp_path_factory.mktemp("concurrent")), torch)
    old = os.environ.get("GPUGREP_CHUNK_BYTES")
    os.environ["GPUGREP_CHUNK_BYTES"] = str(CHUNK_BYTES)
    try:
        serial, cache = {}, {}
        calls = stress_calls()
        for call in calls:
            serial[call] = run_call(gpu_lib, call, sets, inputs)
        for call in sorted(calls, key=lambda c: c[3] != "file"):   # plain files first: compressed forms compare with them
            check_with_oracle(oracle_lib, call, serial[call], sets, inputs, cache)
    finally:
        if old is None:
            del os.environ["GPUGREP_CHUNK_BYTES"]
        else:
            os.environ["GPUGREP_CHUNK_BYTES"] = old
    return {"sets": sets, "data": data, "inputs": inputs, "serial": serial, "calls": calls, "found": found}


@pytest.mark.gpu
def test_stress_sets_reach_their_kernels(stress_state):
    """Both paths ran; the small gram-set inputs took the fast path (untuned 64 KiB table) as the large ones did (128 KiB)."""
    serial = stress_state["serial"]
    paths = 0
    for call, answer in serial.items():
        paths |= answer[5]
        if call[0] in ("gram", "verify_a", "verify_b", "c1", "c2") and call[2] in ("scan", "count"):
            assert answer[5] & 1, f"{call} did not take the fast path: path={answer[5]}"
        if call[0] == "multi":
            assert answer[5] == 2, f"{call}: path={answer[5]}"
    assert paths == 3
    assert stress_state["found"]["verify"][0] != stress_state["found"]["verify"][1]


@pytest.mark.gpu
def test_mixed_stress_on_one_device(stress_state, gpu_lib, monkeypatch):
    """12 threads x 40 calls of every entry point, input and set on device 0: every answer equals the serial one."""
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", str(CHUNK_BYTES))
    monkeypatch.setenv("GPUGREP_DEVICE", "0")
    stress(gpu_lib, stress_state["calls"], stress_state["serial"], stress_state["sets"], stress_state["inputs"])


# ---- b. pooled scratch is not read stale --------------------------------------------------------------------------------------

def _fresh_pool_main(directory: str) -> None:
    """Run in a fresh process: small scans, scans that grow every scratch buffer, the small scans again."""
    import torch as tmod  # pylint: disable=import-outside-toplevel

    lib = ctypes.CDLL(os.path.join(ROOT, "hypergrep_b200", "lib", "libgpugrep.so"))
    bind(lib)
    lib.gpugrep_set_device(0)
    oracle = load_oracle()
    sets = pattern_sets()
    del sets["c3"]
    big = texts()["big"]
    data = {"s_big": big[:big.rfind(b"\n", 0, 600 << 10) + 1], "small": _small(big, 5, GRAM), "short": _short_lines(1 << 20, 9)}
    inputs = Inputs(data, directory, tmod)
    small_calls = [(s, t, e, f) for s, t in (("gram", "small"), ("gram", "s_big"), ("c1", "short"), ("multi", "s_big"), ("c2", "s_big"))
                   for e in ("scan", "count", "invert", "context") for f in ("host", "device")]
    small_calls += [("multi", "s_big", "ends", "device"), ("nfa", "s_big", "scan", "device")]
    first, cache = {}, {}
    for call in small_calls:
        first[call] = run_call(lib, call, sets, inputs)
    for call in small_calls:
        check_with_oracle(oracle, call, first[call], sets, inputs, cache)
    assert {a[5] for a in first.values()} >= {1, 2}
    # grow every scratch buffer: 1 GiB of device-resident text with many records (normal, inverted, context), the
    # short-line text (a record per line), and a general-path piece
    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    grow = tmod.empty(1 << 30, dtype=tmod.uint8, device="cuda")
    host = np.empty(1 << 30, dtype=np.uint8)
    synth.fill_syslog(host, seed=8, plants=GRAM, plant_ppm=30000)
    grow.copy_(tmod.from_numpy(host))
    del host
    short = tmod.from_numpy(np.frombuffer(_short_lines(64 << 20, 10), dtype=np.uint8).copy()).cuda()
    tmod.cuda.synchronize()
    discard = ctypes.cast(lib.gpugrep_discard_results, ctypes.c_void_p)
    for name, (ptr, size) in (("big", (grow.data_ptr(), grow.numel())), ("short", (short.data_ptr(), short.numel()))):
        for set_name in ("c1", "gram", "multi"):
            pa, fa, ia, n = marshal(*sets[set_name])
            st = Stats()
            assert lib.gpugrep_scan_buffer(ptr, size, DEVICE, pa, fa, ia, n, discard, 262140, 4096, 0, None, ctypes.byref(st)) == 0, (name, set_name)
            assert lib.gpugrep_invert_scan_buffer(ptr, size, DEVICE, pa, fa, ia, n, discard, 262140, 4096, 0, None, ctypes.byref(st)) == 0
            assert lib.gpugrep_context_scan_buffer(ptr, size, DEVICE, pa, fa, ia, n, discard, 262140, 4096, 0, 3, 3, 0, None,
                                                   ctypes.byref(st)) == 0
    del grow, short
    for call in reversed(small_calls):
        diff = same_answer(run_call(lib, call, sets, inputs), first[call])
        assert diff is None, f"{call} after the pool grew: {diff}"
    print("fresh pool ok", len(small_calls))


@pytest.mark.gpu
def test_pooled_scratch_is_not_read_stale(tmp_path):
    """Small scans of every kind, then scans that grow every pooled buffer, then the small scans again: identical answers.
    A kernel that reads past what its own scan wrote would read the larger scan's bytes."""
    proc = subprocess.run([sys.executable, os.path.abspath(__file__), "fresh_pool", str(tmp_path)], capture_output=True, text=True,
                          timeout=900, check=False)
    assert proc.returncode == 0, proc.stdout[-4000:] + proc.stderr[-8000:]
    assert "fresh pool ok" in proc.stdout


# ---- c. the caller's stream ---------------------------------------------------------------------------------------------------

STREAM_CALLS = [("gram", "big", "scan", "device"), ("c1", "big", "invert", "device"), ("c2", "big", "context", "device"),
                ("gram", "big", "count", "device"), ("c1", "big", "count", "device"), ("c2", "big", "invert_count", "device"),
                ("multi", "big", "scan", "device")]


def _written_on(torch, stream, encoded):
    """A device text written by kernels on `stream`, behind a delay, so that a scan not ordered after them reads garbage."""
    with torch.cuda.stream(stream):
        out = torch.empty_like(encoded)
        out.fill_(0x41)
        torch.cuda._sleep(20_000_000)   # pylint: disable=protected-access
        torch.bitwise_xor(encoded, 0x5A, out=out)
    return out


@pytest.mark.gpu
def test_scans_on_the_callers_stream(stress_state, gpu_lib, torch, monkeypatch):
    """Text produced on a torch stream and scanned with stream= that stream, without a host synchronisation: normal,
    inverted, context and count-only answers equal the serial ones; also from two threads, each on its own stream."""
    monkeypatch.setenv("GPUGREP_DEVICE", "0")
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", str(CHUNK_BYTES))
    sets, inputs, serial = stress_state["sets"], stress_state["inputs"], stress_state["serial"]
    encoded = torch.bitwise_xor(inputs.device["big"], 0x5A)
    torch.cuda.synchronize()

    def run(stream, calls):
        for call in calls:
            text = _written_on(torch, stream, encoded)
            got = run_call(gpu_lib, call, sets, inputs, stream=stream.cuda_stream, text_override=(text.data_ptr(), text.numel()))
            diff = same_answer(got, serial[call])
            assert diff is None, f"{call} on the caller's stream: {diff}"

    run(torch.cuda.Stream(), STREAM_CALLS)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    errors = run_concurrently(lambda k: run(streams[k], STREAM_CALLS[k::2] + STREAM_CALLS), 2)
    torch.cuda.synchronize()
    assert errors == [None, None], errors


# ---- d. the Python layer ------------------------------------------------------------------------------------------------------

def _grep_files(directory: str, data: dict) -> tuple[list[str], dict]:
    """About 24 files: a few bytes, under 4 KiB, several MiB, gzip and zstd; returns the names and the text of each."""
    big = data["big"]
    rng = random.Random(4)
    files, text_of = [], {}
    for k in range(24):
        kind = k % 6
        if kind == 0:
            text = GRAM[k % len(GRAM)].encode() + b"\n" if k % 12 else b"x\n"
        elif kind in (1, 2):
            text = _small(big, 100 + k, GRAM)
        elif kind == 3:
            start = big.find(b"\n", rng.randrange(len(big) // 2)) + 1
            text = big[start:start + (2 << 20)]
            text = text[:text.rfind(b"\n") + 1]
        else:
            text = big[:big.rfind(b"\n", 0, (1 + k % 3) << 20) + 1]
        name = os.path.join(directory, f"f{k:02d}.log")
        payload = text
        if kind == 4:
            name += ".gz"
            payload = gzip.compress(text, 1)
        elif kind == 5:
            name += ".zst"
            payload = zstd_frame(text)
        with open(name, "wb") as handle:
            handle.write(payload)
        files.append(name)
        text_of[name] = text
    return files, text_of


@pytest.mark.gpu
def test_parallel_grep_and_threaded_grep(stress_state, oracle_lib, capsys, tmp_path):
    """multiscanner.parallel_grep on its default thread pool over 24 files prints every file's records as the oracle finds them;
    utils.grep from 8 threads at once (-v, -B/-A, -o) returns what it returns serially, and that matches the oracle."""
    from hypergrep_b200 import multiscanner, utils  # pylint: disable=import-outside-toplevel

    files, text_of = _grep_files(str(tmp_path), stress_state["data"])
    expected = []
    for name in files:
        plain = str(tmp_path / "plain.txt")
        with open(plain, "wb") as handle:
            handle.write(text_of[name])
        rc, records, _ = run_scan(oracle_lib, plain, GRAM, flags=[utils._DEFAULT_FLAGS] * len(GRAM))   # pylint: disable=protected-access
        assert rc == 0
        expected.append("".join(f"{name}:{line.decode(errors='ignore')}" for _, _, line in records))
    capsys.readouterr()
    code = multiscanner.parallel_grep(files, GRAM, with_file_name=True)
    printed = capsys.readouterr().out
    assert code == 0
    assert printed == "".join(expected)

    # utils.grep: serial answers against the oracle, then 8 threads
    path = str(tmp_path / "grep.log")
    with open(path, "wb") as handle:
        handle.write(stress_state["data"]["mid"])
    patterns = GRAM[:20] + ["sshd"]
    flags = [utils._DEFAULT_FLAGS] * len(patterns)   # pylint: disable=protected-access
    variants = [{}, {"invert_match": True}, {"before_context": 2, "after_context": 1}, {"only_matching": True},
                {"invert_match": True, "after_context": 2}, {"count_only": True}]
    serial = [utils.grep(path, patterns, **kw) for kw in variants]
    rc, records, _ = run_scan(oracle_lib, path, patterns, flags=flags)
    assert serial[0] == ([(ln + 1, line.decode(errors="ignore")) for _, ln, line in records], 0)
    _, inv, _ = oracle_invert(oracle_lib, path, patterns, flags=flags)
    assert serial[1] == ([(ln + 1, line.decode(errors="ignore")) for _, ln, line in inv], 0)
    _, ctx, _ = oracle_context(oracle_lib, path, patterns, flags=flags, before=2, after=1)
    assert serial[2] == ([(ln + 1, line.decode(errors="ignore"), i == CONTEXT_ID) for i, ln, line in ctx], 0)
    first = re.compile(patterns[0])
    assert serial[3] == ([(ln + 1, m.group() + "\n") for _, ln, line in records for m in first.finditer(line.decode(errors="ignore"))], 0)
    _, ctx, _ = oracle_context(oracle_lib, path, patterns, flags=flags, before=0, after=2, invert=True)
    assert serial[4] == ([(ln + 1, line.decode(errors="ignore"), i == CONTEXT_ID) for i, ln, line in ctx], 0)
    assert serial[5] == (len(records), 0)
    failures = []

    def worker(k):
        for j in range(len(variants) * 2):
            v = (k + j) % len(variants)
            if utils.grep(path, patterns, **variants[v]) != serial[v]:
                failures.append((k, variants[v]))

    errors = run_concurrently(worker, 8)
    assert errors == [None] * 8, errors
    assert not failures, failures[:5]


# ---- e. several GPUs ------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_stress_over_several_gpus(stress_state, gpu_lib, torch, monkeypatch):
    """(a) without a device override: the least-loaded choice spreads the file and host calls over the devices, with a sharded
    scan of a 72 MiB host buffer ($GPUGREP_DEVICES=all; the other inputs are under the shard size) running at the same time."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.delenv("GPUGREP_DEVICE", raising=False)
    monkeypatch.delenv("LOCAL_RANK", raising=False)
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", str(CHUNK_BYTES))
    sets, inputs, serial = stress_state["sets"], stress_state["inputs"], dict(stress_state["serial"])
    gpu_lib.gpugrep_set_device(-1)
    calls = stress_calls(with_device=False)
    big = stress_state["data"]["big"]
    sharded = big * 18
    inputs.data["sharded"] = sharded
    inputs.host["sharded"] = np.frombuffer(sharded + bytes(64), dtype=np.uint8).copy()
    call = ("c2", "sharded", "scan", "host")
    serial[call] = run_call(gpu_lib, call, sets, inputs)   # one device: no $GPUGREP_DEVICES yet
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    stress(gpu_lib, calls + [call] * 4, serial, sets, inputs, seed=2)


# ---- f. the host pipeline under ThreadSanitizer ---------------------------------------------------------------------------------

def test_host_pipeline_under_thread_sanitizer(tmp_path):
    """The host logic and the CPU engine stand-in built with -fsanitize=thread: 8 threads in rounds over plain files (one read
    split over helper threads), files of many gzip members and zstd frames (decode helpers), host buffers, inverted, context
    and count-only scans, on one device and sharded over three mock devices, give the serial answers without a report."""
    directory = os.path.join(ROOT, "tests", "tsan_driver")
    subprocess.check_call(["make", "-C", directory], stdout=subprocess.DEVNULL)
    rng = random.Random(17)
    words = ["ERROR", "error", "port 8080", "port 443", "sshd", "timeout", "alpha", "kilo", "xx", "GET /index", "user=bob", "failed", "done"]
    lines = [" ".join(rng.choice(words) for _ in range(rng.randint(1, 8))).encode() + b"\n" for _ in range(40000)]
    text = b"".join(lines)
    pieces = [b"".join(lines[k:k + 200]) for k in range(0, len(lines), 200)]
    plain = (text * (1 + (9 << 20) // len(text)))[:9 << 20]
    (tmp_path / "plain.log").write_bytes(plain[:plain.rfind(b"\n") + 1])
    (tmp_path / "big.log").write_bytes(text[:text.rfind(b"\n", 0, 3 << 20) + 1])
    (tmp_path / "small.log").write_bytes(text[:text.rfind(b"\n", 0, 3000) + 1])
    (tmp_path / "members.gz").write_bytes(gz_members(pieces))
    (tmp_path / "frames.zst").write_bytes(b"".join(zstd_frame(p) for p in pieces))
    env = {k: v for k, v in os.environ.items() if not k.startswith("GPUGREP_")}
    env.update(GPUGREP_MOCK_DEVICES="3", TSAN_OPTIONS=f"exitcode=66 halt_on_error=0 suppressions={directory}/tsan.supp")
    proc = subprocess.run([os.path.join(ROOT, "tests", "_build", "concurrent_driver"), str(tmp_path)], capture_output=True, text=True,
                          env=env, timeout=1200, check=False)
    assert proc.returncode != 66, "ThreadSanitizer report:\n" + proc.stderr[-30000:]
    assert proc.returncode == 0, proc.stdout[-4000:] + proc.stderr[-8000:]
    assert "WARNING: ThreadSanitizer" not in proc.stderr, proc.stderr[-30000:]
    assert "concurrent driver ok" in proc.stdout, proc.stdout


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "fresh_pool":
    _fresh_pool_main(sys.argv[2])
