"""Fixed strings with reports: gpugrep_literal_report_scan_file / gpugrep_literal_report_scan_buffer, scan_literals() and the
automaton-free `grep -F -o`.

The expected answer is the one include/gpugrep.h defines: the records of hyperscan() / gpugrep_scan_* for the same set with
every byte written as \\xHH, the same flags and the same ids (`escaped_set`).  CPU tests run the host logic on the report
stand-in (tests/mock_engine_literal_reports), which finds every occurrence of every literal with memmem, against the PCRE2
oracle and against the regex stand-in's multi-id scan of the escaped set; `gpu` tests run the CUDA engine (fast and general
path) against the CUDA engine's own regex scan of the escaped set and against the oracle."""

from __future__ import annotations

import ctypes
import gzip
import os
import random
import re
import subprocess
import time

import numpy as np
import pytest

import byte_cases
import parity
from gpu_api import Stats, marshal
from hypergrep_b200 import synth
from oracle_api import CALLBACK, run_scan
from test_fixed_strings import EDGE_TEXTS, literal_scan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORTS_LIB = os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal_reports.so")
_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
              ctypes.c_ulonglong, ctypes.c_void_p]
_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
# prefixes and suffixes of one another, duplicates with other ids, caseless and exact copies, '\n'-ended and inner-'\n' ones
EDGE_SET = ([b"foo", b"fo", b"f", b"oo", b"foo", b"FOO", b"bar\n", b"ar", b"ab\nc", b"\xff\xfe", b"\xff", b"`", b"@", b"abab", b"ab",
             b"AbAbA", b"0123456", b"obar"],
            [8, 8, 0, 0, 8, 9, 0, 8, 0, 8, 8, 1, 0, 0, 8, 9, 0, 1],
            [1, 2, 3, 4, 5, 1, 6, 2, 7, 8, 9, 10, 11, 4, 12, 13, 14, 15])


class _Collector:
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


def _arrays(literals, flags, ids):
    n = len(literals)
    arr = (ctypes.c_char_p * max(n, 1))(*literals)
    fl = (ctypes.c_uint * max(n, 1))(*flags) if flags is not None else None
    ia = (ctypes.c_uint * max(n, 1))(*ids) if ids is not None else None
    return arr, fl, ia, n


def report_scan(lib, path, literals, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0, collect=True):
    entry = lib.gpugrep_literal_report_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    la, fa, ia, n = _arrays(literals, flags, ids)
    sink, stats = _Collector(collect), Stats()
    rc = entry(str(path).encode(), la, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def report_scan_buffer(lib, ptr, size, location, literals, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0,
                       collect=True):
    entry = lib.gpugrep_literal_report_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    la, fa, ia, n = _arrays(literals, flags, ids)
    sink, stats = _Collector(collect), Stats()
    rc = entry(ptr, size, location, la, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, None, ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def escaped_set(literals):
    return ["".join(f"\\x{b:02x}" for b in lit) for lit in literals]


def regex_scan(lib, path, literals, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0, collect=True):
    """gpugrep_scan_file of the escaped set: the definition's answer, from a regex engine."""
    n = len(literals)
    pa, fa, ia, n = marshal(escaped_set(literals), list(flags) if flags is not None else [0] * n, list(ids) if ids is not None else [0] * n)
    if flags is None or not any(flags):
        fa = (ctypes.c_uint * n)(*([0] * n))   # (marshal turns an all-zero list into its defaults)
    if ids is None:
        ia = (ctypes.c_uint * n)(*([0] * n))
    entry = lib.gpugrep_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(str(path).encode(), pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def oracle_scan(oracle_lib, path, literals, flags, ids, **kw):
    return run_scan(oracle_lib, str(path), escaped_set(literals), flags=[f | 0 for f in flags] if any(flags) else [0] * len(literals),
                    ids=ids, **kw)


def model_reports(data: bytes, literals, flags, ids, buffer_size: int = 262140):
    """(id, line) records by the definition: every (id, end) per scanned block, by end then id, SINGLEMATCH ids once."""
    from test_fixed_strings import _fold, block_of, pseudo_lines  # pylint: disable=import-outside-toplevel
    out = []
    for number, line in enumerate(pseudo_lines(data, buffer_size)):
        block = block_of(line)
        folded = _fold(block)
        reports = set()
        for lit, flag, ident in zip(literals, flags, ids):
            hay, needle = (folded, _fold(lit)) if flag & 1 else (block, lit)
            at = hay.find(needle)
            while at >= 0:
                reports.add((at + len(needle), ident, bool(flag & 8)))
                at = hay.find(needle, at + 1)
        fired = set()
        for end, ident, single in sorted(reports):
            if single:
                if ident in fired:
                    continue
                fired.add(ident)
            out.append((ident, number, end))
    # (a SINGLEMATCH id and a non-SINGLEMATCH one never share an id, so (id, end) is unique here)
    seen, dedup = set(), []
    for rec in out:
        if rec not in seen:
            seen.add(rec)
            dedup.append(rec)
    return [(ident, number) for ident, number, _ in dedup]


@pytest.fixture(scope="session")
def reports_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal_reports")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(REPORTS_LIB)


@pytest.fixture(scope="session")
def literal_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal.so"))


def random_report_set(rng: random.Random, count: int):
    """Prefix chains, duplicates, mixed CASELESS, shared and distinct ids; SINGLEMATCH per id."""
    lits = []
    while len(lits) < count:
        r = rng.random()
        if lits and r < 0.25:
            base = rng.choice(lits)
            lits.append(base[:rng.randint(1, len(base))])              # a prefix
        elif lits and r < 0.35:
            lits.append(rng.choice(lits))                              # a duplicate
        elif lits and r < 0.5:
            lits.append(rng.choice(lits) + bytes(rng.choice(b"abAB@`\n") for _ in range(rng.randint(1, 3))))   # an extension
        else:
            lits.append(bytes(rng.choice(b"abcAB@`[{\x80\xff.") for _ in range(rng.randint(1, 6))))
    ids = [rng.randrange(max(1, count // 3)) for _ in lits]
    single = {ident: rng.random() < 0.5 for ident in set(ids)}
    flags = [(8 if single[ident] else 0) | rng.choice((0, 1, 2, 4, 1 | 6)) for ident in ids]
    return lits, flags, ids


def random_text(rng: random.Random, size: int, lits) -> bytes:
    parts = []
    while sum(map(len, parts)) < size:
        r = rng.random()
        if r < 0.35:
            parts.append(rng.choice(lits))
        elif r < 0.45:
            parts.append(b"\n")
        elif r < 0.47:
            parts.append(b"\0")
        else:
            parts.append(bytes(rng.choice(b"abcABC@`[{\x80\xff. \n") for _ in range(rng.randint(1, 12))))
    return b"".join(parts)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(EDGE_TEXTS))
@pytest.mark.parametrize("buffer_size", [4, 9, 262140])
def test_edge_texts_against_the_oracles(name, buffer_size, reports_lib, hostmock_lib, oracle_lib, tmp_path):
    path = tmp_path / "t.log"
    data = EDGE_TEXTS[name] + b"foobar FOO\n"
    path.write_bytes(data)
    lits, flags, ids = EDGE_SET
    want = regex_scan(hostmock_lib, path, lits, flags, ids, buffer_size=buffer_size)
    got = report_scan(reports_lib, path, lits, flags, ids, buffer_size=buffer_size)
    assert got[0] == want[0] == 0 and got[1:3] == want[1:3]
    assert got[1] == oracle_scan(oracle_lib, path, lits, flags, ids, buffer_size=buffer_size)[1]
    assert [(r[0], r[1]) for r in got[1]] == model_reports(data, lits, flags, ids, buffer_size)


@pytest.mark.parametrize("seed", range(8))
def test_random_sets_limits_and_batches(seed, reports_lib, hostmock_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    rng = random.Random(seed)
    lits, flags, ids = random_report_set(rng, rng.randint(1, 30))
    data = random_text(rng, 20_000, lits)
    path = tmp_path / "r.log"
    path.write_bytes(data)
    for kw in ({}, {"max_match_count": 7, "buffer_count": 3}, {"max_match_count": 1}, {"buffer_count": 1}, {"buffer_size": 17},
               {"buffer_size": 5, "max_match_count": 40, "buffer_count": 6}):
        want = regex_scan(hostmock_lib, path, lits, flags, ids, **kw)
        got = report_scan(reports_lib, path, lits, flags, ids, **kw)
        assert got[0] == want[0] == 0 and got[1:3] == want[1:3], kw
        counted = report_scan(reports_lib, path, lits, flags, ids, collect=False, **kw)
        assert counted[0] == 0 and counted[3].matches == want[3].matches == len(want[1]), kw
    assert [(r[0], r[1]) for r in report_scan(reports_lib, path, lits, flags, ids)[1]] == model_reports(data, lits, flags, ids)


def test_limit_counts_records_after_a_whole_line(reports_lib, hostmock_lib, tmp_path):
    path = tmp_path / "l.log"
    path.write_bytes(b"aaa\nxyz\naaaa\n")
    lits, flags, ids = [b"a", b"aa"], [0, 0], [1, 2]
    got = report_scan(reports_lib, path, lits, flags, ids, max_match_count=2)
    assert got[1] == regex_scan(hostmock_lib, path, lits, flags, ids, max_match_count=2)[1]
    assert len(got[1]) == 5   # the whole first line: a@1, a@2, aa@2, a@3, aa@3


def test_compressed_and_sharded(reports_lib, hostmock_lib, tmp_path, monkeypatch):
    text = synth.syslog_bytes(1 << 20, seed=3, lib=hostmock_lib)
    lits = [b"Failed password", b"Failed", b"port 22", b"SESSION", b"error:", b"\xff\xfe", b"sshd"]
    flags, ids = [8, 8, 0, 9, 0, 0, 8], [1, 2, 3, 4, 3, 5, 6]
    plain = tmp_path / "p.log"
    plain.write_bytes(text)
    want = regex_scan(hostmock_lib, plain, lits, flags, ids)
    assert len(want[1]) > 100
    gz = tmp_path / "p.log.gz"
    gz.write_bytes(gzip.compress(text))
    assert report_scan(reports_lib, gz, lits, flags, ids)[:3] == want[:3]
    for name, blob in parity.zstd_cases(text).items():
        path = tmp_path / f"{name}.log.zst"
        path.write_bytes(blob)
        assert report_scan(reports_lib, path, lits, flags, ids)[:3] == regex_scan(hostmock_lib, path, lits, flags, ids)[:3], name
    host = ctypes.create_string_buffer(text, len(text))
    assert report_scan_buffer(reports_lib, ctypes.addressof(host), len(text), 0, lits, flags, ids)[:3] == want[:3]
    monkeypatch.setenv("GPUGREP_MOCK_DEVICES", "3")
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
    assert report_scan(reports_lib, plain, lits, flags, ids)[:3] == want[:3]
    assert report_scan_buffer(reports_lib, ctypes.addressof(host), len(text), 0, lits, flags, ids)[:3] == want[:3]
    limited = regex_scan(hostmock_lib, plain, lits, flags, ids, max_match_count=50, buffer_count=7)
    assert report_scan(reports_lib, plain, lits, flags, ids, max_match_count=50, buffer_count=7)[:3] == limited[:3]
    counted = report_scan(reports_lib, plain, lits, flags, ids, collect=False)
    assert counted[3].matches == len(want[1])


def test_return_codes(reports_lib, literal_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(b"foo\nbar\n")
    assert report_scan(reports_lib, path, [b"foo", b""], [0, 0], [1, 2])[0] == 4
    assert report_scan(reports_lib, path, [], [], [])[0] == 4
    for bit in (16, 32, 1 << 31):
        assert report_scan(reports_lib, path, [b"foo"], [bit | 8], [1])[0] == 4
    assert report_scan(reports_lib, path, [b"foo", b"bar"], [8, 0], [1, 1])[0] == 4   # shared id, SINGLEMATCH disagrees
    assert report_scan(reports_lib, path, [b"foo", b"bar"], [8, 0], [1, 2])[0] == 0
    assert report_scan(reports_lib, path, [b"foo", b"bar"], None, None)[:2] == (0, [(0, 0, b"foo\n"), (0, 1, b"bar\n")])
    # an engine without the report stage
    assert report_scan(literal_lib, path, [b"foo"], [8], [1])[0] == 7
    assert report_scan(literal_lib, path, [b""], [8], [1])[0] == 4


def test_report_and_selection_sets_are_cached_apart(reports_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(b"aa\nb\n")
    lits = [b"a", b"aa"]
    line = (0, 0, b"aa\n")
    assert literal_scan(reports_lib, str(path), lits, [8, 8])[1] == [line]
    assert report_scan(reports_lib, path, lits, [0, 0], [0, 0])[1] == [line] * 2   # (0, 1) and (0, 2)
    assert literal_scan(reports_lib, str(path), lits, [0, 0])[1] == [line]
    assert report_scan(reports_lib, path, lits, [8, 8], [0, 1])[1] == [line, (1, 0, b"aa\n")]


@pytest.fixture()
def py_on_mock(reports_lib, monkeypatch):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    monkeypatch.setenv("GPUGREP_LIBRARY", REPORTS_LIB)
    monkeypatch.setitem(utils._state, "lib", None)  # pylint: disable=protected-access
    return utils


def _records(function, *args, **kw):
    out = []

    def cb(matches, count):
        out.extend((matches[k].id, matches[k].line_number, matches[k].line) for k in range(count))

    rc = function(*args, cb, **kw)
    return rc, out


def _escaped_str(literals):
    return ["".join(f"\\x{b:02x}" for b in lit.encode()) for lit in literals]


def test_python_scan_literals(py_on_mock, tmp_path):
    import hypergrep_b200  # pylint: disable=import-outside-toplevel
    utils = py_on_mock
    assert hypergrep_b200.scan_literals is utils.scan_literals
    path = tmp_path / "k.log"
    path.write_bytes("a.b x a.b\nAXB\n(x+ é a.b\nnone\n".encode())
    lits = ["a.b", "a", "(x+", "é", "A.B", "b"]
    flags, ids = [8, 0, 8, 2, 9, 8], [7, 3, 2, 5, 7, 9]
    assert _records(utils.scan_literals, str(path), lits, flags=flags, ids=ids) == \
        _records(utils.scan, str(path), _escaped_str(lits), flags=flags, ids=ids)
    assert _records(utils.scan_literals, str(path), lits, flags=flags, ids=ids, max_match_count=3, buffer_count=2) == \
        _records(utils.scan, str(path), _escaped_str(lits), flags=flags, ids=ids, max_match_count=3, buffer_count=2)
    default = _records(utils.scan_literals, str(path), lits)
    assert default == _records(utils.scan, str(path), lits, fixed_strings=True)
    assert default[1] and all(r[0] == 0 for r in default[1])
    with pytest.raises(ValueError):
        utils.scan(str(path), ["a"], lambda *_: None, ids=[1], fixed_strings=True)
    with pytest.raises(ValueError):
        utils.scan_literals(str(path), ["a", ""], lambda *_: None)


def _regex_route_only_matching(utils, path, literals, **kw):
    """grep -F -o as it was answered before: the re.escape-d list as regular expressions."""
    return utils.grep(str(path), [re.escape(lit) for lit in literals], only_matching=True, **kw)


@pytest.mark.parametrize("seed", range(4))
def test_grep_fixed_only_matching_equals_the_regex_route(seed, py_on_mock, tmp_path):
    utils = py_on_mock
    rng = random.Random(seed)
    words = ["ab", "abab", "a.b", "AB", "x(y", "é", "ü.", "zz", "b"]
    lines = [" ".join(rng.choice(words + ["filler", "x y"]) for _ in range(rng.randint(0, 6))) for _ in range(200)]
    path = tmp_path / "o.log"
    path.write_bytes(("\n".join(lines) + "\n").encode() + b"ab \xff\xfe abab\nlast ab")
    for name, text in EDGE_TEXTS.items():
        edge = tmp_path / f"{name}.log"
        edge.write_bytes(text)
        for lits in (["foo"], ["oo", "bar"], ["ÿ"]):
            assert utils.grep(str(edge), lits, fixed_strings=True, only_matching=True) == _regex_route_only_matching(utils, edge, lits), name
    for _ in range(6):
        lits = rng.sample(words, rng.randint(1, 4))
        for kw in ({}, {"ignore_case": True}, {"errors": "replace"}, {"errors": "backslashreplace"}, {"max_match_count": 5},
                   {"count_only": True}, {"invert_match": True}):
            assert utils.grep(str(path), lits, fixed_strings=True, only_matching=True, **kw) == \
                _regex_route_only_matching(utils, path, lits, **kw), (lits, kw)
    missing = tmp_path / "missing.log"
    assert utils.grep(str(missing), ["a"], fixed_strings=True, only_matching=True, no_messages=True) == \
        _regex_route_only_matching(utils, missing, ["a"], no_messages=True)


def test_grep_fixed_only_matching_builds_no_automata(py_on_mock, tmp_path, monkeypatch):
    """A 100k-literal `grep -F -o` compiles no escaped list, in `re` or in the engine, and finishes quickly."""
    utils = py_on_mock
    rng = np.random.default_rng(7)
    alnum = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    lits = sorted({rng.choice(alnum, size=12).tobytes().decode() for _ in range(100_000)})
    lines = [f"line {k} " + (f"hit={lits[0]} and {lits[0]}" if k % 50 == 0 else f"ioc={lits[k % len(lits)]}") for k in range(5000)]
    path = tmp_path / "ioc.log"
    path.write_text("\n".join(lines) + "\n")
    compiled = []
    real_compile = re.compile

    def counting_compile(pattern, *args, **kw):
        compiled.append(pattern)
        return real_compile(pattern, *args, **kw)

    monkeypatch.setattr(utils.re, "compile", counting_compile)
    monkeypatch.setattr(utils, "_span_widths", lambda *_: pytest.fail("the escaped list reached the span route"))
    t0 = time.perf_counter()
    got, code = utils.grep(str(path), lits, fixed_strings=True, only_matching=True)
    elapsed = time.perf_counter() - t0
    print(f"grep -F -o with 100k literals: {elapsed:.2f} s")
    assert code == 0 and len(compiled) <= 1
    assert got == [(k + 1, lits[0] + "\n") for k in range(0, 5000, 50) for _ in range(2)]
    assert elapsed < 30


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _device(data: bytes):
    import torch  # pylint: disable=import-outside-toplevel
    dev = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return dev


def _gpu_compare(gpu_lib, data: bytes, lits, flags, ids, tmp_path, kinds=("file", "host", "pinned", "device"), **kw):
    """Report scan == regex scan of the escaped set on every input kind; returns the records and the last stats."""
    path = tmp_path / "g.log"
    path.write_bytes(data)
    want = regex_scan(gpu_lib, path, lits, flags, ids, **kw)
    assert want[0] == 0
    got = report_scan(gpu_lib, path, lits, flags, ids, **kw)
    assert got[:3] == want[:3]
    if "host" in kinds:
        host = ctypes.create_string_buffer(data, len(data) + 1)
        assert report_scan_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, lits, flags, ids, **kw)[:3] == want[:3]
    if "pinned" in kinds:
        import torch  # pylint: disable=import-outside-toplevel
        pinned = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).pin_memory()
        assert report_scan_buffer(gpu_lib, pinned.data_ptr(), len(data), 0, lits, flags, ids, **kw)[:3] == want[:3]
    if "device" in kinds:
        dev = _device(data)
        got = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, ids, **kw)
        assert got[:3] == want[:3]
        counted = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, ids, collect=False)
        assert counted[0] == 0 and counted[3].matches == len(regex_scan(gpu_lib, path, lits, flags, ids)[1])
    return want[1], got[3]


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_edges_alphabet_and_oracle(force_general, gpu_lib, oracle_lib, tmp_path, monkeypatch):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    lits, flags, ids = EDGE_SET
    for name, text in EDGE_TEXTS.items():
        for buffer_size in (9, 262140):
            recs, _ = _gpu_compare(gpu_lib, text + b"foobar FOO\n", lits, flags, ids, tmp_path, buffer_size=buffer_size)
            assert recs == oracle_scan(oracle_lib, tmp_path / "g.log", lits, flags, ids, buffer_size=buffer_size)[1], name
    alphabet = byte_cases.alphabet_text() if hasattr(byte_cases, "alphabet_text") else bytes(range(1, 256)) * 4 + b"\n"
    blits = [bytes([b]) for b in range(1, 256) if b != 10] + [bytes([b, b + 1]) for b in range(1, 255) if 10 not in (b, b + 1)]
    bflags = [(1 if k % 3 == 0 else 0) | 8 for k in range(len(blits))]
    bids = [k % 97 for k in range(len(blits))]
    single = {}
    for k, ident in enumerate(bids):   # one SINGLEMATCH value per id
        bflags[k] = (bflags[k] & ~8) | single.setdefault(ident, bflags[k] & 8)
    _gpu_compare(gpu_lib, alphabet, blits, bflags, bids, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_gpu_random_sets_on_syslog(seed, gpu_lib, tmp_path, monkeypatch):
    rng = random.Random(seed)
    base = synth.syslog_bytes(4 << 20, seed=seed)
    lines = base.split(b"\n")
    lits = [bytes(rng.choice(b"abcdefghXYZ0123456789@`[{\x80\xfe ") for _ in range(rng.randint(4 if seed != 1 else 1, 16)))
            for _ in range(rng.choice((50, 1000)))]
    lits += [lit[:rng.randint(min(4, len(lit)), len(lit))] for lit in rng.sample(lits, 20)]   # prefix chains
    lits += [b"Failed password for", b"Failed password", b"sshd[", b"\xff\xfe\xfd\xfc", b"port 22\n", b"@`[{"]
    ids = [rng.randrange(len(lits) // 2) for _ in lits]
    single = {ident: rng.random() < 0.6 for ident in set(ids)}
    flags = [(8 if single[ident] else 0) | rng.choice((0, 1)) for ident in ids]
    for k in range(0, len(lines), 89):
        lines[k] = lines[k] + rng.choice(lits).replace(b"\n", b"") + (b"\0tail" if k % 5 == 0 else b"")
    data = b"\n".join(lines)
    recs, stats = _gpu_compare(gpu_lib, data, lits, flags, ids, tmp_path, buffer_count=4096)
    assert len(recs) > 1000
    if seed != 1:
        assert stats.path & 1
    monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    _gpu_compare(gpu_lib, data, lits, flags, ids, tmp_path, kinds=("device",), buffer_count=4096, max_match_count=3000)


@pytest.mark.gpu
def test_gpu_sharded(gpu_lib, tmp_path, monkeypatch):
    import torch  # pylint: disable=import-outside-toplevel
    data = synth.syslog_bytes(16 << 20, seed=5)
    lits = [b"Failed password", b"Failed", b"port 22", b"SESSION", b"error:", b"sshd"]
    flags, ids = [8, 8, 0, 9, 0, 8], [1, 2, 3, 4, 3, 6]
    path = tmp_path / "s.log"
    path.write_bytes(data)
    want = regex_scan(gpu_lib, path, lits, flags, ids)
    monkeypatch.setenv("GPUGREP_DEVICES", ",".join(["0"] * 3) if torch.cuda.device_count() == 1 else "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", str(1 << 20))
    assert report_scan(gpu_lib, path, lits, flags, ids)[:3] == want[:3]
    host = ctypes.create_string_buffer(data, len(data))
    assert report_scan_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, lits, flags, ids)[:3] == want[:3]
    gz = tmp_path / "s.log.gz"
    gz.write_bytes(gzip.compress(data, compresslevel=1))
    assert report_scan(gpu_lib, gz, lits, flags, ids)[:3] == want[:3]
    for name, blob in list(parity.zstd_cases(data).items())[:1]:
        zst = tmp_path / f"{name}.log.zst"
        zst.write_bytes(blob)
        assert report_scan(gpu_lib, zst, lits, flags, ids)[:3] == want[:3]


def _ioc_set(count: int, seed: int):
    rng = np.random.default_rng(seed)
    iocs = [f"{a}.{b}.{c}.{d}".encode() for a, b, c, d in rng.integers(1, 255, size=(count // 2, 4))]
    hexd = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)
    iocs += [rng.choice(hexd, size=32).tobytes() for _ in range(count - len(iocs))]
    return iocs, rng


def _model_first_ends(data: bytes, lits: list[bytes]) -> list[tuple[int, int]]:
    """(index, line) records of exact SINGLEMATCH literals with ids = index: per line, every literal once at its first end,
    by end then index.  Occurrences come from a rolling hash per distinct length, checked against a dict of literals by
    length; the NUL cut is applied by joining the scanned blocks with a byte that no literal holds."""
    from test_fixed_strings import block_of, pseudo_lines  # pylint: disable=import-outside-toplevel
    blocks = [block_of(line) for line in pseudo_lines(data)]
    text = b"\x01".join(blocks)
    starts = np.cumsum([0] + [len(b) + 1 for b in blocks])
    arr = np.frombuffer(text, dtype=np.uint8).astype(np.uint64)
    by_len: dict[int, dict[bytes, list[int]]] = {}
    for index, lit in enumerate(lits):
        by_len.setdefault(len(lit), {}).setdefault(lit, []).append(index)
    mul = np.uint64(1099511628211)
    first: dict[int, dict[int, int]] = {}
    for length, table in by_len.items():
        if len(arr) < length:
            continue
        h = np.zeros(len(arr) - length + 1, dtype=np.uint64)
        for k in range(length):
            h = h * mul + arr[k:len(arr) - length + 1 + k]
        targets = set()
        for lit in table:
            v = 0
            for b in lit:
                v = (v * 1099511628211 + b) & 0xFFFFFFFFFFFFFFFF
            targets.add(v)
        for pos in np.flatnonzero(np.isin(h, np.array(sorted(targets), dtype=np.uint64))):
            for index in table.get(text[pos:pos + length], ()):
                line = int(np.searchsorted(starts, pos, side="right") - 1)
                end = int(pos - starts[line]) + length
                ends = first.setdefault(line, {})
                ends[index] = min(ends.get(index, end), end)
    return [(index, line) for line in sorted(first) for index, _ in sorted(first[line].items(), key=lambda item: (item[1], item[0]))]


@pytest.mark.gpu
@pytest.mark.parametrize("count", [100_000, 1_000_000])
def test_gpu_large_ioc_sets_against_a_python_model(count, gpu_lib):
    """ids = index, every literal SINGLEMATCH, planted hits: every (id, line) record, by a dict of literals by length."""
    iocs, rng = _ioc_set(count, count)
    lines = synth.syslog_bytes(64 << 20, seed=11).split(b"\n")
    planted = rng.choice(len(iocs), size=4000)
    step = len(lines) // 2001
    for k in range(0, len(planted), 2):
        at = (k // 2 + 1) * step
        lines[at] += b" ioc=" + iocs[planted[k]] + b" also " + iocs[planted[k + 1]] + (b"\0" + iocs[planted[k]] if k % 14 == 0 else b"")
    data = b"\n".join(lines)
    want = _model_first_ends(data, iocs)
    flags = [8] * len(iocs)
    dev = _device(data)
    rc, recs, _, stats = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, flags, list(range(len(iocs))), buffer_count=1 << 16)
    assert rc == 0 and [(r[0], r[1]) for r in recs] == want
    assert len(want) >= 3000 and stats.path & 1


@pytest.mark.gpu
def test_gpu_prefix_chain_over_a_long_pseudo_line(gpu_lib):
    """a, aa, ... a*200 plus near misses, over one 256 KiB pseudo-line of 'a': bounded work, exact records."""
    lits = [b"a" * k for k in range(1, 201)] + [b"a" * k + b"b" for k in range(1, 200, 7)] + [b"A" * 50]
    ids = list(range(len(lits)))
    flags = [8] * (len(lits) - 1) + [9]
    data = b"a" * (256 << 10) + b"\n" + b"aab\n"
    dev = _device(data)
    t0 = time.perf_counter()
    rc, recs, _, _ = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, ids, buffer_size=(256 << 10) + 4, buffer_count=1 << 16)
    print(f"prefix chain over 256 KiB of 'a': {time.perf_counter() - t0:.2f} s")
    # line 0: every chain literal once (SINGLEMATCH), at its first end; the caseless 'A'*50 at 50; line 1: a, aa, ab
    ends = {k: k + 1 for k in range(200)}
    ends[len(lits) - 1] = 50
    want = [(ident, 0) for ident in sorted(ends, key=lambda ident: (ends[ident], ident))] + [(0, 1), (1, 1), (200, 1)]
    assert rc == 0 and [(r[0], r[1]) for r in recs] == want


@pytest.mark.gpu
def test_gpu_plain_scans_keep_their_launches(gpu_lib):
    """The C2 pins of regex scans, and plain fixed-string scans keep their kernels and paths."""
    from test_fixed_strings import C2_REGEX_PIN, literal_scan_buffer  # pylint: disable=import-outside-toplevel
    from gpu_api import scan_buffer  # pylint: disable=import-outside-toplevel
    data = synth.syslog_bytes(8 << 20, seed=42)
    dev = _device(data)
    got = {}
    rc, _, stats = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, synth.C2_PATTERNS)
    got["plain"] = (rc, stats.launches, stats.path)
    rc, _, stats = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, synth.C2_PATTERNS, collect=False)
    got["count"] = (rc, stats.launches, stats.path)
    entry = gpu_lib.gpugrep_invert_scan_buffer
    entry.restype = ctypes.c_int
    pa, fa, ia, n = marshal(synth.C2_PATTERNS)
    stats = Stats()
    rc = entry(ctypes.c_void_p(dev.data_ptr()), ctypes.c_size_t(len(data)), 1, pa, fa, ia, n, None, 262140, 16, ctypes.c_ulonglong(1 << 40),
               None, ctypes.byref(stats))
    got["invert"] = (rc, stats.launches, stats.path)
    assert got == C2_REGEX_PIN
    lits = [b"Failed password for", b"session opened", b"Connection closed"]
    plain = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits)
    reports = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, [14] * 3, [0] * 3)
    assert plain[0] == reports[0] == 0 and plain[1] == reports[1]
    assert plain[3].path == reports[3].path == 1
    assert reports[3].launches == plain[3].launches + 5   # count pass, scan of the counts (3), write pass
    counted = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, collect=False)
    assert counted[3].matches == len(plain[1])


@pytest.mark.gpu
def test_gpu_grep_fixed_only_matching_on_the_cuda_library(tmp_path):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    iocs, _ = _ioc_set(100_000, 3)
    lits = [lit.decode() for lit in iocs]
    lines = synth.syslog_bytes(8 << 20, seed=4).decode(errors="replace").split("\n")
    for k in range(0, len(lines), 97):
        lines[k] += f" ioc={lits[k % 1000]} first={lits[0]}{lits[0]}"
    path = tmp_path / "f.log"
    path.write_text("\n".join(lines))
    t0 = time.perf_counter()
    got, code = utils.grep(str(path), lits, fixed_strings=True, only_matching=True)
    print(f"grep -F -o, 100k literals, 8 MiB: {time.perf_counter() - t0:.2f} s")
    # every line that holds the first literal is selected, and its parts are that literal's non-overlapping occurrences
    want = [(number, lits[0] + "\n") for number, line in enumerate(lines, 1) for _ in range(line.count(lits[0]))]
    assert code == 0 and got == want and len(want) > 100
