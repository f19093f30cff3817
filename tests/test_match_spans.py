"""Leftmost-first match spans (`grep -o` of variable-width patterns): gpugrep_span_exact, gpugrep_match_spans and the span
route of utils.grep(only_matching=True), against Python's re as the oracle.

CPU tests run on the host logic linked against the CPU stand-in of the engine with the span stage
(tests/mock_engine_spans: the same pike_vm.hpp the kernel runs).  `-m gpu` tests run the CUDA library.
"""

from __future__ import annotations

import ctypes
import os
import random
import re
import subprocess

import numpy as np
import pytest

import parity
from dfa_sim import CompiledDb
from gpu_api import Stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OVER = 0xFFFFFFFF
HOST, DEVICE = 0, 1
PROBE_PATTERNS = [r"port [0-9]+", r"user=\w+", r"rhost=10\.[0-9]+\.[0-9]+\.[0-9]+", r"ERROR.*", r"score [0-9]{1,4}",
                  r"sector [0-9]{6,}", r"user=(root|admin)", r"\d+\.\d+\.\d+\.\d+"]


class Span(ctypes.Structure):
    """gpugrep_match_span (include/gpugrep.h)."""

    _fields_ = [("line_number", ctypes.c_ulonglong), ("start", ctypes.c_uint), ("end", ctypes.c_uint)]


@pytest.fixture(scope="session")
def spans_mock_lib() -> ctypes.CDLL:
    """Host logic of the boundary linked against the CPU engine stand-in with the span stage (tests/mock_engine_spans)."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_spans")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_spans.so"))


def span_exact(lib, pattern: bytes) -> int:
    lib.gpugrep_span_exact.restype = ctypes.c_int
    lib.gpugrep_span_exact.argtypes = [ctypes.c_char_p]
    return lib.gpugrep_span_exact(pattern)


def match_spans(lib, ptr, size: int, location: int, pattern: bytes, buffer_size: int = 262140, capacity: int | None = None):
    """gpugrep_match_spans -> (rc, [(line, start, end)] of the stored records, count found, stats).  capacity None: room for
    all (one retry)."""
    entry = lib.gpugrep_match_spans
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                      ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    cap = 1024 if capacity is None else capacity
    while True:
        out = (Span * max(cap, 1))()
        found = ctypes.c_size_t(0)
        stats = Stats()
        rc = entry(ptr, size, location, pattern, buffer_size, out, cap, ctypes.byref(found), ctypes.byref(stats))
        if rc != 0 or capacity is not None or found.value <= cap:
            break
        cap = found.value
    stored = min(found.value, cap)
    return rc, [(out[k].line_number, out[k].start, out[k].end) for k in range(stored)], found.value, stats


def host_spans(lib, data: bytes, pattern: bytes, buffer_size: int = 262140, capacity: int | None = None):
    buf = ctypes.create_string_buffer(data, len(data) + 1)
    return match_spans(lib, ctypes.addressof(buf), len(data), HOST, pattern, buffer_size, capacity)


def pseudo_lines(data: bytes, buffer_size: int):
    """The pseudo-lines of `data` as the engine splits them (at most buffer_size - 1 bytes, ending at '\\n')."""
    limit = max(1, buffer_size - 1)
    pos = 0
    while pos < len(data):
        nl = data.find(b"\n", pos, pos + limit)
        end = nl + 1 if nl >= 0 else min(len(data), pos + limit)
        yield data[pos:end]
        pos = end


def oracle_spans(data: bytes, pattern: bytes, buffer_size: int = 262140):
    """[(line, start, end)] of re.finditer over every stripped block (leading NULs skipped, cut at the next NUL)."""
    compiled = re.compile(pattern)
    out = []
    for line, raw in enumerate(pseudo_lines(data, buffer_size)):
        block = raw.lstrip(b"\0").split(b"\0", 1)[0]
        out += [(line, m.start(), m.end()) for m in compiled.finditer(block)]
    return out


# ---- the exactness screen ---------------------------------------------------------------------------------------------------

ACCEPTED = [r"port [0-9]+", r"user=\w+", r"\d+\.\d+\.\d+\.\d+", "ERROR.*", r'"id":".*?"', "a|ab", "(a+)(ab)?", "(a|ab)(c|bcd)",
            "a*?b", "a+?", "ab??", "a{2,5}?", "a{3,}?", "x{2}", "x{2,}", "x{2,3}", r"\bfoo\B", "^abc", r"\Aab+", "[^a]+", r"\x41+",
            "(?:ab)+", "colou?r", r"sector [0-9]{6,}", "[]a]+", r"a\.b*"]
REJECTED = ["a{,3}", "ab{,3}", r"\s+", r"a\s", "end$", "a$", "(?i)error", "(?i:a)b", "[[:alpha:]]+", "(a*)*b", "(a?)+b", "(|a)+b",
            "(?:a*|b)+", "a*", "x?", "(ab)*", r"\b", "^", "a{0}", "a**", "a*+", "a++", "a{2}{3}", "a{2}+", "a{2}*", "*a", "(*a)",
            r"\bx*?", "é+", r"\Z", r"a\z", r"(?=a)b", r"(?P<n>a)b", "\\", "a{1,2", "a}", "[ab",
            "(?:" + "a|" * 70 + "b)c", "x{200}", "a{1,200}"]


def test_screen_accepts_and_rejects(spans_mock_lib):
    for pattern in ACCEPTED:
        assert span_exact(spans_mock_lib, pattern.encode()) == 1, pattern
        re.compile(pattern)
    for pattern in REJECTED:
        assert span_exact(spans_mock_lib, pattern.encode("utf-8")) == 0, pattern
    # the fixed-width screen keeps its answers
    spans_mock_lib.gpugrep_span_width.argtypes = [ctypes.c_char_p]
    for pattern, width in [("x{2}", 2), ("a|ab", -1), ("port [0-9]+", -1), ("ab*?", -1), ("ERROR", 5)]:
        assert spans_mock_lib.gpugrep_span_width(pattern.encode()) == width, pattern
    # a pattern that fails the screen is refused with 4
    rc, _, found, _ = host_spans(spans_mock_lib, b"aaa\n", b"a*")
    assert rc == 4 and found == 0


def test_instruction_cap_is_the_boundary(spans_mock_lib):
    # a{n}: n Byte instructions + Match; the cap is 128 instructions
    assert span_exact(spans_mock_lib, b"a{127}") == 1
    assert span_exact(spans_mock_lib, b"a{128}") == 0


LAZY_SETS = [["a+?b", "c*?d"], ["x{2,5}?y", "(ab)+?c"], ['"id":".*?"', "port [0-9]+?"], ["a??b", "(a|b)*?c"], ["fo{1,}?o", "[0-9]{3,}?x"]]


@pytest.mark.parametrize("flags", [0, 14, 6])
def test_lazy_quantifiers_leave_the_automata_unchanged(spans_mock_lib, flags):
    """The DFA and NFA builds do not see laziness: the tables of lazy patterns equal those of the same patterns without `?`."""
    for patterns in LAZY_SETS:
        greedy = [re.sub(r"([*+?}])\?", r"\1", p) for p in patterns]
        assert greedy != patterns
        lazy_db = CompiledDb(spans_mock_lib, patterns, flags=[flags] * len(patterns))
        greedy_db = CompiledDb(spans_mock_lib, greedy, flags=[flags] * len(patterns))
        assert lazy_db.handle and greedy_db.handle, patterns
        assert len(lazy_db.groups) == len(greedy_db.groups) > 0
        for (gi_a, cls_a, trans_a, acc_a, rep_a), (gi_b, cls_b, trans_b, acc_b, rep_b) in zip(lazy_db.groups, greedy_db.groups):
            assert bytes(gi_a) == bytes(gi_b)
            assert np.array_equal(cls_a, cls_b) and np.array_equal(trans_a, trans_b) and np.array_equal(acc_a, acc_b)
            assert rep_a == rep_b
        assert all(np.array_equal(a, b) for a, b in zip(lazy_db.depths, greedy_db.depths))


# ---- random differential against re -----------------------------------------------------------------------------------------

_ATOMS = ["a", "b", "c", "ab", ".", "[ab]", "[^a]", "[^\\n]", r"\w", r"\W", r"\d", "(a|ab)", "(?:a|ab)(c|bcd)", "(ab|a)", "(b|ba|bab)",
          "(?:a|b)", "(a+b|a)"]
_ANCHORS = [r"\b", r"\B", "^", r"\A"]


def _quantifier(rng: random.Random) -> str:
    q = rng.choice(["", "", "*", "+", "?", "{m,n}", "{m}", "{m,}"])
    if q == "{m,n}":
        m = rng.randint(0, 2)
        q = "{%d,%d}" % (m, m + rng.randint(0, 3))
    elif q == "{m}":
        q = "{%d}" % rng.randint(1, 3)
    elif q == "{m,}":
        q = "{%d,}" % rng.randint(0, 2)
    if q and rng.random() < 0.4:
        q += "?"
    return q


def random_pattern(rng: random.Random) -> str:
    parts = []
    for _ in range(rng.randint(1, 4)):
        if rng.random() < 0.15:
            parts.append(rng.choice(_ANCHORS))
        else:
            parts.append(rng.choice(_ATOMS) + _quantifier(rng))
    pattern = "".join(parts)
    if rng.random() < 0.25:
        pattern = pattern + "|" + random_pattern(rng)
    return pattern


def random_text(rng: random.Random, size: int) -> bytes:
    kind = rng.random()
    if kind < 0.6:
        alphabet = rng.choice([b"ab\n", b"abc \n", b"aab_c1 .\n", b"ab\r\n\0"])
        data = bytes(rng.choice(alphabet) for _ in range(size))
    else:
        raw = bytearray(rng.randrange(1, 256) for _ in range(size))
        for _ in range(rng.randint(0, 8)):
            raw[rng.randrange(size)] = rng.choice([0, 10, 13, ord("a"), ord("b")])
        data = bytes(raw)
    if rng.random() < 0.5:
        data += b"\n"
    return data


def random_cases(seed: int, count: int, size: int = 300):
    """(pattern, data, buffer_size) cases whose pattern passes the screen (decided by `screen`)."""
    rng = random.Random(seed)
    for _ in range(count):
        yield random_pattern(rng).encode(), random_text(rng, rng.randint(0, size)), rng.choice([262140, 262140, 2, 3, 7, 16, 40])


def test_random_spans_match_re(spans_mock_lib):
    checked = 0
    for pattern, data, buffer_size in random_cases(1, 900):
        if not span_exact(spans_mock_lib, pattern):
            continue
        rc, got, found, _ = host_spans(spans_mock_lib, data, pattern, buffer_size)
        assert rc == 0, pattern
        expected = oracle_spans(data, pattern, buffer_size)
        assert got == expected and found == len(expected), (pattern, data, buffer_size)
        checked += 1
    assert checked >= 300, checked


def test_capacity_retry_and_budget_sentinel(spans_mock_lib):
    data = b"port 1 port 22 port 333\n" * 50 + b"no\n" + b"port 4444"
    expected = oracle_spans(data, b"port [0-9]+")
    rc, got, found, stats = host_spans(spans_mock_lib, data, b"port [0-9]+", capacity=10)
    assert rc == 0 and found == len(expected) == 151 and got == expected[:10]
    assert stats.matches == found and stats.lines == 52
    rc, got, found, _ = host_spans(spans_mock_lib, data, b"port [0-9]+", capacity=0)
    assert rc == 0 and found == 151 and got == []
    # a quadratic search on a long line: one sentinel for that line, the other lines as usual
    data = b"ab a\n" + b"a" * 5000 + b"\n" + b"xa ab\n"
    rc, got, found, _ = host_spans(spans_mock_lib, data, b"a.*b|a")
    expected = [s for s in oracle_spans(data, b"a.*b|a") if s[0] != 1]
    assert rc == 0 and got == expected[:2] + [(1, OVER, OVER)] + expected[2:], got[:6]


def test_absolute_step_cap_bounds_long_blocks(spans_mock_lib):
    """One linear pass over a 7 MB block stays under 128 steps per byte but over the 2^25 steps any block may take: the
    sentinel, whatever buffer_size allows; a shorter block gets its spans."""
    big = 8 << 20
    rc, got, _, _ = host_spans(spans_mock_lib, b"a" * 7_000_000 + b"\n" + b"aac\n", b"[ab]+c", buffer_size=big)
    assert rc == 0 and got == [(0, OVER, OVER), (1, 0, 3)]
    data = b"a" * 200_000 + b"c\n"
    rc, got, _, _ = host_spans(spans_mock_lib, data, b"[ab]+c", buffer_size=big)
    assert rc == 0 and got == oracle_spans(data, b"[ab]+c", big) == [(0, 0, 200_001)]


# ---- grep(only_matching=True) -------------------------------------------------------------------------------------------------

def check_grep_spans(lib, tmp_path, monkeypatch, expect_route: bool):
    """grep(only_matching=True) == the reference route (_span_widths None: re.finditer for every record).  Returns how many
    variable-width records took the span route."""
    from hypergrep_b200 import utils

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: lib)
    routed = []
    original = utils._fill_spans

    def counting(groups, deferred, patterns, widths, python_patterns, errors, span_lines):
        routed.append(len(span_lines) if span_lines is not None else 0)
        return original(groups, deferred, patterns, widths, python_patterns, errors, span_lines)

    monkeypatch.setattr(utils, "_fill_spans", counting)

    def both(path, patterns, **kw):
        got = utils.grep(str(path), patterns, only_matching=True, **kw)
        with monkeypatch.context() as plain:
            plain.setattr(utils, "_span_widths", lambda _patterns: None)
            expected = utils.grep(str(path), patterns, only_matching=True, **kw)
        assert got == expected, (patterns, kw)

    path = tmp_path / "only.log"
    path.write_bytes(parity.only_matching_text())
    for pattern in parity.ONLY_MATCHING_OTHER + ["user=\\w+", "a+?", "(foo|foob)(ar|bar)"]:
        for ignore_case in (False, True):
            both(path, [pattern], ignore_case=ignore_case)
    both(path, parity.ONLY_MATCHING_OTHER[:3])
    both(path, parity.ONLY_MATCHING_FIXED[:3] + parity.ONLY_MATCHING_OTHER[:3])
    rng = random.Random(17)
    for _ in range(25):
        pattern = random_pattern(rng)
        text = b"".join(bytes(rng.choice(b"abc1 _") for _ in range(rng.randint(0, 30))) + b"\n" for _ in range(150))
        text += b"ab\xe9ab\n" + b"a" * 3000 + b"\n"   # a non-ASCII line and a long one (quadratic patterns hit the budget)
        path.write_bytes(text)
        both(path, [pattern])
    if expect_route:
        assert sum(routed) > 1000, routed
    return sum(routed)


def test_grep_only_matching_takes_the_span_route(spans_mock_lib, tmp_path, monkeypatch):
    check_grep_spans(spans_mock_lib, tmp_path, monkeypatch, expect_route=True)


def test_engine_without_span_stage_refuses_and_grep_falls_back(hostmock_lib, tmp_path, monkeypatch):
    rc, _, found, _ = host_spans(hostmock_lib, b"port 1\n", b"port [0-9]+")
    assert rc == 7 and found == 0
    check_grep_spans(hostmock_lib, tmp_path, monkeypatch, expect_route=False)


# ---- GPU --------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    if not module.cuda.is_available():
        pytest.skip("no CUDA device")
    return module


def device_spans(lib, torch, data: bytes, pattern: bytes, buffer_size: int = 262140, capacity: int | None = None):
    dev = torch.frombuffer(bytearray(data) + bytearray(16), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return match_spans(lib, dev.data_ptr(), len(data), DEVICE, pattern, buffer_size, capacity)


@pytest.mark.gpu
def test_gpu_random_spans_match_re(gpu_lib, torch, monkeypatch):
    checked = 0
    for k, (pattern, data, buffer_size) in enumerate(random_cases(2, 700, size=600)):
        if not span_exact(gpu_lib, pattern):
            continue
        expected = oracle_spans(data, pattern, buffer_size)
        rc, got, found, _ = host_spans(gpu_lib, data, pattern, buffer_size)
        assert rc == 0 and got == expected and found == len(expected), ("host", pattern, data, buffer_size)
        if k % 3 == 0:
            rc, got, _, _ = device_spans(gpu_lib, torch, data, pattern, buffer_size)
            assert rc == 0 and got == expected, ("device", pattern, data, buffer_size)
        checked += 1
    assert checked >= 300, checked
    # many segments, from host and device memory (a segment holds at least two pseudo-lines of buffer_size - 1 bytes)
    rng = random.Random(5)
    data = b"".join(random_text(rng, rng.randint(0, 200)) for _ in range(400))
    for pattern in [b"(a|ab)(c|bcd)?", b"a+?b", b"\\b[ab]+\\B", b"[^a]{2,}"]:
        expected = oracle_spans(data, pattern, 256)
        for chunk in ("4096", "16384"):
            monkeypatch.setenv("GPUGREP_CHUNK_BYTES", chunk)
            rc, got, _, stats = host_spans(gpu_lib, data, pattern, 256)
            assert rc == 0 and got == expected and stats.segments > 1, (pattern, chunk)
            rc, got, _, _ = device_spans(gpu_lib, torch, data, pattern, 256)
            assert rc == 0 and got == expected, (pattern, chunk, "device")
        monkeypatch.delenv("GPUGREP_CHUNK_BYTES")


@pytest.mark.gpu
def test_gpu_spans_of_config_text(gpu_lib, torch):
    from hypergrep_b200 import synth  # pylint: disable=import-outside-toplevel

    data = synth.syslog_bytes(64 << 20, seed=23)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    lines = data.split(b"\n")
    for pattern in PROBE_PATTERNS:
        compiled = re.compile(pattern.encode())
        expected = [(k, m.start(), m.end()) for k, line in enumerate(lines) for m in compiled.finditer(line)]
        # (each block also holds its '\n', which none of these patterns can match)
        rc, got, found, stats = match_spans(gpu_lib, dev.data_ptr(), len(data), DEVICE, pattern.encode())
        assert rc == 0 and found == len(expected) and got == expected, pattern
        rc, got, found, _ = host_spans(gpu_lib, data, pattern.encode())
        assert rc == 0 and got == expected, pattern
        assert stats.gpu_ms > 0


@pytest.mark.gpu
def test_gpu_line_at_the_pseudo_line_limit_and_sentinel(gpu_lib, torch):
    rng = random.Random(9)
    limit = 262139
    long_line = bytes(rng.choice(b"ab c") for _ in range(limit - 1)) + b"\n"
    data = b"ab abb\n" + long_line + bytes(rng.choice(b"ab c") for _ in range(limit + 500)) + b"\nab\n"
    for pattern in [b"a+b", b"(a|ab)(c|b )", b"\\bab*?\\b"]:
        expected = oracle_spans(data, pattern)
        rc, got, _, _ = host_spans(gpu_lib, data, pattern)
        assert rc == 0 and got == expected, pattern
        rc, got, _, _ = device_spans(gpu_lib, torch, data, pattern)
        assert rc == 0 and got == expected, pattern
    data = b"ab a\n" + b"a" * 20000 + b"\n" + b"xa ab\n"
    expected = [s for s in oracle_spans(data, b"a.*b|a") if s[0] != 1]
    rc, got, found, _ = host_spans(gpu_lib, data, b"a.*b|a")
    assert rc == 0 and got == expected[:2] + [(1, OVER, OVER)] + expected[2:], got[:6]
    rc, got, found, _ = host_spans(gpu_lib, data, b"port [0-9]+", capacity=0)
    assert rc == 0 and found == 0


@pytest.mark.gpu
def test_gpu_grep_only_matching_takes_the_span_route(gpu_lib, tmp_path, monkeypatch):
    check_grep_spans(gpu_lib, tmp_path, monkeypatch, expect_route=True)
