"""Whole-word and whole-line fixed strings (grep -F -w / -F -x): gpugrep_literal_whole_scan_file / _buffer, the `word_regexp`
and `line_regexp` keywords of scan() / grep() / parallel_grep() and the CLI's -w / -x.

The expected answer is the one include/gpugrep.h defines.  Two routes give it without sharing any code with the engine:
 - the regex route: each literal written as \\xHH escapes inside (?:^|[^0-9A-Za-z_])...(?:[^0-9A-Za-z_]|$) (word) or ^...$
   (line; literals holding a '\\n' are left out first, since ^a\\n$ would match the line a\\n), with the literal's flags plus
   SINGLEMATCH and id 0, scanned by the PCRE2 oracle, by the context stand-in (tests/mock_engine_context) and, on the GPU,
   by the CUDA engine's own regex scan;
 - a Python model (`model_selected`): per pseudo-line, re with look-arounds over the scanned block.
CPU tests run the host logic on the whole-word / whole-line stand-in (tests/mock_engine_literal_whole), which filters the
fixed-string stand-in's selection with memmem and an explicit boundary check; `gpu` tests run the CUDA engine (fast and
general path)."""

from __future__ import annotations

import ctypes
import gzip
import os
import random
import re
import shutil
import subprocess

import numpy as np
import pytest

import byte_cases
import parity
from gpu_api import Stats, marshal
from hypergrep_b200 import synth
from oracle_api import CALLBACK, run_scan
from test_fixed_strings import EDGE_TEXTS, block_of, literal_scan, literal_scan_buffer, pseudo_lines

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WHOLE_LIB = os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal_whole.so")
WORD, LINE = 1, 2
_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
              ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint, ctypes.c_void_p,
                ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
_CTX_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int,
                  ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
# prefixes, suffixes and overlaps of one another, duplicates, caseless copies, '\n'-ended and inner-'\n' ones, high bytes,
# non-word first / last bytes, and the whole texts of some edge lines
EDGE_SET = ([b"foo", b"fo", b"oo", b"foobar", b"FOO", b"bar\n", b"bar", b"ab\nc", b"\xff\xfe", b"\xff", b"`", b"@", b"a a", b"ab", b"AbAbA",
             b"0123456", b"obar", b"foo bar", b"[{", b"x" * 700 + b"foo", b"foo\r", b"_foo", b"foo.", b"b"],
            [0, 0, 0, 0, 1, 0, 8, 0, 0, 2, 1, 0, 0, 0, 9, 0, 0, 14, 1, 0, 0, 0, 0, 1])
# the high-byte alphabet of the byte tests (high, control and near-miss bytes around newlines and NULs)
ALPHABET_TEXT = byte_cases.byte_text(random.Random(7), 300, nul_rate=0.02)


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


def _lits(literals, flags):
    n = len(literals)
    arr = (ctypes.c_char_p * max(n, 1))(*literals)
    fl = (ctypes.c_uint * max(n, 1))(*flags) if flags is not None else None
    return arr, fl, n


def whole_scan(lib, path, literals, flags, whole, buffer_size=262140, buffer_count=16, max_match_count=0, before=0, after=0, invert=False,
               collect=True):
    entry = lib.gpugrep_literal_whole_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    la, fa, n = _lits(literals, flags)
    sink, stats = _Collector(collect), Stats()
    rc = entry(str(path).encode(), la, fa, n, whole, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def whole_scan_buffer(lib, ptr, size, location, literals, flags, whole, buffer_size=262140, buffer_count=16, max_match_count=0, before=0,
                      after=0, invert=False, collect=True):
    entry = lib.gpugrep_literal_whole_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    la, fa, n = _lits(literals, flags)
    sink, stats = _Collector(collect), Stats()
    rc = entry(ptr, size, location, la, fa, n, whole, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               None, ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def regex_set(literals, flags, whole):
    """The regex route: one pattern per literal (flags | SINGLEMATCH, ids 0).  Line mode leaves literals with a '\\n' out."""
    pats, fl = [], []
    for lit, flag in zip(literals, flags or [0] * len(literals)):
        body = "".join(f"\\x{b:02x}" for b in lit)
        if whole == LINE:
            if b"\n" in lit:
                continue
            pats.append(f"^(?:{body})$")
        else:
            pats.append(f"(?:^|[^0-9A-Za-z_])(?:{body})(?:[^0-9A-Za-z_]|$)")
        fl.append(flag | 8)
    return pats, fl


def oracle_records(oracle_lib, path, literals, flags, whole, **kw):
    """PCRE2 oracle (hyperscan()) of the regex route: the records of a whole scan without context or inversion."""
    pats, fl = regex_set(literals, flags, whole)
    if not pats:
        return 0, [], []
    return run_scan(oracle_lib, str(path), pats, flags=fl, ids=[0] * len(pats), **kw)


def regex_context(lib, path, literals, flags, whole, buffer_size=262140, buffer_count=16, max_match_count=0, before=0, after=0,
                  invert=False, collect=True):
    """gpugrep_context_scan_file of the regex route (the context stand-in on the CPU, the CUDA engine on the GPU)."""
    pats, fl = regex_set(literals, flags, whole)
    if not pats:   # nothing can match: every line is a line without a match
        pats, fl = ["\\x00\\x00"], [8]
    pa, fa, ia, n = marshal(pats, fl, [0] * len(pats))
    entry = lib.gpugrep_context_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _CTX_FILE_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(str(path).encode(), pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def _model_regex(literals, flags, whole):
    parts = []
    for lit, flag in zip(literals, flags or [0] * len(literals)):
        if whole == LINE and b"\n" in lit:
            continue
        body = re.escape(lit)
        parts.append(b"(?i:" + body + b")" if flag & 1 else body)
    if not parts:
        return None
    alt = b"|".join(parts)
    if whole == LINE:
        return re.compile(b"(?:" + alt + b")\\n?\\Z")
    return re.compile(b"(?<![0-9A-Za-z_])(?:" + alt + b")(?![0-9A-Za-z_])")


def model_selected(data: bytes, literals, flags, whole, buffer_size: int = 262140) -> list[bool]:
    """The definition, with Python's re: per pseudo-line, a look-around search (word) or a full match of the block without
    its final '\\n' (line) over the scanned block.  re's IGNORECASE on bytes folds A-Z / a-z only."""
    pattern = _model_regex(literals, flags, whole)
    out = []
    for line in pseudo_lines(data, buffer_size):
        block = block_of(line)
        if pattern is None:
            out.append(False)
        elif whole == LINE:
            out.append(pattern.match(block) is not None)
        else:
            out.append(pattern.search(block) is not None)
    return out


def model_lines(data: bytes, literals, flags, whole, buffer_size: int = 262140) -> list[int]:
    return [k for k, hit in enumerate(model_selected(data, literals, flags, whole, buffer_size)) if hit]


def _numbers(records) -> list[int]:
    assert all(r[0] == 0 for r in records)
    return [r[1] for r in records]


@pytest.fixture(scope="session")
def whole_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal_whole")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(WHOLE_LIB)


@pytest.fixture(scope="session")
def literal_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal.so"))


@pytest.fixture(scope="session")
def context_mock_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_context")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_context.so"))


def random_set(rng: random.Random, count: int):
    """Prefixes, suffixes, overlaps, duplicates, caseless copies and '\\n'-holding literals over a small alphabet with word and
    non-word bytes, high bytes included."""
    lits = []
    while len(lits) < count:
        r = rng.random()
        if lits and r < 0.2:
            base = rng.choice(lits)
            lits.append(base[:rng.randint(1, len(base))])          # a prefix
        elif lits and r < 0.3:
            base = rng.choice(lits)
            lits.append(base[rng.randint(0, len(base) - 1):])      # a suffix
        elif lits and r < 0.38:
            lits.append(rng.choice(lits))                          # a duplicate
        elif lits and r < 0.48:
            lits.append(rng.choice(lits) + bytes(rng.choice(b"aB_ .\n") for _ in range(rng.randint(1, 2))))   # an extension
        else:
            lits.append(bytes(rng.choice(b"abAB_09 .-@`[{\x80\xff") for _ in range(rng.randint(1, 6))))
    return lits, [rng.choice((0, 1, 2, 4, 8, 9, 14, 15)) for _ in lits]


def random_text(rng: random.Random, size: int, lits) -> bytes:
    parts, total = [], 0
    while total < size:
        r = rng.random()
        if r < 0.3:
            parts.append(rng.choice(lits))
        elif r < 0.45:
            parts.append(b"\n")
        elif r < 0.47:
            parts.append(b"\0")
        else:
            parts.append(bytes(rng.choice(b"abAB_09 .-@`[{\x80\xff") for _ in range(rng.randint(0, 4))))
        total += len(parts[-1])
    return b"".join(parts)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("whole", [WORD, LINE])
@pytest.mark.parametrize("name", sorted(EDGE_TEXTS) + ["alphabet"])
@pytest.mark.parametrize("buffer_size", [4, 9, 262140])
def test_edge_texts_against_the_oracle(name, buffer_size, whole, whole_lib, oracle_lib, tmp_path):
    text = ALPHABET_TEXT if name == "alphabet" else EDGE_TEXTS[name]
    data = text + b"foobar FOO\nfoo\nfoo bar\n_foo foo.\nxfoo foobar\nba a a\naab ab\n\xfffoo\xff\n"
    path = tmp_path / "t.log"
    path.write_bytes(data)
    lits, flags = EDGE_SET
    got = whole_scan(whole_lib, path, lits, flags, whole, buffer_size=buffer_size)
    want = oracle_records(oracle_lib, path, lits, flags, whole, buffer_size=buffer_size)
    assert got[0] == want[0] == 0 and got[1] == want[1]
    assert _numbers(got[1]) == model_lines(data, lits, flags, whole, buffer_size)


def test_gnu_grep_examples(whole_lib, tmp_path):
    """The cases from the issue that GNU grep 3.11 selects, and their near misses."""
    path = tmp_path / "g.log"
    path.write_bytes(b"xfoo foobar\nba a a\naab ab\nxfoo foobarx\n10.1.2.3\n110.1.2.34\nab\n")
    assert [r[1] for r in whole_scan(whole_lib, path, [b"foo", b"foobar"], [0, 0], WORD)[1]] == [0]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"a a"], [0], WORD)[1]] == [1]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"ab"], [0], WORD)[1]] == [2, 6]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"10.1.2.3"], [0], WORD)[1]] == [4]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"ab", b"10.1.2.3", b"ab\n"], [0, 0, 0], LINE)[1]] == [4, 6]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"AB"], [1], LINE)[1]] == [6]


@pytest.mark.parametrize("seed", range(10))
def test_random_sets_limits_batches_invert_and_context(seed, whole_lib, oracle_lib, context_mock_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    rng = random.Random(seed)
    lits, flags = random_set(rng, rng.randint(1, 25))
    data = random_text(rng, 12_000, lits)
    path = tmp_path / "r.log"
    path.write_bytes(data)
    for whole in (WORD, LINE):
        assert whole_scan(whole_lib, path, lits, flags, whole)[1] == oracle_records(oracle_lib, path, lits, flags, whole)[1]
        assert _numbers(whole_scan(whole_lib, path, lits, flags, whole)[1]) == model_lines(data, lits, flags, whole)
        for kw in ({}, {"max_match_count": 7, "buffer_count": 3}, {"max_match_count": 1}, {"buffer_size": 17}, {"invert": True},
                   {"invert": True, "max_match_count": 5}, {"before": 2, "after": 1}, {"after": 1, "max_match_count": 4},
                   {"before": 1, "invert": True, "buffer_size": 9}):
            want = regex_context(context_mock_lib, path, lits, flags, whole, **kw)
            got = whole_scan(whole_lib, path, lits, flags, whole, **kw)
            assert got[0] == want[0] == 0 and got[1:3] == want[1:3], (whole, kw)
            counted = whole_scan(whole_lib, path, lits, flags, whole, collect=False, **kw)
            assert counted[0] == 0 and counted[3].matches == regex_context(context_mock_lib, path, lits, flags, whole, collect=False,
                                                                          **kw)[3].matches, (whole, kw)


@pytest.mark.parametrize("seed", range(3))
def test_larger_random_sets_against_the_python_model(seed, whole_lib, tmp_path):
    rng = random.Random(100 + seed)
    lits, flags = random_set(rng, 300)
    data = random_text(rng, 200_000, lits)
    path = tmp_path / "m.log"
    path.write_bytes(data)
    for whole in (WORD, LINE):
        for buffer_size in (262140, 11):
            got = whole_scan(whole_lib, path, lits, flags, whole, buffer_size=buffer_size)
            assert got[0] == 0 and _numbers(got[1]) == model_lines(data, lits, flags, whole, buffer_size)
        assert whole_scan(whole_lib, path, lits, flags, whole)[1]


def test_compressed_and_sharded(whole_lib, context_mock_lib, tmp_path, monkeypatch):
    text = synth.syslog_bytes(1 << 20, seed=3)
    lits = [b"Failed password", b"sshd", b"port 22", b"SESSION", b"error", b"\xff\xfe", b"root"]
    flags = [0, 0, 0, 1, 0, 0, 9]
    plain = tmp_path / "p.log"
    plain.write_bytes(text)
    for whole in (WORD, LINE):
        want = regex_context(context_mock_lib, plain, lits, flags, whole)
        if whole == WORD:
            assert len(want[1]) > 100
        gz = tmp_path / "p.log.gz"
        gz.write_bytes(gzip.compress(text))
        assert whole_scan(whole_lib, gz, lits, flags, whole)[:3] == want[:3]
        for name, blob in parity.zstd_cases(text).items():
            path = tmp_path / f"{name}.log.zst"
            path.write_bytes(blob)
            assert whole_scan(whole_lib, path, lits, flags, whole)[:3] == regex_context(context_mock_lib, path, lits, flags, whole)[:3], name
        host = ctypes.create_string_buffer(text, len(text))
        assert whole_scan_buffer(whole_lib, ctypes.addressof(host), len(text), 0, lits, flags, whole)[:3] == want[:3]
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_MOCK_DEVICES", "3")
            env.setenv("GPUGREP_DEVICES", "all")
            env.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
            assert whole_scan(whole_lib, plain, lits, flags, whole)[:3] == want[:3]
            assert whole_scan_buffer(whole_lib, ctypes.addressof(host), len(text), 0, lits, flags, whole)[:3] == want[:3]
            for kw in ({"max_match_count": 50, "buffer_count": 7}, {"invert": True, "max_match_count": 30}, {"before": 1, "after": 2}):
                assert whole_scan(whole_lib, plain, lits, flags, whole, **kw)[:3] == regex_context(context_mock_lib, plain, lits, flags,
                                                                                                 whole, **kw)[:3], kw
            assert whole_scan(whole_lib, plain, lits, flags, whole, collect=False)[3].matches == len(want[1])


def test_return_codes(whole_lib, literal_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(b"foo\nbar\n")
    for whole in (0, 3, 4, 1 << 31):
        assert whole_scan(whole_lib, path, [b"foo"], [0], whole)[0] == 4
    for whole in (WORD, LINE):
        assert whole_scan(whole_lib, path, [b"foo", b""], [0, 0], whole)[0] == 4
        assert whole_scan(whole_lib, path, [], [], whole)[0] == 4
        for bit in (16, 32, 1 << 31):
            assert whole_scan(whole_lib, path, [b"foo"], [bit | 1], whole)[0] == 4
        for bits in (2, 4, 8, 14, 15):   # accepted, and change nothing but CASELESS
            assert whole_scan(whole_lib, path, [b"FOO"], [bits], whole)[:2] == (0, [(0, 0, b"foo\n")] if bits & 1 else [])
        assert whole_scan(whole_lib, path, [b"foo"], None, whole)[:2] == (0, [(0, 0, b"foo\n")])
        # an engine without the whole-word / whole-line stage
        assert whole_scan(literal_lib, path, [b"foo"], [0], whole)[0] == 7
        assert whole_scan(literal_lib, path, [b""], [0], whole)[0] == 4


def test_whole_and_plain_sets_are_cached_apart(whole_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(b"foobar\nfoo\n")
    lits = [b"foo", b"foobar"]
    assert [r[1] for r in literal_scan(whole_lib, str(path), lits, [0, 0])[1]] == [0, 1]
    assert [r[1] for r in whole_scan(whole_lib, path, lits, [0, 0], WORD)[1]] == [0, 1]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"foo"], [0], WORD)[1]] == [1]
    assert [r[1] for r in whole_scan(whole_lib, path, [b"foo"], [0], LINE)[1]] == [1]
    assert [r[1] for r in literal_scan(whole_lib, str(path), [b"foo"], [0])[1]] == [0, 1]


@pytest.fixture()
def py_on_mock(whole_lib, monkeypatch):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    monkeypatch.setenv("GPUGREP_LIBRARY", WHOLE_LIB)
    monkeypatch.setitem(utils._state, "lib", None)  # pylint: disable=protected-access
    return utils


def _records(function, *args, **kw):
    out = []

    def cb(matches, count):
        out.extend((matches[k].id, matches[k].line_number, matches[k].line) for k in range(count))

    rc = function(*args, cb, **kw)
    return rc, out


def test_python_keywords(py_on_mock, tmp_path):
    utils = py_on_mock
    path = tmp_path / "k.log"
    path.write_bytes("a.b x\nxa.b\nA.B\n(x+ é\né\nnone\n".encode())
    lits = ["a.b", "é", "(x+"]
    flags = [9, 8, 8]
    assert _records(utils.scan, str(path), lits, flags=flags, fixed_strings=True, word_regexp=True) == \
        (0, [(0, 0, b"a.b x\n"), (0, 2, b"A.B\n"), (0, 3, "(x+ é\n".encode()), (0, 4, "é\n".encode())])
    assert _records(utils.scan, str(path), lits, flags=flags, fixed_strings=True, line_regexp=True) == \
        (0, [(0, 2, b"A.B\n"), (0, 4, "é\n".encode())])
    # both: the line test wins
    assert _records(utils.scan, str(path), lits, flags=flags, fixed_strings=True, word_regexp=True, line_regexp=True) == \
        _records(utils.scan, str(path), lits, flags=flags, fixed_strings=True, line_regexp=True)
    assert utils.grep(str(path), lits, fixed_strings=True, word_regexp=True, ignore_case=True) == \
        ([(1, "a.b x\n"), (3, "A.B\n"), (4, "(x+ é\n"), (5, "é\n")], 0)
    assert utils.grep(str(path), lits, fixed_strings=True, word_regexp=True) == ([(1, "a.b x\n"), (4, "(x+ é\n"), (5, "é\n")], 0)
    assert utils.grep(str(path), lits, fixed_strings=True, line_regexp=True, count_only=True) == (1, 0)
    assert utils.grep(str(path), lits, fixed_strings=True, line_regexp=True, invert_match=True, count_only=True) == (5, 0)
    assert utils.grep(str(path), lits, fixed_strings=True, word_regexp=True, max_match_count=2) == ([(1, "a.b x\n"), (4, "(x+ é\n")], 0)
    assert utils.grep(str(path), ["é"], fixed_strings=True, line_regexp=True, after_context=1) == \
        ([(5, "é\n", False), (6, "none\n", True)], 0)
    for kw in ({"word_regexp": True}, {"line_regexp": True}):
        with pytest.raises(ValueError):
            utils.scan(str(path), lits, lambda *_: None, **kw)
        with pytest.raises(ValueError):
            utils.grep(str(path), lits, **kw)
        with pytest.raises(ValueError):
            utils.grep(str(path), lits, fixed_strings=True, only_matching=True, **kw)
        with pytest.raises(ValueError):
            utils.grep(str(path), lits, fixed_strings=True, only_matching=True, invert_match=True, **kw)


_SYSTEM_GREP = shutil.which("grep")


def _cli(monkeypatch, capsys, argv):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel
    monkeypatch.setattr("sys.argv", ["hyperscanner"] + argv)
    with pytest.raises(SystemExit) as done:
        multiscanner.main()
    return done.value.code, capsys.readouterr().out


def test_cli_options_and_usage_errors(py_on_mock, monkeypatch, capsys, tmp_path):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel
    args = multiscanner.parse_args(["-F", "-w", "-x", "x", "f"])
    assert args.word_regexp and args.line_regexp
    path = tmp_path / "c.log"
    path.write_bytes(b"a.b\nxa.b\na.b c\n")
    assert _cli(monkeypatch, capsys, ["-F", "-w", "a.b", str(path)]) == (0, "a.b\na.b c\n")
    assert _cli(monkeypatch, capsys, ["-F", "--line-regexp", "-n", "a.b", str(path)]) == (0, "1:a.b\n")
    assert _cli(monkeypatch, capsys, ["-F", "-x", "-w", "-c", "a.b", str(path)]) == (0, "1\n")
    for argv in (["-w", "a.b"], ["-x", "a.b"], ["-E", "-w", "a"], ["-F", "-w", "-o", "a.b"], ["-F", "-x", "-o", "-v", "a.b"]):
        code, out = _cli(monkeypatch, capsys, argv + [str(path)])
        assert code == 2 and out.count("\n") == 1, argv
    from hypergrep_b200.multiscanner import parallel_grep  # pylint: disable=import-outside-toplevel
    with pytest.raises(ValueError):
        parallel_grep([str(path)], ["a.b"], word_regexp=True)
    assert parallel_grep([str(path)], ["a.b"], fixed_strings=True, line_regexp=True, count_results=True) == 0
    assert capsys.readouterr().out == "1\n"


@pytest.mark.skipif(_SYSTEM_GREP is None, reason="no system grep")
@pytest.mark.parametrize("seed", range(3))
def test_cli_against_system_grep(seed, py_on_mock, monkeypatch, capsys, tmp_path):
    rng = random.Random(seed)
    words = [b"alpha", b"Beta", b"gamma.x", b"de(lta", b"EPS", b"zz", b"10.1.2.3", b"alpha_2", b"xalpha"]
    lines = [b" ".join(rng.choice(words + [b"filler", b"x y", b"110.1.2.34"]) for _ in range(rng.randint(0, 3))) for _ in range(300)]
    path = tmp_path / "s.log"
    path.write_bytes(b"\n".join(lines) + b"\n")
    other = tmp_path / "empty.log"
    other.write_bytes(b"nothing here\n")
    plist = tmp_path / "iocs.txt"
    plist.write_bytes(b"\n".join(rng.sample(words, 3)) + b"\n")
    for mode in ("-w", "-x"):
        for opts in ([], ["-c"], ["-v"], ["-n"], ["-i"], ["-A", "1", "-B", "2"], ["-l"], ["-i", "-v", "-c"], ["-m", "3", "-n"]):
            files = [str(path), str(other)] if "-l" in opts else [str(path)]
            argv = ["-F", mode] + opts + ["-f", str(plist)] + files
            want = subprocess.run([_SYSTEM_GREP] + argv, capture_output=True, text=True, check=False, env={"LC_ALL": "C"})
            code, out = _cli(monkeypatch, capsys, argv)
            assert (code, out) == (want.returncode, want.stdout), (mode, opts)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _device(data: bytes):
    import torch  # pylint: disable=import-outside-toplevel
    dev = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return dev


def _gpu_compare(gpu_lib, data: bytes, lits, flags, whole, tmp_path, kinds=("file", "host", "pinned", "device"), **kw):
    """Whole scan == the CUDA engine's regex route on every input kind; returns the records and the last stats."""
    path = tmp_path / "g.log"
    path.write_bytes(data)
    want = regex_context(gpu_lib, path, lits, flags, whole, **kw)
    assert want[0] == 0
    got = whole_scan(gpu_lib, path, lits, flags, whole, **kw)
    assert got[:3] == want[:3]
    if "host" in kinds:
        host = ctypes.create_string_buffer(data, len(data) + 1)
        assert whole_scan_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, lits, flags, whole, **kw)[:3] == want[:3]
    if "pinned" in kinds:
        import torch  # pylint: disable=import-outside-toplevel
        pinned = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).pin_memory()
        assert whole_scan_buffer(gpu_lib, pinned.data_ptr(), len(data), 0, lits, flags, whole, **kw)[:3] == want[:3]
    if "device" in kinds:
        dev = _device(data)
        got = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, whole, **kw)
        assert got[:3] == want[:3]
        counted = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, whole, collect=False, **kw)
        assert counted[0] == 0 and counted[3].matches == regex_context(gpu_lib, path, lits, flags, whole, collect=False, **kw)[3].matches
    return want[1], got[3]


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_edges_alphabet_and_oracle(force_general, gpu_lib, oracle_lib, tmp_path, monkeypatch):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    lits, flags = EDGE_SET
    for whole in (WORD, LINE):
        for name, text in list(EDGE_TEXTS.items()) + [("alphabet", ALPHABET_TEXT)]:
            data = text + b"foobar FOO\nxfoo foobar\nfoo\n"
            for buffer_size in (9, 262140):
                recs, _ = _gpu_compare(gpu_lib, data, lits, flags, whole, tmp_path, kinds=("file", "device"), buffer_size=buffer_size)
                assert _numbers(recs) == model_lines(data, lits, flags, whole, buffer_size), (whole, name, buffer_size)
                assert recs == oracle_records(oracle_lib, tmp_path / "g.log", lits, flags, whole, buffer_size=buffer_size)[1]
        _gpu_compare(gpu_lib, EDGE_TEXTS["inner_nul"] * 50, lits, flags, whole, tmp_path, before=1, after=1)
        _gpu_compare(gpu_lib, EDGE_TEXTS["crlf"] * 50, lits, flags, whole, tmp_path, invert=True, max_match_count=20)


def _planted_syslog(size: int, seed: int, lits: list[bytes], every: int = 37):
    """syslog with literals planted as words, inside longer words, at line ends, as whole lines and behind NULs."""
    rng = random.Random(seed)
    lines = synth.syslog_bytes(size, seed=seed).split(b"\n")
    for k in range(0, len(lines), every):
        lit = rng.choice(lits).replace(b"\n", b"")
        form = k // every % 6
        if form == 0:
            lines[k] += b" ioc=" + lit + b" end"
        elif form == 1:
            lines[k] += b" x" + lit + b"y"                # inside a longer word: no word match
        elif form == 2:
            lines[k] += b" " + lit                        # at the line end
        elif form == 3:
            lines[k] = lit                                # the whole line
        elif form == 4:
            lines[k] += b"\0" + lit + b" "                # behind a NUL: outside the scanned block
        else:
            lines[k] = b"\0\0" + lit                      # the whole scanned block after leading NULs
    return b"\n".join(lines)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_gpu_random_sets_on_syslog(seed, gpu_lib, tmp_path, monkeypatch):
    rng = random.Random(seed)
    lits = [bytes(rng.choice(b"abcdefXYZ0123456789_.-@ \x80\xfe") for _ in range(rng.randint(4 if seed != 1 else 1, 14)))
            for _ in range(rng.choice((50, 400)))]
    lits += [lit[:rng.randint(min(4, len(lit)), len(lit))] for lit in rng.sample(lits, 20)]   # prefixes
    lits += [lit[rng.randint(0, len(lit) - 4):] for lit in rng.sample(lits, 10) if len(lit) >= 4]   # suffixes
    lits += [b"Failed password for", b"Failed", b"sshd", b"port 22\n", b"error", b"session opened"]
    flags = [rng.choice((0, 1, 8, 9, 14)) for _ in lits]
    data = _planted_syslog(4 << 20, seed, lits)
    for whole in (WORD, LINE):
        recs, stats = _gpu_compare(gpu_lib, data, lits, flags, whole, tmp_path, buffer_count=4096)
        assert len(recs) > (1000 if whole == WORD else 100)
        if seed != 1:
            assert stats.path & 1
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_FORCE_GENERAL", "1")
            _gpu_compare(gpu_lib, data, lits, flags, whole, tmp_path, kinds=("device",), buffer_count=4096, max_match_count=3000)
            _gpu_compare(gpu_lib, data, lits, flags, whole, tmp_path, kinds=("device",), invert=True, before=1)


@pytest.mark.gpu
def test_gpu_sharded_and_compressed(gpu_lib, tmp_path, monkeypatch):
    import torch  # pylint: disable=import-outside-toplevel
    lits = [b"Failed password", b"sshd", b"port 22", b"SESSION", b"error", b"root"]
    flags = [0, 0, 0, 1, 0, 9]
    data = _planted_syslog(16 << 20, 5, lits)
    path = tmp_path / "s.log"
    path.write_bytes(data)
    for whole in (WORD, LINE):
        want = regex_context(gpu_lib, path, lits, flags, whole)
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_DEVICES", ",".join(["0"] * 3) if torch.cuda.device_count() == 1 else "all")
            env.setenv("GPUGREP_MIN_SHARD_BYTES", str(1 << 20))
            assert whole_scan(gpu_lib, path, lits, flags, whole)[:3] == want[:3]
            host = ctypes.create_string_buffer(data, len(data))
            assert whole_scan_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, lits, flags, whole)[:3] == want[:3]
        gz = tmp_path / "s.log.gz"
        gz.write_bytes(gzip.compress(data, compresslevel=1))
        assert whole_scan(gpu_lib, gz, lits, flags, whole)[:3] == want[:3]
        for name, blob in list(parity.zstd_cases(data).items())[:1]:
            zst = tmp_path / f"{name}.log.zst"
            zst.write_bytes(blob)
            assert whole_scan(gpu_lib, zst, lits, flags, whole)[:3] == want[:3]


def ioc_set(count: int, seed: int) -> list[bytes]:
    """IPv4 addresses, MD5 hashes, SHA-256 hashes and domains, as tools/literal_probe.py models them."""
    rng = np.random.default_rng(seed)
    hexd = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)
    quarter = count // 4
    iocs = [f"{a}.{b}.{c}.{d}".encode() for a, b, c, d in rng.integers(1, 255, size=(quarter, 4))]
    iocs += [rng.choice(hexd, size=32).tobytes() for _ in range(quarter)]
    iocs += [rng.choice(hexd, size=64).tobytes() for _ in range(quarter)]
    letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    iocs += [rng.choice(letters, size=int(rng.integers(5, 12))).tobytes() + b"." + rng.choice([b"com", b"net", b"io"])
             for _ in range(count - len(iocs))]
    return iocs


def model_ioc_lines(data: bytes, literals: list[bytes], selected: list[int], whole: int, buffer_size: int = 262140) -> list[int]:
    """The definition over the lines that the plain fixed-string scan selected (a superset), with a dict of literals by
    length: every start that no word byte precedes, every literal length, a word-byte test behind the end (word); the
    block without its '\\n' in the set (line)."""
    lits = set(literals)
    lengths = sorted({len(lit) for lit in lits})
    lines = pseudo_lines(data, buffer_size)
    word = set(b"0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz_")
    out = []
    for k in selected:
        block = block_of(lines[k])
        if whole == LINE:
            hit = (block[:-1] if block.endswith(b"\n") else block) in lits
        else:
            hit = any(block[s:s + n] in lits and (s + n == len(block) or block[s + n] not in word)
                      for s in range(len(block)) if s == 0 or block[s - 1] not in word for n in lengths)
        if hit:
            out.append(k)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("count", [10_000, 100_000])
def test_gpu_ioc_sets_against_a_python_model(count, gpu_lib):
    iocs = ioc_set(count, count)
    rng = random.Random(count)
    data = _planted_syslog(32 << 20, 11, [rng.choice(iocs) for _ in range(500)], every=29)
    # near misses: IPs with a digit in front or behind, hashes inside longer hex runs
    data += b"".join(b"src=1" + rng.choice(iocs) + b"4 dst=" + rng.choice(iocs) + b"_\n" for _ in range(300))
    dev = _device(data)
    flags = [0] * len(iocs)
    plain = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, flags, buffer_count=1 << 16)
    assert plain[0] == 0
    selected = [r[1] for r in plain[1]]
    for whole in (WORD, LINE):
        want = model_ioc_lines(data, iocs, selected, whole)
        rc, recs, _, stats = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, flags, whole, buffer_count=1 << 16)
        assert rc == 0 and [r[1] for r in recs] == want
        assert len(want) >= 1000 and len(want) < len(selected) and stats.path & 1
        counted = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, flags, whole, collect=False)
        assert counted[3].matches == len(want) and counted[3].path & 1
        inverted = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, flags, whole, invert=True, collect=False)
        assert inverted[3].matches == plain[3].lines - len(want)


@pytest.mark.gpu
def test_gpu_dense_reject_filter_and_dedupe(gpu_lib, tmp_path):
    """Many candidate chunks and records per line, nearly all rejected: every line is counted and delivered once."""
    data, words = synth.dense_reject_bytes(200_000, 1)
    lits, flags = [b"error"], [0]
    dev = _device(data)
    plain = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags)
    assert len(plain[1]) == 200_000 and plain[3].path & 1
    rc, recs, _, stats = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, WORD)
    assert rc == 0 and [r[1] for r in recs] == words and stats.path & 1
    assert stats.launches == plain[3].launches + 1
    counted = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, WORD, collect=False)
    assert counted[3].matches == len(words) and counted[3].path & 1
    inverted = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, WORD, invert=True)
    assert [r[1] for r in inverted[1]] == sorted(set(range(200_000)) - set(words))
    ctx = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, WORD, before=1, after=1)
    path = tmp_path / "d.log"
    path.write_bytes(data)
    assert ctx[1] == regex_context(gpu_lib, path, lits, flags, WORD, before=1, after=1)[1]
    line = data.split(b"\n")[7]
    assert [r[1] for r in whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, [line], flags, LINE)[1]] == \
        [k for k, text in enumerate(data.split(b"\n")[:-1]) if text == line]


@pytest.mark.gpu
def test_gpu_launch_pins(gpu_lib):
    """Regex scans keep the C2 pins, plain fixed-string and report scans keep their launches and paths, and a whole scan on
    the fast path is the plain scan plus one launch (count-only too: it emits records instead of keys)."""
    from test_fixed_strings import C2_REGEX_PIN  # pylint: disable=import-outside-toplevel
    from test_literal_reports import report_scan_buffer  # pylint: disable=import-outside-toplevel
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
    counted = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, collect=False)
    reports = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, [14] * 3, [0] * 3)
    assert plain[3].path == counted[3].path == reports[3].path == 1
    assert reports[3].launches == plain[3].launches + 5 and counted[3].launches == plain[3].launches
    for whole in (WORD, LINE):
        w = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, None, whole)
        c = whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, None, whole, collect=False)
        assert w[3].path == c[3].path == 1
        assert w[3].launches == plain[3].launches + 1 and c[3].launches == counted[3].launches + 1
        assert c[3].matches == len(w[1])
    assert len(whole_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, None, WORD)[1]) == len(plain[1])


@pytest.mark.gpu
def test_gpu_grep_word_regexp_on_the_cuda_library(tmp_path):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    iocs = ioc_set(10_000, 3)
    lits = [lit.decode() for lit in iocs]
    lines = synth.syslog_bytes(4 << 20, seed=4).decode(errors="replace").split("\n")
    for k in range(0, len(lines), 97):
        lines[k] += f" ioc={lits[k % 1000]}" if k % 2 else f" ioc=x{lits[k % 1000]}"
    path = tmp_path / "f.log"
    path.write_text("\n".join(lines))
    got, code = utils.grep(str(path), lits, fixed_strings=True, word_regexp=True)
    want = [(number + 1, line + "\n") for number, line in enumerate(lines[:-1]) if number % 97 == 0 and number % 2]
    assert code == 0 and got == want and len(want) > 100
