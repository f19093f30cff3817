"""Context lines (grep -A/-B/-C): gpugrep_context_scan_file / gpugrep_context_scan_buffer, scan()/grep() with before_context /
after_context and the CLI's -A/-B/-C.  The expected answer comes from the unchanged oracle: its normal scan says which
pseudo-lines match, a scan for `.` reads every pseudo-line with its stripped text, and `context_model` applies the semantics
(window, invert, the trailing context after max_match_count, batching).  CPU tests run the host logic on the CPU engine
stand-in with context lines (tests/mock_engine_context); `gpu` tests run the CUDA engine (fast and general path)."""

from __future__ import annotations

import ctypes
import os
import random
import shutil
import subprocess
import sys
import zlib

import numpy as np
import pytest

import parity
from gpu_api import Stats, marshal, scan_buffer
from hypergrep_b200 import synth
from oracle_api import CALLBACK, run_scan
from test_host_logic import EDGE_TEXTS

CONTEXT_ID = 0xFFFFFFFF
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
              ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
WIDTHS = (0, 1, 2, 7, 100, 0xFFFFFFFF)


class _Collector:
    """Callback that keeps (id, line_number, line) records, or (id, line_number) and a CRC of the texts (large scans)."""

    def __init__(self, mode: str | None):
        self.mode, self.records, self.batches, self.crc = mode, [], [], 0

        def cb(results, count):
            self.batches.append(count)
            for i in range(count):
                r = results[i]
                if self.mode == "numbers":
                    self.records.append((r.id, r.line_number))
                    self.crc = zlib.crc32(r.line, self.crc)
                else:
                    self.records.append((r.id, r.line_number, r.line))

        self.c_callback = CALLBACK(cb) if mode else None

    def pointer(self):
        return ctypes.cast(self.c_callback, ctypes.c_void_p) if self.c_callback else None


def context_scan(lib, path: str, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0, before=0, after=0,
                 invert=False, collect="records"):
    """gpugrep_context_scan_file -> (rc, records or None, batch sizes, crc, stats)."""
    pa, fa, ia, n = marshal(patterns, flags, ids)
    entry = lib.gpugrep_context_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(path.encode(), pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               ctypes.byref(stats))
    return rc, (sink.records if collect else None), sink.batches, sink.crc, stats


def context_scan_buffer(lib, ptr: int, size: int, location: int, patterns, buffer_size=262140, buffer_count=4096, max_match_count=0,
                        before=0, after=0, invert=False, collect="numbers"):
    """gpugrep_context_scan_buffer -> (rc, records or None, batch sizes, crc, stats)."""
    pa, fa, ia, n = marshal(patterns, None, None)
    entry = lib.gpugrep_context_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(ptr, size, location, pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               None, ctypes.byref(stats))
    return rc, (sink.records if collect else None), sink.batches, sink.crc, stats


def context_model(selected: np.ndarray, before: int, after: int, max_match_count: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """The delivered lines of a context scan: (line numbers, is_context), from the selected-line mask of all pseudo-lines.
    A line is output iff a selected line lies in [i - after, i + before].  With a limit, the selected lines after the one
    that reaches it do not count: the `after` lines behind it are then output as context, and nothing after them."""
    sel = np.asarray(selected, dtype=bool).copy()
    if max_match_count > 0:
        hits = np.flatnonzero(sel)
        if len(hits) > max_match_count:
            sel[hits[max_match_count - 1] + 1:] = False
    n = len(sel)
    prefix = np.concatenate(([0], np.cumsum(sel, dtype=np.int64)))
    idx = np.arange(n, dtype=np.int64)
    hi = np.minimum(idx + before + 1, n)
    lo = np.maximum(idx - after, 0)
    out = prefix[hi] > prefix[lo]
    lines = np.flatnonzero(out)
    return lines, ~sel[lines]


def batches_of(total: int, buffer_count: int, max_match_count: int) -> list[int]:
    batch = buffer_count
    if 0 < max_match_count < batch:
        batch = max_match_count
    batch = max(1, batch)
    return [batch] * (total // batch) + ([total % batch] if total % batch else [])


def oracle_context(oracle, path: str, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0, before=0,
                   after=0, invert=False):
    """Expected (rc, [(id, line_number, line)], [batch sizes]) of a context scan, from the oracle (see the module docstring;
    a pseudo-line of NULs only is missing from the `.` scan: such inputs are excluded)."""
    rc, matched, _ = run_scan(oracle, path, patterns, flags=flags, ids=ids, buffer_size=buffer_size, buffer_count=4096)
    if rc != 0:
        return rc, [], []
    rc, every, _ = run_scan(oracle, path, ["."], flags=[10], ids=[0], buffer_size=buffer_size, buffer_count=4096)
    assert rc == 0
    assert [ln for _, ln, _ in every] == list(range(len(every)))
    selected = np.zeros(len(every), dtype=bool)
    selected[[ln for _, ln, _ in matched]] = True
    if invert:
        selected = ~selected
    lines, is_context = context_model(selected, before, after, max_match_count)
    records = [(CONTEXT_ID if c else 0, int(ln), every[ln][2]) for ln, c in zip(lines, is_context)]
    return rc, records, batches_of(len(records), buffer_count, max_match_count)


def compare_context(lib, oracle, data: bytes | None, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0,
                    before=0, after=0, invert=False, path: str | None = None, tmp_dir: str | None = None) -> int:
    """`lib`'s context scan == oracle_context (records, order, batches, return code, stats.matches); count-only counts the
    selected lines of the scan without context."""
    own = path is None
    if own:
        path = os.path.join(tmp_dir or "/tmp", f"context_{os.getpid()}_{random.getrandbits(48):x}.log")
        with open(path, "wb") as handle:
            handle.write(data)
    try:
        kw = {"flags": flags, "ids": ids, "buffer_size": buffer_size, "buffer_count": buffer_count, "max_match_count": max_match_count,
              "before": before, "after": after, "invert": invert}
        exp_rc, exp, exp_batches = oracle_context(oracle, path, patterns, **kw)
        rc, got, batches, _, stats = context_scan(lib, path, patterns, **kw)
        where = f"patterns={patterns} bs={buffer_size} B={before} A={after} invert={invert} max={max_match_count} bc={buffer_count}"
        assert rc == exp_rc, f"return code {rc} != oracle {exp_rc}; {where}"
        if got != exp:
            for k, (a, b) in enumerate(zip(got, exp)):
                assert a == b, f"record {k}: got {a} expected {b}; {where}"
            raise AssertionError(f"record count {len(got)} != expected {len(exp)}; {where}")
        assert batches == exp_batches, f"batch sizes differ: {batches[:8]} vs {exp_batches[:8]}; {where}"
        if rc == 0:
            assert stats.matches == sum(1 for i, _, _ in got if i == 0), where
            count_rc, _, _, _, counted = context_scan(lib, path, patterns, collect=None, **kw)
            plain = dict(kw, before=0, after=0)
            _, _, _, _, without = context_scan(lib, path, patterns, collect=None, **plain)
            assert count_rc == 0 and counted.matches == without.matches, where
        return len(got)
    finally:
        if own:
            os.unlink(path)


@pytest.fixture(scope="session")
def context_mock_lib() -> ctypes.CDLL:
    """Host logic of the boundary linked against the CPU engine stand-in with context lines (tests/mock_engine_context)."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_context")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_context.so"))


# ---- the model itself -------------------------------------------------------------------------------------------------------

def test_model_follows_gnu_grep_examples():
    # grep -m1 -A3 a on "a b a c d": a, b, a (context), c
    lines, ctx = context_model(np.array([1, 0, 1, 0, 0], dtype=bool), 0, 3, max_match_count=1)
    assert lines.tolist() == [0, 1, 2, 3] and ctx.tolist() == [False, True, True, True]
    lines, ctx = context_model(np.array([0, 0, 0, 1, 0, 0, 0, 0, 1], dtype=bool), 2, 1)
    assert lines.tolist() == [1, 2, 3, 4, 6, 7, 8] and ctx.tolist() == [True, True, False, True, True, True, False]
    lines, _ = context_model(np.array([0, 1, 0], dtype=bool), 0xFFFFFFFF, 0xFFFFFFFF)
    assert lines.tolist() == [0, 1, 2]


# ---- CPU: host logic on the engine stand-in with context lines ------------------------------------------------------------

@pytest.mark.parametrize("seed", range(40))
def test_random_cases_match_model(seed, context_mock_lib, oracle_lib, tmp_path):
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line: the reference reads stale bytes, excluded from parity")
    rng = random.Random(seed)
    for _ in range(2):
        before, after = rng.choice(WIDTHS), rng.choice(WIDTHS)
        compare_context(context_mock_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match, before, after,
                        invert=rng.random() < 0.3, tmp_dir=str(tmp_path))


_EDGE_SETS = ((["foo"], None, None), (["foo$", "^bar"], None, None), (["o+b", "x{3}"], None, None),
              (["foo", "bar", "o"], [14, 14, 6], [1, 2, 3]))


@pytest.mark.parametrize("name", sorted(EDGE_TEXTS))
@pytest.mark.parametrize("buffer_size", [262140, 64, 8])
def test_edge_texts(name, buffer_size, context_mock_lib, oracle_lib, tmp_path):
    data = EDGE_TEXTS[name]
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    for k, (patterns, flags, ids) in enumerate(_EDGE_SETS):
        for j, (before, after) in enumerate(((0, 0), (1, 0), (0, 2), (2, 7), (100, 1), (0xFFFFFFFF, 0xFFFFFFFF))):
            compare_context(context_mock_lib, oracle_lib, data, patterns, flags, ids, buffer_size=buffer_size, before=before, after=after,
                            invert=(j + k) % 2 == 1, tmp_dir=str(tmp_path))


def test_windows_across_many_segments(context_mock_lib, oracle_lib, monkeypatch, tmp_path):
    """Tiny segments: one window spans several segments in both directions; limits and batches with trailing context."""
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    data = synth.syslog_bytes(192 << 10, seed=5, lib=context_mock_lib)
    for before, after in ((7, 0), (0, 7), (2, 2), (100, 100), (0xFFFFFFFF, 1)):
        compare_context(context_mock_lib, oracle_lib, data, ["Failed password"], before=before, after=after, tmp_dir=str(tmp_path))
    for limit, batch, before, after, invert in ((1, 16, 2, 3, False), (7, 16, 0, 100, False), (100, 7, 3, 1, True), (3, 1, 1, 7, False),
                                               (50, 4096, 0xFFFFFFFF, 2, False), (2, 5, 7, 0xFFFFFFFF, True)):
        compare_context(context_mock_lib, oracle_lib, data, synth.C2_PATTERNS, buffer_count=batch, max_match_count=limit, before=before,
                        after=after, invert=invert, tmp_dir=str(tmp_path))
    # the trailing context after the limit is owed across segments: the scan goes on into the next ones
    text = b"a\n" + b"b\n" * 5 + b"a\n"
    path = tmp_path / "trailing.log"
    path.write_bytes(text)
    rc, got, _, _, st = context_scan(context_mock_lib, str(path), ["a"], max_match_count=1, after=3)
    assert rc == 0 and [(i, ln) for i, ln, _ in got] == [(0, 0), (CONTEXT_ID, 1), (CONTEXT_ID, 2), (CONTEXT_ID, 3)] and st.matches == 1


def test_limit_trailing_context_example(context_mock_lib, oracle_lib, tmp_path):
    """grep -m1 -A3 a on a b a c d: a, b, a, c, the second a a context line."""
    path = tmp_path / "abacd.log"
    path.write_bytes(b"a\nb\na\nc\nd\n")
    rc, got, batches, _, st = context_scan(context_mock_lib, str(path), ["a"], max_match_count=1, after=3)
    assert rc == 0 and got == [(0, 0, b"a\n"), (CONTEXT_ID, 1, b"b\n"), (CONTEXT_ID, 2, b"a\n"), (CONTEXT_ID, 3, b"c\n")]
    assert batches == [1, 1, 1, 1] and st.matches == 1
    compare_context(context_mock_lib, oracle_lib, None, ["a"], max_match_count=1, after=3, path=str(path))


def test_zero_width_equals_the_scan_without_context(context_mock_lib, oracle_lib, tmp_path):
    data = synth.syslog_bytes(256 << 10, seed=21, lib=context_mock_lib)
    path = tmp_path / "zero.log"
    path.write_bytes(data)
    rc, got, batches, _, _ = context_scan(context_mock_lib, str(path), ["ERROR", "port [0-9]+"], ids=[3, 4], buffer_count=9)
    rc0, normal, nbatches = run_scan(context_mock_lib, str(path), ["ERROR", "port [0-9]+"], buffer_count=9)
    assert rc == rc0 == 0 and got == normal and batches == nbatches
    from test_invert_match import invert_scan  # pylint: disable=import-outside-toplevel

    rc, got, batches, _, _ = context_scan(context_mock_lib, str(path), ["ERROR"], buffer_count=9, max_match_count=100, invert=True)
    rc1, inverted, ibatches, _ = invert_scan(context_mock_lib, str(path), ["ERROR"], buffer_count=9, max_match_count=100)
    assert rc == rc1 == 0 and got == inverted and batches == ibatches


def test_rejected_patterns_missing_file_and_nul_lines(context_mock_lib, oracle_lib, tmp_path):
    path = tmp_path / "rejected.log"
    path.write_bytes(b"foo\nbar\n")
    for patterns, flags, ids in ((["(?=x)foo"], None, None), (["foo", ""], None, None), (["foo", "bar"], [14, 6], [1, 1])):
        rc, got, _, _, _ = context_scan(context_mock_lib, str(path), patterns, flags, ids, before=1, after=1)
        assert rc == 4 and got == []
        compare_context(context_mock_lib, oracle_lib, None, patterns, flags, ids, before=1, after=1, path=str(path))
    rc, got, _, _, _ = context_scan(context_mock_lib, str(tmp_path / "missing.log"), ["foo"], after=2)
    assert rc == 6 and got == []
    # a NUL-only pseudo-line used as context is delivered as ""
    path.write_bytes(b"abc\0\0\0\0\0\0\nfoo\n\0\0")
    rc, got, _, _, _ = context_scan(context_mock_lib, str(path), ["foo"], buffer_size=4, before=2, after=2)
    assert rc == 0 and got == [(CONTEXT_ID, 2, b""), (CONTEXT_ID, 3, b"\n"), (0, 4, b"foo"), (CONTEXT_ID, 5, b"\n"), (CONTEXT_ID, 6, b"")]


def test_engine_without_context_lines_refuses_them(tmp_path):
    """Host logic linked against an engine build without slot_set_context (the inverted-scan stand-in) fails context scans
    with 7; a rejected pattern set still gives 4."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_invert")], stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_invert.so"))
    path = tmp_path / "plain.log"
    path.write_bytes(b"foo\nbar\n")
    for before, after in ((0, 0), (1, 1)):
        rc, got, _, _, _ = context_scan(lib, str(path), ["foo"], before=before, after=after)
        assert rc == 7 and got == []
    assert context_scan(lib, str(path), ["(?=x)foo"], after=1)[0] == 4


def test_compressed_inputs(context_mock_lib, oracle_lib, monkeypatch, tmp_path):
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    text = synth.syslog_bytes(256 << 10, seed=9, lib=context_mock_lib)
    half = text.rfind(b"\n", 0, len(text) // 2) + 1
    gz = tmp_path / "multi.log.gz"
    gz.write_bytes(parity.gz_members([text[:half], text[half:]]))
    assert compare_context(context_mock_lib, oracle_lib, None, ["Failed password"], before=3, after=2, path=str(gz)) > 40
    compare_context(context_mock_lib, oracle_lib, None, synth.C2_PATTERNS, max_match_count=30, buffer_count=7, after=5, invert=True, path=str(gz))
    for name, blob in parity.zstd_cases(text).items():
        path = tmp_path / f"{name}.log.zst"
        path.write_bytes(blob)
        compare_context(context_mock_lib, oracle_lib, None, ["ERROR", "port [0-9]+"], before=2, after=1, path=str(path))


@pytest.mark.parametrize("devices", ["all", "0,1,2"])
def test_sharded_scan_windows_across_shards(devices, context_mock_lib, oracle_lib, monkeypatch, tmp_path):
    """$GPUGREP_DEVICES over three mock devices: windows that reach across shard bounds, limits with trailing context into
    the next shard, and the same records as one device."""
    monkeypatch.setenv("GPUGREP_MOCK_DEVICES", "3")
    monkeypatch.setenv("GPUGREP_DEVICES", devices)
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
    data = synth.syslog_bytes(1 << 20, seed=77)
    bounds = [parity_bound(data, g, 3) for g in range(4)]
    # a selected line just before and just after each shard bound
    lines = data.split(b"\n")
    starts = np.cumsum([0] + [len(x) + 1 for x in lines])
    marked = set()
    for b in bounds[1:3]:
        k = int(np.searchsorted(starts, b))
        marked.update({k - 2, k + 1})
    data = b"\n".join(b"MARK " + x if i in marked else x for i, x in enumerate(lines))
    for before, after, invert in ((3, 3, False), (100, 0, False), (0, 100, False), (0xFFFFFFFF, 0xFFFFFFFF, False), (2, 2, True)):
        compare_context(context_mock_lib, oracle_lib, data, ["MARK"], before=before, after=after, invert=invert, tmp_dir=str(tmp_path))
    compare_context(context_mock_lib, oracle_lib, data, ["MARK"], max_match_count=1, after=5, tmp_dir=str(tmp_path))
    compare_context(context_mock_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=1000, buffer_count=7, before=2, after=3,
                    tmp_dir=str(tmp_path))
    buf = ctypes.create_string_buffer(data, len(data))
    rc, sharded, _, crc, stats = context_scan_buffer(context_mock_lib, ctypes.addressof(buf), len(data), 0, ["MARK"], before=3, after=3)
    assert rc == 0 and stats.segments >= 3
    monkeypatch.delenv("GPUGREP_DEVICES")
    rc, single, _, crc1, stats1 = context_scan_buffer(context_mock_lib, ctypes.addressof(buf), len(data), 0, ["MARK"], before=3, after=3)
    assert rc == 0 and single == sharded and crc1 == crc and stats1.matches == stats.matches == len(marked)


def parity_bound(data: bytes, rank: int, world: int) -> int:
    """gpugrep_shard_begin for a host buffer: rank * size / world advanced past the next newline."""
    if rank == 0:
        return 0
    if rank >= world:
        return len(data)
    pos = len(data) * rank // world
    if data[pos - 1:pos] == b"\n":
        return pos
    nl = data.find(b"\n", pos)
    return nl + 1 if nl >= 0 else len(data)


def test_scan_and_grep_keywords(context_mock_lib, oracle_lib, monkeypatch, tmp_path):
    from hypergrep_b200 import CONTEXT_ID as exported  # pylint: disable=import-outside-toplevel
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel

    assert exported == CONTEXT_ID
    text = b"".join(b"line %d %s\n" % (k, b"foobar" if k % 13 == 0 else b"nothing") for k in range(3000)) + b"tail foobar"
    path = tmp_path / "grep.log"
    path.write_bytes(text)
    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: context_mock_lib)
    got = []

    def on_batch(matches, count):
        got.extend((matches[k].id, matches[k].line_number, matches[k].line) for k in range(count))

    assert utils.scan(str(path), ["foobar", "^line 7 "], on_batch, ids=[4, 5], before_context=2, after_context=1) == 0
    rc, expected, _ = oracle_context(oracle_lib, str(path), ["foobar", "^line 7 "], ids=[4, 5], before=2, after=1)
    assert rc == 0 and got == expected
    lines, rc = utils.grep(str(path), ["foobar", "^line 7 "], before_context=2, after_context=1)
    assert rc == 0 and lines == [(ln + 1, line.decode(), i == CONTEXT_ID) for i, ln, line in expected]
    lines, rc = utils.grep(str(path), ["foobar"], after_context=3, max_match_count=2, invert_match=True)
    _, expected, _ = oracle_context(oracle_lib, str(path), ["foobar"], after=3, max_match_count=2, invert=True)
    assert rc == 0 and lines == [(ln + 1, line.decode(), i == CONTEXT_ID) for i, ln, line in expected]
    # count_only and only_matching ignore context; zero widths keep the old shape
    assert utils.grep(str(path), ["foobar"], count_only=True, before_context=5) == utils.grep(str(path), ["foobar"], count_only=True)
    assert utils.grep(str(path), ["foo"], only_matching=True, after_context=5) == utils.grep(str(path), ["foo"], only_matching=True)
    assert utils.grep(str(path), ["foobar"], before_context=0, after_context=0) == utils.grep(str(path), ["foobar"])
    with pytest.raises(ValueError):
        utils.grep(str(path), ["foobar"], before_context=-1)
    with pytest.raises(ValueError):
        utils.scan(str(path), ["foobar"], on_batch, after_context=-2)
    # positional calls keep their meaning: the new keywords come last
    assert utils.grep(str(path), ["foobar"], False, True) == (232, 0)

    class CallbackOnly:   # a plain libhyperscanner.so: no context entry point, and no CPU fallback for it
        hyperscan = context_mock_lib.hyperscan
        check_patterns = context_mock_lib.check_patterns

        def __getattr__(self, name):
            raise AttributeError(name)

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", CallbackOnly)
    with pytest.raises(NotImplementedError, match="gpugrep_context_scan_file"):
        utils.grep(str(path), ["foobar"], after_context=1)


def _cli(argv, monkeypatch, capsys):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel

    monkeypatch.setattr("sys.argv", ["hyperscanner"] + argv)
    with pytest.raises(SystemExit) as leave:
        multiscanner.main()
    return leave.value.code, capsys.readouterr().out


def render(records: list, name: str | None, numbers: bool, separator: str | None = "--", printed: bool = False) -> tuple[str, bool]:
    """GNU grep's output of context records [(id, line_number, text)] of one file."""
    out, previous = [], None
    for i, ln, text in records:
        mark = "-" if i == CONTEXT_ID else ":"
        if separator is not None and (ln != previous + 1 if previous is not None else printed):
            out.append(separator + "\n")
        previous, printed = ln, True
        out.append((f"{name}{mark}" if name else "") + (f"{ln + 1}{mark}" if numbers else "") + text.decode())
    return "".join(out), printed


def test_cli_context_options(context_mock_lib, oracle_lib, monkeypatch, capsys, tmp_path):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: context_mock_lib)
    a, b = tmp_path / "a.log", tmp_path / "b.log"
    a.write_bytes(b"".join(b"row %d%s\n" % (k, b" foo" if k in (3, 4, 12, 30) else b"") for k in range(40)))
    b.write_bytes(b"foo first\nbar\nbaz\nqux\nfoo again\n")
    a, b = str(a), str(b)

    def expect(path, before, after, invert=False, limit=0, name=None, numbers=False, separator="--", printed=False):
        rc, records, _ = oracle_context(oracle_lib, path, ["foo"], before=before, after=after, invert=invert, max_match_count=limit)
        assert rc == 0
        return render(records, name, numbers, separator, printed)

    text, _ = expect(a, 1, 2)
    assert _cli(["-B", "1", "-A", "2", "foo", a], monkeypatch, capsys) == (0, text)
    assert _cli(["-C", "5", "-B", "1", "--after-context", "2", "foo", a], monkeypatch, capsys) == (0, text)
    text, _ = expect(a, 3, 3, numbers=True)
    assert _cli(["-n", "-C", "3", "foo", a], monkeypatch, capsys) == (0, text)
    text, _ = expect(a, 0, 1, separator="::")
    assert _cli(["--group-separator", "::", "-A", "1", "foo", a], monkeypatch, capsys) == (0, text)
    text, _ = expect(a, 0, 1, separator=None)
    assert _cli(["--no-group-separator", "-A", "1", "foo", a], monkeypatch, capsys) == (0, text)
    # several files: prefixes name:/name-, and a separator between files too, in either print order
    first, printed = expect(a, 1, 1, name=a, numbers=True)
    second, _ = expect(b, 1, 1, name=b, numbers=True, printed=printed)
    assert _cli(["-n", "-C", "1", "foo", a, b], monkeypatch, capsys) == (0, first + second)
    code, out = _cli(["-n", "-C", "1", "--no-order", "foo", a, b], monkeypatch, capsys)
    assert code == 0 and sorted(out.split("\n")) == sorted((first + second).split("\n"))
    text, _ = expect(a, 0, 3, limit=1, numbers=True)
    assert _cli(["-m", "1", "-n", "-A", "3", "foo", a], monkeypatch, capsys) == (0, text)
    text, _ = expect(a, 2, 1, invert=True)
    assert _cli(["-v", "-B", "2", "-A", "1", "foo", a], monkeypatch, capsys) == (0, text)
    # -o: matched parts only; a separator between selected lines whose gap exceeds A+B lines
    assert _cli(["-o", "-A", "1", "foo", a], monkeypatch, capsys) == (0, "foo\nfoo\n--\nfoo\n--\nfoo\n")
    assert _cli(["-o", "-C", "4", "foo", a], monkeypatch, capsys) == (0, "foo\nfoo\nfoo\n--\nfoo\n")
    # -c, -t, -l, -L, -q ignore context
    assert _cli(["-c", "-C", "2", "foo", a, b], monkeypatch, capsys) == (0, f"{a}:4\n{b}:2\n")
    assert _cli(["-t", "-A", "2", "foo", a, b], monkeypatch, capsys) == (0, "6\n")
    assert _cli(["-l", "-B", "2", "foo", a, b], monkeypatch, capsys) == (0, f"{a}\n{b}\n")
    assert _cli(["-L", "-B", "2", "foo", a, b], monkeypatch, capsys) == (0, "")
    assert _cli(["-q", "-C", "2", "foo", a], monkeypatch, capsys) == (0, "")
    for bad in (["-A", "-1"], ["-B", "-3"], ["-C", "-2"]):
        code, out = _cli(bad + ["foo", a], monkeypatch, capsys)
        assert code == 2 and "invalid context length" in out


_SYSTEM_GREP = shutil.which("grep")


@pytest.mark.skipif(_SYSTEM_GREP is None, reason="no system grep")
@pytest.mark.parametrize("seed", range(8))
def test_cli_against_system_grep(seed, context_mock_lib, monkeypatch, capsys, tmp_path):
    """ASCII literal patterns: the CLI prints what the system grep prints, for random widths, limits and separators."""
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: context_mock_lib)
    rng = random.Random(seed)
    words = ["alpha", "beta", "gamma", "delta", "", "eps"]
    paths = []
    for k in range(2):
        path = tmp_path / f"f{k}.log"
        path.write_text("".join(" ".join(rng.choice(words) for _ in range(rng.randint(0, 3))) + "\n" for _ in range(rng.randint(0, 60))))
        paths.append(str(path))
    for _ in range(6):
        opts = [rng.choice(["-A", "-B", "-C"]), str(rng.choice([0, 1, 2, 5]))]
        if rng.random() < 0.5:
            opts += [rng.choice(["-A", "-B"]), str(rng.choice([0, 1, 3]))]
        opts += rng.sample(["-n", "-v", "-H", "--no-group-separator", "-o"], rng.randint(0, 2))
        if rng.random() < 0.3:
            opts += ["-m", str(rng.randint(1, 4))]
        if "-o" in opts and "-v" in opts:
            continue
        argv = opts + ["-e", rng.choice(["alpha", "eps", "gamma"])] + paths
        want = subprocess.run([_SYSTEM_GREP] + argv, capture_output=True, text=True, check=False, env={"LC_ALL": "C"})
        code, out = _cli(argv, monkeypatch, capsys)
        assert (code, out) == (want.returncode, want.stdout), argv


# ---- GPU: the CUDA engine ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_zero_width_equals_the_scans_without_context(force_general, gpu_lib, monkeypatch, tmp_path):
    """A = B = 0: the records of gpugrep_scan_* (ids 0) and gpugrep_invert_scan_*, record for record, on C1, C2, C3 and an
    NFA-fallback set, from a file and from device memory."""
    import torch  # pylint: disable=import-outside-toplevel
    from test_invert_match import invert_scan, invert_scan_buffer  # pylint: disable=import-outside-toplevel

    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    c3, plants = synth.c3_patterns()
    sets = ((synth.C1_PATTERNS, None), (synth.C2_PATTERNS, None), (c3, plants), ([r"e.{60}d\b", r"ERROR", r"\bport .{40,80}x"], None))
    for k, (patterns, plant) in enumerate(sets):
        data = synth.syslog_bytes(4 << 20, seed=40 + k, plants=plant, plant_ppm=20000 if plant else 0, lib=gpu_lib)
        path = tmp_path / f"z{k}.log"
        path.write_bytes(data)
        rc, got, batches, _, _ = context_scan(gpu_lib, str(path), patterns, buffer_count=4096)
        rc0, normal, nbatches = run_scan(gpu_lib, str(path), patterns, ids=[0] * len(patterns), buffer_count=4096)
        assert rc == rc0 == 0 and got == normal and batches == nbatches and len(got) > 100
        rc, got, batches, _, _ = context_scan(gpu_lib, str(path), patterns, buffer_count=4096, invert=True)
        rc1, inverted, ibatches, _ = invert_scan(gpu_lib, str(path), patterns, buffer_count=4096)
        assert rc == rc1 == 0 and got == inverted and batches == ibatches
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        for invert in (False, True):
            rc, nums, _, crc, _ = context_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, invert=invert)
            if invert:
                rc2, want, wcrc, _ = invert_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, buffer_count=4096, collect="numbers")
            else:
                rc2, recs, _ = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, buffer_count=4096)
                want, wcrc = [ln for _, ln, _ in recs], zlib.crc32(b"".join(line for _, _, line in recs))
            assert rc == rc2 == 0 and [ln for _, ln in nums] == want and crc == wcrc


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
@pytest.mark.parametrize("seed", range(40))
def test_gpu_random_cases_match_model(seed, force_general, gpu_lib, oracle_lib, monkeypatch, tmp_path):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    rng = random.Random(1000 + seed)
    before, after = rng.choice(WIDTHS), rng.choice(WIDTHS)
    compare_context(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match, before, after,
                    invert=rng.random() < 0.3, tmp_dir=str(tmp_path))


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_edges_limits_and_segments(force_general, gpu_lib, oracle_lib, monkeypatch, tmp_path):
    """EDGE_TEXTS (buffer_size 64 takes the general path), then windows over many tiny segments, limits and factorless sets."""
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    for _name, data in sorted(EDGE_TEXTS.items()):
        for buffer_size in (262140, 64):
            if parity.has_all_nul_pseudo_line(data, buffer_size):
                continue
            for j, (before, after) in enumerate(((1, 2), (0xFFFFFFFF, 0), (0, 7))):
                compare_context(gpu_lib, oracle_lib, data, ["foo", "bar"], buffer_size=buffer_size, before=before, after=after, invert=j == 1,
                                tmp_dir=str(tmp_path))
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    data = synth.syslog_bytes(1 << 20, seed=5, lib=gpu_lib)
    for before, after, invert in ((2, 2, False), (100, 0, False), (0, 100, True), (0xFFFFFFFF, 3, False)):
        compare_context(gpu_lib, oracle_lib, data, ["Failed password"], before=before, after=after, invert=invert, tmp_dir=str(tmp_path))
    compare_context(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=500, buffer_count=7, before=2, after=5, tmp_dir=str(tmp_path))
    compare_context(gpu_lib, oracle_lib, data[: 256 << 10], ["e.{3}d", "[0-9]{4}:"], buffer_size=64, before=1, after=2, tmp_dir=str(tmp_path))


def _expected_numbers(data: bytes, normal_lines, nlines: int, before: int, after: int, invert: bool = False):
    """(id, line_number) records and the CRC of their texts for default-buffer text without NULs, from the normal scan."""
    selected = np.zeros(nlines, dtype=bool)
    selected[np.asarray(normal_lines, dtype=np.int64)] = True
    if invert:
        selected = ~selected
    lines, ctx = context_model(selected, before, after)
    split = data.split(b"\n")
    pieces = [line + b"\n" for line in split[:-1]] + ([split[-1]] if split[-1] else [])
    if any(len(piece) > 262139 for piece in pieces):   # gzgets cuts such lines into several pseudo-lines
        from test_invert_match import pseudo_lines  # pylint: disable=import-outside-toplevel

        pieces = pseudo_lines(data, 262140)
    assert len(pieces) == nlines
    texts = b"".join(pieces[ln] for ln in lines.tolist())
    return [(CONTEXT_ID if c else 0, ln) for ln, c in zip(lines.tolist(), ctx.tolist())], zlib.crc32(texts)


@pytest.mark.gpu
def test_gpu_multi_segment_text_from_file_host_pinned_and_device(gpu_lib, monkeypatch, tmp_path):
    """72 MiB of C2 text: file (32 MiB segments), pageable and pinned host memory (64 MiB segments), device memory (one
    segment, then 8 MiB segments): line numbers and a CRC of the texts equal the model over the normal scan."""
    import torch  # pylint: disable=import-outside-toplevel

    data = synth.syslog_bytes(72 << 20, seed=61, lib=gpu_lib)
    path = tmp_path / "c2.log"
    path.write_bytes(data)
    rc, normal, _ = run_scan(gpu_lib, str(path), synth.C2_PATTERNS, buffer_count=4096)
    assert rc == 0 and len(normal) > 10000
    host = np.frombuffer(data, dtype=np.uint8)
    pinned = torch.from_numpy(host.copy()).pin_memory()
    dev = pinned.cuda()
    torch.cuda.synchronize()
    for before, after, invert in ((2, 2, False), (0, 7, True), (100, 1, False)):
        rc, got, _, crc, st = context_scan(gpu_lib, str(path), synth.C2_PATTERNS, buffer_count=4096, before=before, after=after, invert=invert,
                                           collect="numbers")
        assert rc == 0 and st.segments >= 3 and st.path == 1
        want, wcrc = _expected_numbers(data, [ln for _, ln, _ in normal], st.lines, before, after, invert)
        assert got == want and crc == wcrc
        for ptr, location in ((host.ctypes.data, 0), (pinned.data_ptr(), 0), (dev.data_ptr(), 1)):
            rc, nums, _, bcrc, _ = context_scan_buffer(gpu_lib, ptr, len(data), location, synth.C2_PATTERNS, before=before, after=after,
                                                       invert=invert)
            assert rc == 0 and nums == want and bcrc == wcrc
    monkeypatch.setenv("GPUGREP_DEVICE_SEGMENT_MB", "8")
    rc, nums, _, bcrc, st = context_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, synth.C2_PATTERNS, before=3, after=3)
    want, wcrc = _expected_numbers(data, [ln for _, ln, _ in normal], st.lines, 3, 3)
    assert rc == 0 and st.segments >= 9 and nums == want and bcrc == wcrc


@pytest.mark.gpu
def test_gpu_long_line_in_a_large_device_segment(gpu_lib):
    """A 300 KiB line in a 192 MiB device segment, and selected lines next to the 64 MiB piece bounds: the segment is scanned
    again in pieces (one on the general path), and windows reach across the piece bounds."""
    import torch  # pylint: disable=import-outside-toplevel

    size = 192 << 20
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=77, lib=gpu_lib)
    view = host.numpy()
    start = 100 << 20
    while view[start - 1] != 10:
        start += 1
    view[start:start + (300 << 10)] = ord("x")
    for bound in (64 << 20, 128 << 20):
        for offset in (-300, 200):
            at = bound + offset
            while view[at - 1] != 10:
                at += 1
            view[at:at + 6] = np.frombuffer(b"ZZMARK", dtype=np.uint8)
    dev = host.cuda()
    torch.cuda.synchronize()
    data = bytes(view)
    patterns = ["ZZMARK", "Failed password"]
    rc, normal, _ = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, patterns, buffer_count=4096)
    assert rc == 0
    for before, after in ((5, 5), (0, 40)):
        rc, nums, _, crc, st = context_scan_buffer(gpu_lib, dev.data_ptr(), size, 1, patterns, before=before, after=after)
        assert rc == 0 and st.split_segments == 1 and st.path == 3, (st.split_segments, st.path)
        want, wcrc = _expected_numbers(data, [ln for _, ln, _ in normal], st.lines, before, after)
        assert nums == want and crc == wcrc
        rc, hnums, _, hcrc, hst = context_scan_buffer(gpu_lib, host.data_ptr(), size, 0, patterns, before=before, after=after)
        assert rc == 0 and hnums == nums and hcrc == crc and hst.split_segments == 0


@pytest.mark.gpu
def test_gpu_short_lines_output_every_line(gpu_lib, oracle_lib, tmp_path):
    """Lines under 16 bytes with -C100: nearly every line is output (with -v -C100 every line), far more records than the fast
    path's n/48 record buffer; at 1 GiB (about 200 million lines, delivered through gpugrep_discard_results) -v -C100 still
    brings every line back as a record."""
    import torch  # pylint: disable=import-outside-toplevel
    from test_invert_match import _short_lines  # pylint: disable=import-outside-toplevel

    patterns = ["ERROR", "port [0-9]+"]
    data = _short_lines(32 << 20, seed=5)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    rc, normal, _ = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, buffer_count=4096)
    assert rc == 0
    for invert in (False, True):
        rc, nums, _, crc, st = context_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, before=100, after=100, invert=invert)
        want, wcrc = _expected_numbers(data, [ln for _, ln, _ in normal], st.lines, 100, 100, invert)
        assert rc == 0 and st.path == 1 and nums == want and crc == wcrc
        assert len(nums) > 4 * len(data) // 48 and (len(nums) == st.lines or not invert)
    assert compare_context(gpu_lib, oracle_lib, data[: 1 << 20], patterns, before=2, after=2, tmp_dir=str(tmp_path)) > 10000
    del dev
    big = _short_lines(1 << 30, seed=6)
    dev = torch.frombuffer(bytearray(big), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    del big
    pa, fa, ia, n = marshal(patterns, None, None)
    discard = ctypes.cast(gpu_lib.gpugrep_discard_results, ctypes.c_void_p)
    entry = gpu_lib.gpugrep_context_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    counted, st = Stats(), Stats()
    rc0 = entry(dev.data_ptr(), dev.numel(), 1, pa, fa, ia, n, None, 262140, 4096, 0, 0, 0, 1, None, ctypes.byref(counted))
    rc = entry(dev.data_ptr(), dev.numel(), 1, pa, fa, ia, n, discard, 262140, 4096, 0, 100, 100, 1, None, ctypes.byref(st))
    assert rc0 == rc == 0 and st.path == 1 and st.matches == counted.matches and st.lines == counted.lines > 150_000_000
    assert st.d2h_bytes >= 12 * st.lines   # every line came back as a record


@pytest.mark.gpu
def test_gpu_count_only_context_scans_launch_what_the_count_launches(gpu_lib):
    import torch  # pylint: disable=import-outside-toplevel

    data = synth.syslog_bytes(32 << 20, seed=81, lib=gpu_lib)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    for patterns in (synth.C2_PATTERNS, synth.C1_PATTERNS):
        for invert in (False, True):
            rc, _, _, _, plain = context_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, invert=invert, collect=None)
            rc2, _, _, _, ctx = context_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, before=3, after=3, invert=invert,
                                                    collect=None)
            _, _, normal = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, collect=False)
            assert rc == rc2 == 0 and plain.path == ctx.path == 1
            assert ctx.launches == plain.launches == normal.launches and ctx.matches == plain.matches and ctx.lines == plain.lines


@pytest.mark.gpu
def test_gpu_cli_context_in_a_fresh_process(gpu_lib, oracle_lib, tmp_path):
    path = tmp_path / "cli.log"
    path.write_bytes(synth.syslog_bytes(512 << 10, seed=301, lib=gpu_lib))
    rc, expected, _ = oracle_context(oracle_lib, str(path), ["Failed password"], before=2, after=1)
    assert rc == 0 and expected
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "hypergrep_b200.multiscanner"]
    proc = subprocess.run(cmd + ["-n", "-B", "2", "-A", "1", "Failed password", str(path)], env=env, capture_output=True, text=True,
                          timeout=300, check=False)
    assert proc.returncode == 0, proc.stderr
    assert proc.stdout == render(expected, None, True)[0]


@pytest.mark.gpu
def test_gpu_context_scan_over_two_gpus(gpu_lib, oracle_lib, monkeypatch, tmp_path):
    import torch  # pylint: disable=import-outside-toplevel

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", str(1 << 20))
    data = synth.syslog_bytes(16 << 20, seed=31)
    assert compare_context(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, before=2, after=3, tmp_dir=str(tmp_path)) > 10000
    compare_context(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=5000, buffer_count=7, after=100, tmp_dir=str(tmp_path))
