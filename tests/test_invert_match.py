"""Inverted matching (grep -v): gpugrep_invert_scan_file / gpugrep_invert_scan_buffer, scan()/grep(invert_match=True) and
the CLI's -v.  An inverted scan selects the pseudo-lines in which no pattern reports: its line numbers must equal
{0 .. lines-1} minus the line numbers of the normal scan, and its records, batches and return codes must equal what the
oracle gives for the same question (`oracle_invert`).  CPU tests run the host logic on the CPU engine stand-in with inverted
scans (tests/mock_engine_invert); `gpu` tests run the CUDA engine (fast and general path)."""

from __future__ import annotations

import ctypes
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import parity
from gpu_api import Stats, marshal, scan_buffer
from hypergrep_b200 import synth
from oracle_api import CALLBACK, run_scan
from test_host_logic import EDGE_TEXTS

_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
              ctypes.c_ulonglong, ctypes.c_void_p]
_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]


class _Collector:
    """Callback that keeps (id, line_number, line) records, or only line numbers and a CRC of the texts (large scans)."""

    def __init__(self, mode: str | None):
        self.mode, self.records, self.batches, self.crc = mode, [], [], 0

        def cb(results, count):
            self.batches.append(count)
            for i in range(count):
                r = results[i]
                if self.mode == "numbers":
                    self.records.append(r.line_number)
                    self.crc = zlib.crc32(r.line, self.crc)
                else:
                    self.records.append((r.id, r.line_number, r.line))

        self.c_callback = CALLBACK(cb) if mode else None

    def pointer(self):
        return ctypes.cast(self.c_callback, ctypes.c_void_p) if self.c_callback else None


def invert_scan(lib, path: str, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0, collect="records"):
    """gpugrep_invert_scan_file -> (rc, records or None, batch sizes, stats)."""
    pa, fa, ia, n = marshal(patterns, flags, ids)
    entry = lib.gpugrep_invert_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(path.encode(), pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, ctypes.byref(stats))
    return rc, (sink.records if collect else None), sink.batches, stats


def invert_scan_buffer(lib, ptr: int, size: int, location: int, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16,
                       max_match_count=0, collect="records"):
    """gpugrep_invert_scan_buffer -> (rc, records or None, crc of the texts, stats)."""
    pa, fa, ia, n = marshal(patterns, flags, ids)
    entry = lib.gpugrep_invert_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(ptr, size, location, pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, None, ctypes.byref(stats))
    return rc, (sink.records if collect else None), sink.crc, stats


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def invert_mock_lib() -> ctypes.CDLL:
    """Host logic of the boundary linked against the CPU engine stand-in with inverted scans (tests/mock_engine_invert)."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_invert")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_invert.so"))


def oracle_invert(oracle, path: str, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0):
    """What the reference loop (hyperscanner.c:179-231) delivers when a pseudo-line is reported iff no pattern reports in it,
    taken from the oracle: its normal scan says which pseudo-lines match, and a scan for `.` (DOTALL) reads every pseudo-line
    with its stripped text (a pseudo-line of NULs only is missing there: such inputs are excluded).  The stop rule counts
    selected lines, the batches are full batches of buffer_count (clamped to max_match_count), then the remainder.
    Returns (rc, [(0, line_number, line)], [batch sizes]) like oracle_api.run_scan."""
    rc, matched, _ = run_scan(oracle, path, patterns, flags=flags, ids=ids, buffer_size=buffer_size, buffer_count=4096)
    if rc != 0:
        return rc, [], []
    rc, every, _ = run_scan(oracle, path, ["."], flags=[10], ids=[0], buffer_size=buffer_size, buffer_count=4096)
    assert rc == 0
    hit = {ln for _, ln, _ in matched}
    selected = [(0, ln, text) for _, ln, text in every if ln not in hit]
    batch = buffer_count
    if 0 < max_match_count < batch:
        batch = max_match_count
    batch = max(1, batch)
    if max_match_count > 0:
        selected = selected[:max_match_count]
    batches = [batch] * (len(selected) // batch) + ([len(selected) % batch] if len(selected) % batch else [])
    return rc, selected, batches


def pseudo_lines(data: bytes, buffer_size: int) -> list[bytes]:
    """gzgets(buffer_size) splitting, as the reference reads the file."""
    out, pos, lim = [], 0, buffer_size - 1
    while pos < len(data):
        nl = data.find(b"\n", pos, pos + lim)
        end = nl + 1 if nl >= 0 else min(len(data), pos + lim)
        out.append(data[pos:end])
        pos = end
    return out


def stripped(chunk: bytes) -> bytes:
    """What a record delivers for a pseudo-line: leading NULs skipped, cut at the next NUL."""
    return chunk.lstrip(b"\0").split(b"\0", 1)[0]


def compare_invert(lib, oracle, data: bytes | None, patterns, flags=None, ids=None, buffer_size=262140, buffer_count=16, max_match_count=0,
                   path: str | None = None, tmp_dir: str | None = None) -> int:
    """`lib`'s inverted scan == oracle_invert (records, order, batches, return code); without a limit its line numbers are
    also the complement of the oracle's normal scan over all `stats.lines` pseudo-lines, its texts follow the strip rule on
    the pseudo-lines split here, and count-only == the number of records."""
    own = path is None
    if own:
        path = os.path.join(tmp_dir or "/tmp", f"invert_{os.getpid()}_{random.getrandbits(48):x}.log")
        with open(path, "wb") as handle:
            handle.write(data)
    try:
        kw = {"flags": flags, "ids": ids, "buffer_size": buffer_size, "buffer_count": buffer_count, "max_match_count": max_match_count}
        exp_rc, exp, exp_batches = oracle_invert(oracle, path, patterns, **kw)
        rc, got, batches, stats = invert_scan(lib, path, patterns, **kw)
        assert rc == exp_rc, f"return code {rc} != oracle {exp_rc} for {patterns}"
        if got != exp:
            for k, (a, b) in enumerate(zip(got, exp)):
                assert a == b, f"record {k}: got {a} expected {b}; patterns={patterns} flags={flags} ids={ids} bs={buffer_size}"
            raise AssertionError(f"record count {len(got)} != oracle {len(exp)}; patterns={patterns} bs={buffer_size}")
        assert batches == exp_batches, f"batch sizes differ: {batches[:8]} vs {exp_batches[:8]}"
        if rc == 0:
            assert all(i == 0 for i, _, _ in got)
            assert stats.matches == len(got)
        if rc == 0 and max_match_count == 0:
            normal_rc, normal, _ = run_scan(oracle, path, patterns, flags=flags, ids=ids, buffer_size=buffer_size)
            assert normal_rc == 0
            matched = {ln for _, ln, _ in normal}
            assert [ln for _, ln, _ in got] == [k for k in range(stats.lines) if k not in matched]
            if data is not None:
                lines = pseudo_lines(data, buffer_size)
                assert stats.lines == len(lines)
                assert [text for _, _, text in got] == [stripped(lines[ln]) for _, ln, _ in got]
            count_rc, _, _, counted = invert_scan(lib, path, patterns, collect=None, **kw)
            assert count_rc == 0 and counted.matches == len(got) and counted.lines == stats.lines
        return len(got)
    finally:
        if own:
            os.unlink(path)


# ---- CPU: host logic on the engine stand-in with inverted scans -------------------------------------------------------------

@pytest.mark.parametrize("seed", range(120))
def test_random_cases_match_oracle(seed, invert_mock_lib, oracle_lib, tmp_path):
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line: the reference reads stale bytes, excluded from parity")
    compare_invert(invert_mock_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match, tmp_dir=str(tmp_path))


_EDGE_SETS = ((["foo"], None, None), (["foo$", "^bar"], None, None), (["o+b", "x{3}"], None, None), (["foo."], None, None),
              (["foo", "bar", "o"], [14, 14, 6], [1, 2, 3]))


@pytest.mark.parametrize("name", sorted(EDGE_TEXTS))
@pytest.mark.parametrize("buffer_size", [262140, 64, 8])
def test_edge_texts(name, buffer_size, invert_mock_lib, oracle_lib, tmp_path):
    data = EDGE_TEXTS[name]
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    for patterns, flags, ids in _EDGE_SETS:
        compare_invert(invert_mock_lib, oracle_lib, data, patterns, flags, ids, buffer_size=buffer_size, tmp_dir=str(tmp_path))


def test_limits_batches_and_segments(invert_mock_lib, oracle_lib, monkeypatch, tmp_path):
    """max_match_count counts selected lines; buffer_count (clamped to the limit) batches them; segment cuts change nothing."""
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    data = synth.syslog_bytes(1 << 20, seed=5, lib=invert_mock_lib)
    assert compare_invert(invert_mock_lib, oracle_lib, data, synth.C2_PATTERNS, tmp_dir=str(tmp_path)) > 1000
    for limit, batch in ((1, 16), (7, 16), (1000, 7), (4097, 4096), (3, 1)):
        compare_invert(invert_mock_lib, oracle_lib, data, synth.C2_PATTERNS, buffer_count=batch, max_match_count=limit, tmp_dir=str(tmp_path))
    # several ids and a non-SINGLEMATCH pattern select the same lines
    compare_invert(invert_mock_lib, oracle_lib, data[: 256 << 10], ["ERROR", "port [0-9]+", "WARN"], flags=[14, 6, 14], ids=[3, 1, 2],
                   max_match_count=500, buffer_count=9, tmp_dir=str(tmp_path))
    compare_invert(invert_mock_lib, oracle_lib, data[: 256 << 10], ["ERROR", "ssh2$"], buffer_size=50, tmp_dir=str(tmp_path))


def test_rejected_patterns_and_missing_file(invert_mock_lib, oracle_lib, tmp_path):
    data = b"foo\nbar\n"
    for patterns, flags, ids in ((["(?=x)foo"], None, None), (["foo", ""], None, None), (["a*"], None, None),
                                 (["foo", "bar"], [14, 6], [1, 1]), (["foo"], [14 | 64], None)):
        path = tmp_path / "rejected.log"
        path.write_bytes(data)
        rc, got, _, _ = invert_scan(invert_mock_lib, str(path), patterns, flags, ids)
        assert rc == 4 and got == []
        compare_invert(invert_mock_lib, oracle_lib, None, patterns, flags, ids, path=str(path))
    rc, got, _, _ = invert_scan(invert_mock_lib, str(tmp_path / "missing.log"), ["foo"])
    assert rc == 6 and got == []
    compare_invert(invert_mock_lib, oracle_lib, None, ["foo"], path=str(tmp_path / "missing.log"))


def test_engine_without_inverted_scans_refuses_them(hostmock_lib, tmp_path):
    """The host logic linked against an engine build that has no inverted scan (the plain CPU stand-in) fails such scans with
    7 instead of answering them some other way; a rejected pattern set still gives 4, and normal scans are unaffected."""
    path = tmp_path / "plain.log"
    path.write_bytes(b"foo\nbar\n")
    rc, got, _, _ = invert_scan(hostmock_lib, str(path), ["foo"])
    assert rc == 7 and got == []
    assert invert_scan(hostmock_lib, str(path), ["(?=x)foo"])[0] == 4
    rc, got, _ = run_scan(hostmock_lib, str(path), ["foo"])
    assert rc == 0 and got == [(0, 0, b"foo\n")]


def test_compressed_inputs(invert_mock_lib, oracle_lib, tmp_path):
    text = synth.syslog_bytes(512 << 10, seed=9, lib=invert_mock_lib)
    half = text.rfind(b"\n", 0, len(text) // 2) + 1
    gz = tmp_path / "multi.log.gz"
    gz.write_bytes(parity.gz_members([text[:half], text[half:]]))
    assert compare_invert(invert_mock_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(gz)) > 1000
    compare_invert(invert_mock_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(gz), max_match_count=300, buffer_count=7)
    for name, blob in parity.zstd_cases(text).items():
        path = tmp_path / f"{name}.log.zst"
        path.write_bytes(blob)
        compare_invert(invert_mock_lib, oracle_lib, None, ["ERROR", "port [0-9]+"], path=str(path))


@pytest.mark.parametrize("devices", ["all", "0,1,2"])
def test_sharded_scan_merges_like_one_device(devices, invert_mock_lib, oracle_lib, monkeypatch, tmp_path):
    """$GPUGREP_DEVICES over three mock devices: line numbers rebased by the merge, same records as one device."""
    monkeypatch.setenv("GPUGREP_MOCK_DEVICES", "3")
    monkeypatch.setenv("GPUGREP_DEVICES", devices)
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
    data = synth.syslog_bytes(1 << 20, seed=77)
    assert compare_invert(invert_mock_lib, oracle_lib, data, synth.C2_PATTERNS, tmp_dir=str(tmp_path)) > 1000
    compare_invert(invert_mock_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=1000, buffer_count=7, tmp_dir=str(tmp_path))
    compare_invert(invert_mock_lib, oracle_lib, data, ["ERROR", "port [0-9]+", "o"], flags=[14, 14, 6], ids=[3, 1, 2], tmp_dir=str(tmp_path))
    buf = ctypes.create_string_buffer(data, len(data))
    rc, sharded, crc, stats = invert_scan_buffer(invert_mock_lib, ctypes.addressof(buf), len(data), 0, synth.C2_PATTERNS)
    assert rc == 0 and stats.segments >= 3
    rc, counted, _, cstats = invert_scan_buffer(invert_mock_lib, ctypes.addressof(buf), len(data), 0, synth.C2_PATTERNS, collect=None)
    assert rc == 0 and counted is None and cstats.matches == len(sharded)
    monkeypatch.delenv("GPUGREP_DEVICES")
    rc, single, crc1, stats1 = invert_scan_buffer(invert_mock_lib, ctypes.addressof(buf), len(data), 0, synth.C2_PATTERNS)
    assert rc == 0 and single == sharded and crc1 == crc and stats1.lines == stats.lines


def test_all_nul_pseudo_line_is_delivered_empty(invert_mock_lib, tmp_path):
    """A pseudo-line of NUL bytes only has no match and is selected; its stripped text is "" (the reference would read stale
    buffer bytes there, so this pins the engine's own behaviour)."""
    check_all_nul_lines(invert_mock_lib, tmp_path)


def check_all_nul_lines(lib, tmp_path):
    path = tmp_path / "nul.log"
    path.write_bytes(b"abc\0\0\0\0\0\0\nfoo\n\0\0")
    rc, got, _, st = invert_scan(lib, str(path), ["zzz"], buffer_size=4)
    assert rc == 0 and got == [(0, 0, b"abc"), (0, 1, b""), (0, 2, b""), (0, 3, b"\n"), (0, 4, b"foo"), (0, 5, b"\n"), (0, 6, b"")]
    assert st.lines == 7 and st.matches == 7
    rc, got, _, _ = invert_scan(lib, str(path), ["foo"], buffer_size=4)
    assert rc == 0 and [ln for _, ln, _ in got] == [0, 1, 2, 3, 5, 6]
    path.write_bytes(b"foo\nbar\n\0\0\0")   # default buffer: the last line is NULs only
    rc, got, _, st = invert_scan(lib, str(path), ["foo"])
    assert rc == 0 and got == [(0, 1, b"bar\n"), (0, 2, b"")] and st.lines == 3
    rc, _, _, st = invert_scan(lib, str(path), ["foo"], collect=None)
    assert rc == 0 and st.matches == 2


def test_scan_and_grep_invert_match(invert_mock_lib, oracle_lib, monkeypatch, tmp_path):
    from hypergrep_b200 import utils

    text = b"".join(b"line %d %s\n" % (k, b"foobar" if k % 3 == 0 else b"nothing") for k in range(5000)) + b"tail without newline"
    path = tmp_path / "grep.log"
    path.write_bytes(text)
    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: invert_mock_lib)
    got = []

    def on_batch(matches, count):
        got.extend((matches[k].id, matches[k].line_number, matches[k].line) for k in range(count))

    assert utils.scan(str(path), ["foobar", "^line 7 "], on_batch, ids=[4, 5], invert_match=True) == 0
    rc, expected, _ = oracle_invert(oracle_lib, str(path), ["foobar", "^line 7 "], ids=[4, 5])
    assert rc == 0 and got == expected and len(got) == 5001 - 1667 - 1
    lines, rc = utils.grep(str(path), ["foobar", "^line 7 "], invert_match=True)
    assert rc == 0 and lines == [(ln + 1, line.decode()) for _, ln, line in expected]
    for limit in (0, 1, 16, 17, 1000):
        want = len(lines) if limit == 0 else min(limit, len(lines))
        assert utils.grep(str(path), ["foobar", "^line 7 "], count_only=True, max_match_count=limit, invert_match=True) == (want, 0)
        assert utils.grep(str(path), ["foobar", "^line 7 "], max_match_count=limit, invert_match=True) == (lines[:want], 0)
    assert utils.grep(str(path), ["FOOBAR"], ignore_case=True, count_only=True, invert_match=True) == (5001 - 1667, 0)
    assert utils.grep(str(path), ["foobar"], only_matching=True, invert_match=True) == ([], 0)
    # positional calls keep their meaning: the new keyword comes last
    assert utils.grep(str(path), ["foobar"], False, True) == (1667, 0)

    class CallbackOnly:   # a plain libhyperscanner.so: no inverted entry point, and no CPU fallback for it
        hyperscan = invert_mock_lib.hyperscan
        check_patterns = invert_mock_lib.check_patterns

        def __getattr__(self, name):
            raise AttributeError(name)

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", CallbackOnly)
    with pytest.raises(NotImplementedError, match="gpugrep_invert_scan_file"):
        utils.grep(str(path), ["foobar"], invert_match=True)
    with pytest.raises(NotImplementedError, match="gpugrep_invert_scan_file"):
        utils.grep(str(path), ["foobar"], count_only=True, invert_match=True)


def _cli(argv, monkeypatch, capsys):
    from hypergrep_b200 import multiscanner

    monkeypatch.setattr("sys.argv", ["hyperscanner"] + argv)
    with pytest.raises(SystemExit) as leave:
        multiscanner.main()
    return leave.value.code, capsys.readouterr().out


def test_cli_invert_options(invert_mock_lib, monkeypatch, capsys, tmp_path):
    from hypergrep_b200 import utils

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: invert_mock_lib)
    mixed, full = tmp_path / "a.log", tmp_path / "b.log"
    mixed.write_bytes(b"foo one\nbar two\nfoo three\nbaz four\nqux five")
    full.write_bytes(b"foo\nfoo foo\n")
    a, b = str(mixed), str(full)
    assert _cli(["-v", "foo", a, b], monkeypatch, capsys) == (0, f"{a}:bar two\n{a}:baz four\n{a}:qux five")
    assert _cli(["-v", "-h", "foo", a], monkeypatch, capsys) == (0, "bar two\nbaz four\nqux five")
    assert _cli(["-v", "-c", "foo", a, b], monkeypatch, capsys) == (0, f"{a}:3\n{b}:0\n")
    assert _cli(["--invert-match", "-c", "foo", b], monkeypatch, capsys) == (1, "0\n")
    assert _cli(["-v", "-t", "foo", a, b], monkeypatch, capsys) == (0, "3\n")
    assert _cli(["-v", "-l", "foo", a, b], monkeypatch, capsys) == (0, f"{a}\n")
    assert _cli(["-v", "-L", "foo", a, b], monkeypatch, capsys) == (0, f"{b}\n")
    assert _cli(["-v", "-q", "foo", a, b], monkeypatch, capsys) == (0, "")
    assert _cli(["-v", "-q", "foo", b], monkeypatch, capsys) == (1, "")
    assert _cli(["-v", "-m", "2", "foo", a], monkeypatch, capsys) == (0, "bar two\nbaz four\n")
    assert _cli(["-v", "-n", "foo", a], monkeypatch, capsys) == (0, "2:bar two\n4:baz four\n5:qux five")
    assert _cli(["-v", "-n", "-H", "-m", "1", "foo", a], monkeypatch, capsys) == (0, f"{a}:2:bar two\n")
    assert _cli(["-v", "-o", "foo", a, b], monkeypatch, capsys) == (0, "")
    assert _cli(["-v", "-o", "foo", b], monkeypatch, capsys) == (1, "")
    assert _cli(["-v", "-o", "-c", "foo", a], monkeypatch, capsys) == (0, "3\n")
    assert _cli(["-v", "-E", "-e", "foo|bar", "-e", "qux", a], monkeypatch, capsys) == (0, "baz four\n")


# ---- GPU: the CUDA engine ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
@pytest.mark.parametrize("seed", range(150))
def test_gpu_random_cases_match_oracle(seed, force_general, gpu_lib, oracle_lib, monkeypatch, tmp_path):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    compare_invert(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match, tmp_dir=str(tmp_path))


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
@pytest.mark.parametrize("buffer_size", [262140, 2048, 64, 8])
def test_gpu_edge_texts(buffer_size, force_general, gpu_lib, oracle_lib, monkeypatch, tmp_path):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    for name, data in sorted(EDGE_TEXTS.items()):
        if parity.has_all_nul_pseudo_line(data, buffer_size):
            continue
        for patterns, flags, ids in _EDGE_SETS + ((["foobar"], None, None),):
            compare_invert(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size=buffer_size, tmp_dir=str(tmp_path))


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_limits_and_segments(force_general, gpu_lib, oracle_lib, monkeypatch, tmp_path):
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    data = synth.syslog_bytes(3 << 20, seed=5, lib=gpu_lib)
    assert compare_invert(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, tmp_dir=str(tmp_path)) > 1000
    compare_invert(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=1000, buffer_count=7, tmp_dir=str(tmp_path))
    compare_invert(gpu_lib, oracle_lib, data[: 1 << 20], ["ERROR", "port [0-9]+", "WARN"], flags=[14, 6, 14], ids=[3, 1, 2], tmp_dir=str(tmp_path))
    compare_invert(gpu_lib, oracle_lib, data[: 1 << 20], ["ERROR", "ssh2$"], buffer_size=50, tmp_dir=str(tmp_path))
    check_all_nul_lines(gpu_lib, tmp_path)


@pytest.mark.gpu
def test_gpu_compressed_inputs(gpu_lib, oracle_lib, tmp_path):
    text = synth.syslog_bytes(4 << 20, seed=9, lib=gpu_lib)
    half = text.rfind(b"\n", 0, len(text) // 2) + 1
    gz = tmp_path / "multi.log.gz"
    gz.write_bytes(parity.gz_members([text[:half], text[half:]]))
    assert compare_invert(gpu_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(gz)) > 1000
    for kind in ("gzip", "zstd"):
        for name, blob in parity.member_layout_cases(kind, text[: 1 << 20]).items():
            if kind == "gzip" and name == "corrupt_member":
                # How much garbage zlib inflates from a corrupt member before it reports the error differs between the
                # reference's gzgets() and the engine's decoder; a normal scan agrees only because no pattern matches the
                # garbage, while an inverted scan selects every garbage line.
                continue
            path = tmp_path / f"{kind}_{name}"
            path.write_bytes(blob)
            compare_invert(gpu_lib, oracle_lib, None, ["ERROR", "port [0-9]+"], path=str(path))


def _complement(normal_lines, nlines):
    mask = np.ones(nlines, dtype=bool)
    mask[np.asarray(normal_lines, dtype=np.int64)] = False
    return np.flatnonzero(mask)


def _sample_texts(data: bytes, numbers, texts, count=2000, seed=3):
    """The stripped text of a sample of selected lines == the pseudo-line it names (default buffer: lines are '\n' lines)."""
    lines = data.split(b"\n")
    rng = random.Random(seed)
    for k in rng.sample(range(len(numbers)), min(count, len(numbers))):
        ln = numbers[k]
        raw = lines[ln] + (b"\n" if ln < len(lines) - 1 else b"")
        assert texts[k] == stripped(raw), (ln, texts[k][:80])


@pytest.mark.gpu
def test_gpu_multi_segment_text_from_file_host_and_device(gpu_lib, tmp_path):
    """72 MiB of C2 text: file (32 MiB segments), pageable host memory (64 MiB segments) and device memory (one segment), each
    with a callback and count-only: the complement of the normal scan, the same records everywhere."""
    import torch

    data = synth.syslog_bytes(72 << 20, seed=61, lib=gpu_lib)
    path = tmp_path / "c2.log"
    path.write_bytes(data)
    rc, normal, _ = run_scan(gpu_lib, str(path), synth.C2_PATTERNS, buffer_count=4096)
    assert rc == 0 and len(normal) > 10000
    rc, got, _, st = invert_scan(gpu_lib, str(path), synth.C2_PATTERNS, buffer_count=4096)
    assert rc == 0 and st.segments >= 3 and st.path == 1
    numbers = [ln for _, ln, _ in got]
    assert np.array_equal(np.asarray(numbers), _complement([ln for _, ln, _ in normal], st.lines))
    _sample_texts(data, numbers, [text for _, _, text in got])
    crc = zlib.crc32(b"".join(text for _, _, text in got))
    rc, _, _, cst = invert_scan(gpu_lib, str(path), synth.C2_PATTERNS, collect=None)
    assert rc == 0 and cst.matches == len(got)
    host = np.frombuffer(data, dtype=np.uint8)
    dev = torch.from_numpy(host.copy()).cuda()
    torch.cuda.synchronize()
    for ptr, location in ((host.ctypes.data, 0), (dev.data_ptr(), 1)):
        rc, nums, bcrc, bst = invert_scan_buffer(gpu_lib, ptr, len(data), location, synth.C2_PATTERNS, buffer_count=4096, collect="numbers")
        assert rc == 0 and nums == numbers and bcrc == crc and bst.lines == st.lines
        rc, _, _, cst = invert_scan_buffer(gpu_lib, ptr, len(data), location, synth.C2_PATTERNS, collect=None)
        assert rc == 0 and cst.matches == len(got)


@pytest.mark.gpu
def test_gpu_lines_with_nuls_on_the_fast_path(gpu_lib, oracle_lib, tmp_path):
    rng = random.Random(7)
    lines = synth.syslog_bytes(2 << 20, seed=71, lib=gpu_lib).split(b"\n")
    out = []
    for line in lines:
        roll = rng.random()
        if roll < 0.03:
            line = line[:20] + b"\0ERROR behind a NUL"          # the block ends at the NUL: no match there
        elif roll < 0.06:
            line = b"\0\0\0" + line[:30] + b" ERROR after leading NULs"
        elif roll < 0.08:
            line = line + b"\0" + b"x" * rng.randint(0, 3000)
        out.append(line)
    data = b"\n".join(out)
    assert not parity.has_all_nul_pseudo_line(data, 262140)
    assert compare_invert(gpu_lib, oracle_lib, data, ["ERROR", "port [0-9]+"], tmp_dir=str(tmp_path)) > 1000
    path = tmp_path / "nul.log"
    path.write_bytes(data)
    rc, _, _, st = invert_scan(gpu_lib, str(path), ["ERROR", "port [0-9]+"], collect=None)
    assert rc == 0 and st.path == 1, "expected the fast path"


@pytest.mark.gpu
def test_gpu_long_line_in_a_large_device_segment(gpu_lib):
    """A 300 KiB line in a 192 MiB device segment: the segment is scanned again in 64 MiB pieces (one takes the general
    path).  Same records as the same scan from host memory, and the complement of the normal scan."""
    import torch

    size = 192 << 20
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=77, lib=gpu_lib)
    view = host.numpy()
    start = 100 << 20
    while view[start - 1] != 10:
        start += 1
    view[start:start + (300 << 10)] = ord("x")
    dev = host.cuda()
    torch.cuda.synchronize()
    rc, normal, _ = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, buffer_count=4096)
    assert rc == 0
    rc, nums, crc, st = invert_scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, buffer_count=4096, collect="numbers")
    assert rc == 0 and st.split_segments == 1 and st.path == 3, (st.split_segments, st.path)
    assert np.array_equal(np.asarray(nums), _complement([ln for _, ln, _ in normal], st.lines))
    rc, _, _, cst = invert_scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, collect=None)
    assert rc == 0 and cst.matches == len(nums) == st.lines - len(normal)
    rc, hnums, hcrc, hst = invert_scan_buffer(gpu_lib, host.data_ptr(), size, 0, synth.C1_PATTERNS, buffer_count=4096, collect="numbers")
    assert rc == 0 and hnums == nums and hcrc == crc and hst.split_segments == 0


def _short_lines(size: int, seed: int) -> bytes:
    rng = np.random.default_rng(seed)
    words = [b"ok", b"a1", b"ERROR", b"zz9", b"port 80", b"", b"\tq", b"GET /x", b"abcdefghij", b"12:34"]
    weights = np.array([10, 10, 1, 10, 1, 10, 10, 10, 10, 10], dtype=float)   # a few per cent of the lines match
    picks = rng.choice(len(words), size=size // 5, p=weights / weights.sum())
    data = b"\n".join(words[k] for k in picks) + b"\n"
    return data[:size - size % 16]


@pytest.mark.gpu
def test_gpu_short_lines_select_more_records_than_the_fast_path_holds(gpu_lib, oracle_lib, tmp_path):
    """Lines under 16 bytes: nearly every line is selected, far more records than the fast path's n/48 record buffer."""
    import torch

    data = _short_lines(96 << 20, seed=5)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    patterns = ["ERROR", "port [0-9]+"]
    rc, normal, _ = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, buffer_count=4096)
    assert rc == 0
    rc, nums, crc, st = invert_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, buffer_count=4096, collect="numbers")
    assert rc == 0 and st.path == 1 and len(nums) > 4 * len(data) // 48
    assert np.array_equal(np.asarray(nums), _complement([ln for _, ln, _ in normal], st.lines))
    lines = data.split(b"\n")
    assert crc == zlib.crc32(b"".join(lines[ln] + b"\n" for ln in nums))
    rc, _, _, cst = invert_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, collect=None)
    assert rc == 0 and cst.matches == len(nums)
    assert compare_invert(gpu_lib, oracle_lib, data[: 1 << 20], patterns, tmp_dir=str(tmp_path)) > 100000


@pytest.mark.gpu
def test_gpu_multi_group_and_nfa_sets(gpu_lib, oracle_lib, tmp_path):
    patterns, plants = synth.c3_patterns()
    data = synth.syslog_bytes(1 << 20, seed=11, plants=plants, plant_ppm=20000, lib=gpu_lib)
    assert compare_invert(gpu_lib, oracle_lib, data, patterns, tmp_dir=str(tmp_path)) > 1000
    text = synth.syslog_bytes(256 << 10, seed=13, lib=gpu_lib)
    nfa = [r"e.{60}d\b", r"ERROR", r"\bport .{40,80}x"]
    assert compare_invert(gpu_lib, oracle_lib, text, nfa, tmp_dir=str(tmp_path)) > 100
    compare_invert(gpu_lib, oracle_lib, text[: 64 << 10], nfa, flags=[14, 14, 6], ids=[1, 2, 3], tmp_dir=str(tmp_path))
    compare_invert(gpu_lib, oracle_lib, text, [r"session .{150}closed", "ERROR"], tmp_dir=str(tmp_path))


@pytest.mark.gpu
def test_gpu_inverted_count_launches_no_extra_kernel(gpu_lib):
    """Inverted count-only on the fast path is lines - matched lines: no kernel beyond the normal count-only scan."""
    import torch

    data = synth.syslog_bytes(32 << 20, seed=81, lib=gpu_lib)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    for patterns in (synth.C2_PATTERNS, synth.C1_PATTERNS):
        rc, _, normal = scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, collect=False)
        rc2, _, _, inverted = invert_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, patterns, collect=None)
        assert rc == 0 and rc2 == 0 and normal.path == 1 and inverted.path == 1
        assert inverted.launches == normal.launches, (inverted.launches, normal.launches)
        assert inverted.matches == normal.lines - normal.matches and inverted.lines == normal.lines


@pytest.mark.gpu
def test_gpu_cli_invert_in_a_fresh_process(gpu_lib, oracle_lib, tmp_path):
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = tmp_path / "cli.log"
    path.write_bytes(synth.syslog_bytes(512 << 10, seed=301, lib=gpu_lib))
    rc, expected, _ = oracle_invert(oracle_lib, str(path), ["Failed password"])
    assert rc == 0 and expected
    env = dict(os.environ, PYTHONPATH=root)
    cmd = [sys.executable, "-m", "hypergrep_b200.multiscanner"]
    proc = subprocess.run(cmd + ["-v", "-n", "Failed password", str(path)], env=env, capture_output=True, text=True, timeout=300, check=False)
    assert proc.returncode == 0, proc.stderr
    assert proc.stdout == "".join(f"{ln + 1}:{line.decode()}" for (_i, ln, line) in expected)
    proc = subprocess.run(cmd + ["-v", "-c", "Failed password", str(path)], env=env, capture_output=True, text=True, timeout=300, check=False)
    assert proc.returncode == 0 and proc.stdout == f"{len(expected)}\n"


@pytest.mark.gpu
def test_gpu_inverted_scan_over_all_gpus(gpu_lib, oracle_lib, monkeypatch, tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", str(1 << 20))
    data = synth.syslog_bytes(16 << 20, seed=31)
    assert compare_invert(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, tmp_dir=str(tmp_path)) > 10000
    compare_invert(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=5000, buffer_count=7, tmp_dir=str(tmp_path))
