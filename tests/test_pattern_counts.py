"""Per-pattern line counts: gpugrep_pattern_counts_file / _buffer, hypergrep_b200.count_patterns and the CLI's
--count-per-pattern.

The expected counts come from per-id records: counts[i] is the number of distinct lines among the records with id i that
hyperscan() delivers for the same patterns with flags | SINGLEMATCH and ids = index (`record_counts`).  The PCRE2 oracle
gives them on the CPU (fixed strings written as \\xHH escapes), and on the GPU so does the CUDA engine's own multi-id scan
and scan_literals.  CPU tests run the host logic on the stand-in tests/mock_engine_pattern_counts; `gpu` tests run the CUDA
engine on both paths."""

from __future__ import annotations

import ctypes
import gzip
import os
import random
import subprocess

import pytest

import byte_cases
import parity
from gpu_api import Stats, scan_buffer
from hypergrep_b200 import synth
from oracle_api import run_scan
from regex_gen import gen_regex, gen_text
from test_fixed_strings import EDGE_LITERALS, EDGE_TEXTS, escaped

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNTS_LIB = os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_pattern_counts.so")
LITERAL_LIB = os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal.so")
_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_int, ctypes.c_int,
                ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
REGEX_SET = (["foo", "ba[rz]", "o+b", "^x", "o$", "(?:ab|cd)e", "\\d{3}", "foo", "\\xff", "\\x00?q"], [0, 1, 0, 2, 4, 1, 0, 0, 0, 0])


def _arrays(patterns, flags):
    n = len(patterns)
    pa = (ctypes.c_char_p * max(n, 1))(*[p if isinstance(p, bytes) else p.encode() for p in patterns])
    fa = (ctypes.c_uint * max(n, 1))(*(flags if flags is not None else [0] * n))
    return pa, fa, n


def counts_file(lib, path, patterns, flags=None, fixed=False, buffer_size=262140):
    entry = lib.gpugrep_pattern_counts_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    pa, fa, n = _arrays(patterns, flags)
    counts, stats = (ctypes.c_ulonglong * max(n, 1))(), Stats()
    rc = entry(str(path).encode(), pa, fa, n, int(fixed), buffer_size, counts, ctypes.byref(stats))
    return rc, list(counts[:n]), stats


def counts_buffer(lib, ptr, size, location, patterns, flags=None, fixed=False, buffer_size=262140):
    entry = lib.gpugrep_pattern_counts_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _BUFFER_ARGS
    pa, fa, n = _arrays(patterns, flags)
    counts, stats = (ctypes.c_ulonglong * max(n, 1))(), Stats()
    rc = entry(ptr, size, location, pa, fa, n, int(fixed), buffer_size, None, counts, ctypes.byref(stats))
    return rc, list(counts[:n]), stats


def record_counts(records, n):
    """Distinct lines per id of hyperscan() records."""
    lines = [set() for _ in range(n)]
    for rid, number, _ in records:
        lines[rid].add(number)
    return [len(s) for s in lines]


def oracle_counts(oracle_lib, path, patterns, flags, fixed=False, buffer_size=262140):
    """(counts, matched lines) from the oracle: ids = index, flags | SINGLEMATCH; fixed strings as \\xHH escapes."""
    pats, fl = escaped(patterns, flags) if fixed else (patterns, [f | 8 for f in flags])
    rc, recs, _ = run_scan(oracle_lib, str(path), pats, fl, list(range(len(pats))), buffer_size=buffer_size)
    assert rc == 0
    rc, lines, _ = run_scan(oracle_lib, str(path), pats, fl, [0] * len(pats), buffer_size=buffer_size)
    assert rc == 0
    return record_counts(recs, len(pats)), len(lines)


@pytest.fixture(scope="module")
def counts_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_pattern_counts")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(COUNTS_LIB)


@pytest.fixture(scope="module")
def literal_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(LITERAL_LIB)


def _random_set(rng: random.Random, count: int):
    pats = [gen_regex(rng) for _ in range(count)]
    return pats, [rng.choice([0, 1, 2, 4, 7]) for _ in pats]


def _compiles(oracle_lib, pats, flags) -> bool:
    from oracle_api import check  # pylint: disable=import-outside-toplevel
    return check(oracle_lib, pats, [f | 8 for f in flags], list(range(len(pats)))) == 0


def _cases(oracle_lib, seed: int):
    """Random regex sets and texts that the oracle compiles, the edge texts and the byte alphabet."""
    rng = random.Random(seed)
    while True:
        pats, flags = _random_set(rng, rng.randint(2, 12))
        if _compiles(oracle_lib, pats, flags):
            break
    yield "random", gen_text(rng, 200, nul_rate=0.02), pats, flags
    for name, text in EDGE_TEXTS.items():
        yield name, text, REGEX_SET[0], REGEX_SET[1]
    yield "alphabet", byte_cases.byte_text(random.Random(seed), 300, nul_rate=0.02), REGEX_SET[0], REGEX_SET[1]


# ---- CPU: the host logic on the stand-in --------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("buffer_size", [4, 9, 262140])
def test_regex_counts_against_the_oracle(seed, buffer_size, counts_lib, oracle_lib, tmp_path):
    for name, text, pats, flags in _cases(oracle_lib, seed):
        path = tmp_path / f"{name}.log"
        path.write_bytes(text)
        want, matched = oracle_counts(oracle_lib, path, pats, flags, buffer_size=buffer_size)
        rc, got, stats = counts_file(counts_lib, path, pats, flags, buffer_size=buffer_size)
        assert (rc, got, stats.matches) == (0, want, matched), name


@pytest.mark.parametrize("buffer_size", [4, 9, 262140])
def test_fixed_counts_against_the_oracle(buffer_size, counts_lib, oracle_lib, tmp_path):
    lits, flags = EDGE_LITERALS[0] + [b"foo", b"fo", b"oo"], EDGE_LITERALS[1] + [1, 0, 0]
    texts = dict(EDGE_TEXTS, alphabet=byte_cases.byte_text(random.Random(3), 300, nul_rate=0.02))
    for name, text in texts.items():
        path = tmp_path / f"{name}.log"
        path.write_bytes(text)
        want, matched = oracle_counts(oracle_lib, path, lits, flags, fixed=True, buffer_size=buffer_size)
        rc, got, stats = counts_file(counts_lib, path, lits, flags, fixed=True, buffer_size=buffer_size)
        assert (rc, got, stats.matches) == (0, want, matched), name
        assert got[lits.index(b"ab\nc")] == 0


def test_inputs_segments_and_shards(counts_lib, oracle_lib, tmp_path, monkeypatch):
    """gzip, zstd, host buffers, several segments and three shards give the counts of one plain scan."""
    text = synth.syslog_bytes(3 << 20, seed=5)
    pats = ["Failed password", "sshd\\[[0-9]+\\]", "port 22", "session", "root", "x{3}", "kernel:", "port 22"]
    flags = [0, 0, 0, 1, 0, 0, 0, 0]
    lits = [b"Failed password", b"sshd", b"port 22", b"SESSION", b"root", b"zzzz", b"port 22"]
    lflags = [0, 0, 0, 1, 0, 0, 0]
    plain = tmp_path / "p.log"
    plain.write_bytes(text)
    for patterns, fl, fixed in ((pats, flags, False), (lits, lflags, True)):
        want = oracle_counts(oracle_lib, plain, patterns, fl, fixed=fixed)
        assert sum(want[0]) > 1000
        gz = tmp_path / "p.log.gz"
        gz.write_bytes(gzip.compress(text, compresslevel=1))
        got = counts_file(counts_lib, gz, patterns, fl, fixed)
        assert (got[0], got[1], got[2].matches) == (0, want[0], want[1])
        blob = next(iter(parity.zstd_cases(text).values()))
        zst = tmp_path / "p.log.zst"
        zst.write_bytes(blob)
        assert counts_file(counts_lib, zst, patterns, fl, fixed)[1] == want[0]
        host = ctypes.create_string_buffer(text, len(text))
        assert counts_buffer(counts_lib, ctypes.addressof(host), len(text), 0, patterns, fl, fixed)[1] == want[0]
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_CHUNK_MB", "1")
            got = counts_file(counts_lib, plain, patterns, fl, fixed)
            assert got[1] == want[0] and got[2].segments >= 3
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_MOCK_DEVICES", "3")
            env.setenv("GPUGREP_DEVICES", "all")
            env.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
            for got in (counts_file(counts_lib, plain, patterns, fl, fixed),
                        counts_buffer(counts_lib, ctypes.addressof(host), len(text), 0, patterns, fl, fixed)):
                assert (got[0], got[1], got[2].matches) == (0, want[0], want[1])


def test_return_codes(counts_lib, literal_lib, tmp_path):
    path = tmp_path / "r.log"
    path.write_bytes(b"foo\nbar\n")
    assert counts_file(counts_lib, path, [], [])[0] == 4
    entry = counts_lib.gpugrep_pattern_counts_file
    entry.restype, entry.argtypes = ctypes.c_int, _FILE_ARGS
    pa, fa, n = _arrays(["foo"], [0])
    assert entry(str(path).encode(), pa, fa, n, 0, 262140, None, None) == 4
    assert counts_file(counts_lib, path, ["foo", "("], [0, 0])[0] == 4          # does not compile, as hyperscan() says
    assert counts_file(counts_lib, path, ["foo", "a*"], [0, 0])[0] == 4         # matches the empty buffer
    assert counts_file(counts_lib, path, ["foo", ""], [0, 0], fixed=True)[0] == 4
    assert counts_file(counts_lib, path, ["foo"], [64], fixed=True)[0] == 4
    assert counts_file(counts_lib, path, ["foo"], [64])[0] == 4
    assert counts_file(counts_lib, tmp_path / "missing.log", ["foo"], [0])[0] != 0
    # an error leaves every count 0, whatever the array held
    counts = (ctypes.c_ulonglong * 2)(5, 5)
    assert entry(str(tmp_path / "missing.log").encode(), *_arrays(["foo", "bar"], [0, 0]), 0, 262140, counts, None) != 0
    assert list(counts) == [0, 0]
    # a build of the engine without the stage
    assert counts_file(literal_lib, path, ["foo", "bar"], [0, 0])[0] == 7
    assert counts_file(literal_lib, path, ["foo"], [0], fixed=True)[0] == 7
    # one pattern; identical patterns each get their own count; SINGLEMATCH changes nothing
    assert counts_file(counts_lib, path, ["o"], [0])[1] == [1]
    assert counts_file(counts_lib, path, ["o", "o", "[ab]"], [8, 0, 8])[1] == [1, 1, 1]
    assert counts_file(counts_lib, path, [b"o", b"o", b"FOO"], [0, 8, 1], fixed=True)[1] == [1, 1, 1]


@pytest.fixture()
def py_on_mock(counts_lib, monkeypatch):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    monkeypatch.setenv("GPUGREP_LIBRARY", COUNTS_LIB)
    monkeypatch.setitem(utils._state, "lib", None)  # pylint: disable=protected-access
    return utils


def test_python_count_patterns(py_on_mock, monkeypatch, tmp_path):
    import hypergrep_b200  # pylint: disable=import-outside-toplevel
    utils = py_on_mock
    assert hypergrep_b200.count_patterns is utils.count_patterns
    path = tmp_path / "k.log"
    path.write_bytes("a.b x\nxa.b\nA.B\n(x+ é\né\nnone\n".encode())
    assert utils.count_patterns(str(path), ["a.b", "é", "zz", "A"]) == ([2, 2, 0, 1], 0)
    assert utils.count_patterns(str(path), ["a.b", "é", "zz", "A"], ignore_case=True) == ([3, 2, 0, 3], 0)
    assert utils.count_patterns(str(path), ["a.b", "(x+"], fixed_strings=True) == ([2, 1], 0)
    assert utils.count_patterns(str(path), ["a.b", "(x+"], flags=[9, 8], fixed_strings=True) == ([3, 1], 0)
    assert utils.count_patterns(str(path), ["(x+"]) == ([0], 4)
    assert utils.count_patterns(str(path), ["x"], buffer_size=3) == ([3], 0)
    with pytest.raises(ValueError):
        utils.count_patterns(str(path), ["a", ""])
    with pytest.raises(ValueError):
        utils.count_patterns(str(path), ["a", "b"], flags=[0])
    monkeypatch.setitem(utils._state, "lib", object())  # pylint: disable=protected-access
    with pytest.raises(NotImplementedError):
        utils.count_patterns(str(path), ["a"])


def _cli(monkeypatch, capsys, argv):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel
    monkeypatch.setattr("sys.argv", ["hyperscanner"] + argv)
    with pytest.raises(SystemExit) as done:
        multiscanner.main()
    return done.value.code, capsys.readouterr().out


def test_cli_count_per_pattern(py_on_mock, monkeypatch, capsys, tmp_path):
    a, b = tmp_path / "a.log", tmp_path / "b.log"
    a.write_bytes(b"foo bar\nfoo\nBAR x\n")
    b.write_bytes(b"nothing\nbar\n")
    plist = tmp_path / "p.txt"
    plist.write_bytes(b"x\nzz\n")
    cpp = ["--count-per-pattern"]
    assert _cli(monkeypatch, capsys, cpp + ["-e", "foo", "-e", "bar", str(a)]) == (0, "2:foo\n1:bar\n")
    assert _cli(monkeypatch, capsys, cpp + ["-i", "-e", "foo", "-e", "bar", str(a), str(b)]) == \
        (0, f"{a}:2:foo\n{a}:2:bar\n{b}:0:foo\n{b}:1:bar\n")
    assert _cli(monkeypatch, capsys, cpp + ["-h", "-e", "foo", "-f", str(plist), str(b), str(a)]) == (0, "2:foo\n1:x\n0:zz\n0:foo\n0:x\n0:zz\n")
    assert _cli(monkeypatch, capsys, cpp + ["-H", "foo", str(a)]) == (0, f"{a}:2:foo\n")
    assert _cli(monkeypatch, capsys, cpp + ["-t", "-i", "-e", "foo", "-e", "bar", str(a), str(b)]) == (0, "2:foo\n3:bar\n")
    assert _cli(monkeypatch, capsys, cpp + ["-F", "-e", "o b", "-e", "o.b", str(a)]) == (0, "1:o b\n0:o.b\n")
    assert _cli(monkeypatch, capsys, cpp + ["-E", "-e", "fo+|x", str(a)]) == (0, "3:fo+|x\n")
    # the pattern as written, before the BRE / GNU rewrites
    assert _cli(monkeypatch, capsys, cpp + ["-e", "fo\\+", "-e", "\\<bar", str(a)]) == (0, "2:fo\\+\n1:\\<bar\n")
    assert _cli(monkeypatch, capsys, cpp + ["--no-order", "--no-sort", "--no-gnu", "-s", "zz", str(a)]) == (1, "0:zz\n")
    code, out = _cli(monkeypatch, capsys, cpp + ["-s", "foo", str(tmp_path / "missing.log"), str(a)])
    assert code == 2 and out == f"{a}:2:foo\n"
    code, out = _cli(monkeypatch, capsys, cpp + ["foo", str(tmp_path / "missing.log")])
    assert code == 2 and out.count("\n") == 1
    for extra in (["-v"], ["-o"], ["-F", "-w"], ["-F", "-x"], ["-c"], ["-l"], ["-L"], ["-q"], ["-m", "2"], ["-n"], ["-A", "1"], ["-B", "1"],
                  ["-C", "1"], ["-m", "0"], ["-A", "0"], ["-B", "0"], ["-C", "0"]):
        code, out = _cli(monkeypatch, capsys, cpp + extra + ["foo", str(a)])
        assert code == 2 and out.count("\n") == 1, extra


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _device(data: bytes, offset: int = 0):
    import torch  # pylint: disable=import-outside-toplevel
    dev = torch.frombuffer(bytearray(b"\n" * offset + data) or bytearray(1), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return dev


def _gpu_counts_both_paths(gpu_lib, path, patterns, flags, fixed, monkeypatch, buffer_size=262140):
    fast = counts_file(gpu_lib, path, patterns, flags, fixed, buffer_size)
    with monkeypatch.context() as env:
        env.setenv("GPUGREP_FORCE_GENERAL", "1")
        general = counts_file(gpu_lib, path, patterns, flags, fixed, buffer_size)
    assert fast[0] == general[0] == 0 and not general[2].path & 1
    assert fast[1] == general[1] and fast[2].matches == general[2].matches
    return fast


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_gpu_against_the_oracle(seed, gpu_lib, oracle_lib, tmp_path, monkeypatch):
    for buffer_size in (9, 262140):
        for name, text, pats, flags in _cases(oracle_lib, seed):
            path = tmp_path / f"{name}.log"
            path.write_bytes(text)
            want, matched = oracle_counts(oracle_lib, path, pats, flags, buffer_size=buffer_size)
            got = _gpu_counts_both_paths(gpu_lib, path, pats, flags, False, monkeypatch, buffer_size)
            assert (got[1], got[2].matches) == (want, matched), (name, buffer_size)
    lits, lflags = EDGE_LITERALS[0] + [b"foo", b"fo", b"oo", b"\n"], EDGE_LITERALS[1] + [1, 0, 0, 0]
    for name, text in dict(EDGE_TEXTS, alphabet=byte_cases.byte_text(random.Random(seed), 300, nul_rate=0.02)).items():
        path = tmp_path / f"{name}.fixed.log"
        path.write_bytes(text)
        want, matched = oracle_counts(oracle_lib, path, lits, lflags, fixed=True)
        got = _gpu_counts_both_paths(gpu_lib, path, lits, lflags, True, monkeypatch)
        assert (got[1], got[2].matches) == (want, matched), name


def _engine_counts(gpu_lib, ptr, size, patterns, flags):
    rc, recs, _ = scan_buffer(gpu_lib, ptr, size, 1, patterns, flags, list(range(len(patterns))))
    assert rc == 0
    return record_counts(recs, len(patterns))


@pytest.mark.gpu
def test_gpu_configs_against_the_engine_and_both_paths(gpu_lib, monkeypatch):
    """configs[1], configs[2] with its plants and a configs[4] sample: counts equal the per-id records of the engine's own
    multi-id scan; the fast path and the general path agree; stats.matches is the count-only scan."""
    c3, plants = synth.c3_patterns()
    c5 = synth.c5_patterns(10000)
    cases = [
        ("c1", synth.syslog_bytes(32 << 20, seed=11), synth.C2_PATTERNS, [14] * len(synth.C2_PATTERNS)),
        ("c2", synth.syslog_bytes(32 << 20, seed=12, plants=plants, plant_ppm=1000), c3, [14] * len(c3)),
        ("c4", synth.jsonish_bytes(4 << 20, patterns_to_plant=["session_4242 failed", "code=E31337abcd"]), c5, [15] * len(c5)),
    ]
    for name, data, pats, flags in cases:
        dev = _device(data)
        rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, pats, flags)
        assert rc == 0 and stats.path == 1, name
        assert got == _engine_counts(gpu_lib, dev.data_ptr(), len(data), pats, flags), name
        assert stats.matches == scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, pats, flags, collect=False)[2].matches
        assert sum(1 for c in got if c) > (1 if name == "c1" else 5), name
        with monkeypatch.context() as env:
            env.setenv("GPUGREP_FORCE_GENERAL", "1")
            general = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, pats, flags)
        assert general[1] == got and general[2].path == 2 and general[2].matches == stats.matches, name


@pytest.mark.gpu
def test_gpu_record_overflow_and_fan_out(gpu_lib):
    """A dense text whose fast-path segment overflows its records takes the general path with the same counts; one line
    matched by all 1,000 patterns counts 1 for each; 10^5 events of one pattern in one line count 1."""
    pats = [f"k{i:03d}" for i in range(1000)]
    flags = [0] * 1000
    dense = b"".join(f"k{i % 1000:03d}\n".encode() for i in range(400_000))
    dev = _device(dense)
    rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(dense), 1, pats, flags)
    assert rc == 0 and got == [400] * 1000 and stats.matches == 400_000 and stats.path & 2
    every = b"x " + b" ".join(p.encode() for p in pats) + b"\n"
    text = b"filler\n" * 1000 + every + b"filler k007\n" * 5 + (b"ab" * 100_000) + b"\n"
    dev = _device(text)
    for extra in ([], ["(?:ab)"]):
        rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(text), 1, pats + extra, flags + [0] * len(extra))
        assert rc == 0 and got[:1000] == [1] * 7 + [6] + [1] * 992 and got[1000:] == [1] * len(extra)
    rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(text), 1, ["ab", "b", "zzz"], [0, 0, 0])
    assert rc == 0 and got == [1, 1, 0] and stats.matches == 1


def _wide_lines_text(seed: int, universe: int, widths: list[int]) -> tuple[bytes, list[set[int]]]:
    """configs[1] text with one line per entry of `widths` inserted at intervals: that many distinct `kNNNN` tokens (NNNN
    below `universe`), some repeated.  Returns the text and, per line of it, the set of NNNN it holds."""
    rng = random.Random(seed)
    lines = synth.syslog_bytes(16 << 20, seed=seed).split(b"\n")[:-1]
    step = len(lines) // (len(widths) + 1)
    for k, width in enumerate(widths):
        tokens = rng.sample(range(universe), width)
        tokens += rng.choices(tokens, k=width // 3)   # repeats: more events, no more ids
        rng.shuffle(tokens)
        lines[(k + 1) * step] = b"wide " + b" ".join(b"k%04d" % t for t in tokens)
    import re  # pylint: disable=import-outside-toplevel
    held = [{int(m) for m in re.findall(rb"k(\d{4})", line)} for line in lines]
    return b"\n".join(lines) + b"\n", held


@pytest.mark.gpu
def test_gpu_lines_over_the_shared_memory_set(gpu_lib, monkeypatch):
    """Lines with more distinct ids than the per-warp hash set holds (1,024) go to the global fallback: more of them in one
    segment than that kernel has blocks (32), so a block reuses its bitmap, and lines just around the cap.  Counts equal a
    model of the text and the engine's own multi-id scan, on both paths; fixed strings too, where each report node carries
    two ids (every literal given twice)."""
    widths = list(range(1500, 5000, 90)) + [1000, 1020, 1023, 1024, 1025, 1026, 1030, 1060, 2, 700]
    assert sum(1 for w in widths if w > 1024) > 32
    data, held = _wide_lines_text(21, 10000, widths)
    dev = _device(data)
    pats = [f"k{i:04d}" for i in range(10000)]
    want = [0] * 10000
    for line in held:
        for t in line:
            want[t] += 1
    matched = sum(1 for line in held if line)
    assert max(len(line) for line in held) >= 4900 and matched >= len(widths)
    rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, pats, [0] * 10000)
    assert (rc, got, stats.matches) == (0, want, matched)
    assert got == _engine_counts(gpu_lib, dev.data_ptr(), len(data), pats, [8] * 10000)
    with monkeypatch.context() as env:
        env.setenv("GPUGREP_FORCE_GENERAL", "1")
        general = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, pats, [0] * 10000)
    assert (general[1], general[2].matches, general[2].path) == (want, matched, 2)
    # fixed strings: 3,000 literals, each given twice (ids i and i + 3,000 share a node); 513 distinct tokens are 1,026 ids
    widths = list(range(600, 2900, 60)) + [500, 510, 511, 512, 513, 514, 530, 3]
    data, held = _wide_lines_text(22, 3000, widths)
    dev = _device(data)
    lits = [b"k%04d" % i for i in range(3000)] * 2
    held = [{t for t in line if t < 3000} for line in held]
    want = [0] * 3000
    for line in held:
        for t in line:
            want[t] += 1
    matched = sum(1 for line in held if line)
    for force in (False, True):
        with monkeypatch.context() as env:
            if force:
                env.setenv("GPUGREP_FORCE_GENERAL", "1")
            rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, [0] * 6000, fixed=True)
        assert (rc, got, stats.matches) == (0, want * 2, matched), force
        assert not force or stats.path == 2


@pytest.mark.gpu
def test_gpu_fixed_strings_against_regex_and_scan_literals(gpu_lib, monkeypatch):
    from test_literal_reports import report_scan_buffer  # pylint: disable=import-outside-toplevel
    from test_whole_literals import ioc_set  # pylint: disable=import-outside-toplevel
    iocs = ioc_set(1000, 5)
    lits = iocs[:300] + [iocs[0], iocs[1][:5], iocs[2][3:], iocs[3].upper(), b"sshd", b"port 22\n", b"a\nb", b"SSHD"]
    flags = [0] * 300 + [0, 0, 0, 1, 0, 0, 0, 1]
    lines = synth.syslog_bytes(16 << 20, seed=7).split(b"\n")
    for k in range(0, len(lines) - 1, 53):
        lines[k] += b" ioc=" + iocs[k % 400]
    data = b"\n".join(lines)
    dev = _device(data)
    rc, got, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, fixed=True)
    assert rc == 0 and stats.path == 1 and got[-2] == 0 and got[300] == got[0] > 0
    pats, rflags = escaped(lits, flags)
    assert got == _engine_counts(gpu_lib, dev.data_ptr(), len(data), pats, rflags)
    rc, recs, _, _ = report_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, [f | 8 for f in flags], list(range(len(lits))))
    assert rc == 0 and record_counts(recs, len(lits)) == got
    with monkeypatch.context() as env:
        env.setenv("GPUGREP_FORCE_GENERAL", "1")
        general = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, fixed=True)
    assert general[1] == got and general[2].path == 2


@pytest.mark.gpu
def test_gpu_inputs_and_shards(gpu_lib, tmp_path, monkeypatch):
    import torch  # pylint: disable=import-outside-toplevel
    c3, plants = synth.c3_patterns()
    data = synth.syslog_bytes(96 << 20, seed=9, plants=plants, plant_ppm=1000)
    path = tmp_path / "i.log"
    path.write_bytes(data)
    want = counts_file(gpu_lib, path, c3, [14] * len(c3))
    assert want[0] == 0 and sum(want[1]) > 300
    gz = tmp_path / "i.log.gz"
    gz.write_bytes(gzip.compress(data[: 8 << 20], compresslevel=1))
    head = counts_file(gpu_lib, gz, c3, [14] * len(c3))
    zst = tmp_path / "i.log.zst"
    zst.write_bytes(next(iter(parity.zstd_cases(data[: 8 << 20]).values())))
    assert counts_file(gpu_lib, zst, c3, [14] * len(c3))[1] == head[1]
    plain_head = tmp_path / "h.log"
    plain_head.write_bytes(data[: 8 << 20])
    assert counts_file(gpu_lib, plain_head, c3, [14] * len(c3))[1] == head[1]
    host = ctypes.create_string_buffer(data, len(data))
    pinned = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    dev = _device(data, offset=3)
    for ptr, location in ((ctypes.addressof(host), 0), (pinned.data_ptr(), 0), (dev.data_ptr() + 3, 1), (dev.data_ptr(), 1)):
        size = len(data) + (3 if ptr == dev.data_ptr() else 0)
        got = counts_buffer(gpu_lib, ptr, size, location, c3, [14] * len(c3))
        assert (got[0], got[1], got[2].matches) == (0, want[1], want[2].matches), (location, ptr % 16)
    with monkeypatch.context() as env:
        env.setenv("GPUGREP_DEVICES", "0,0")
        env.setenv("GPUGREP_MIN_SHARD_BYTES", str(16 << 20))
        env.setenv("GPUGREP_CHUNK_MB", "8")
        for got in (counts_file(gpu_lib, path, c3, [14] * len(c3)), counts_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, c3, [14] * len(c3))):
            assert (got[0], got[1], got[2].matches) == (0, want[1], want[2].matches)
            assert got[2].segments > 2


@pytest.mark.gpu
def test_gpu_regex_scans_keep_their_launches_and_paths(gpu_lib):
    """The C2 regex scans (normal, inverted, count-only) keep the launches and paths read at the parent commit, and a
    pattern-count scan on the fast path is a scan with records plus the line events, their scan and the count."""
    from test_fixed_strings import C2_REGEX_PIN  # pylint: disable=import-outside-toplevel
    from gpu_api import marshal  # pylint: disable=import-outside-toplevel
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
    assert got == C2_REGEX_PIN == {"plain": (0, 9, 1), "invert": (0, 15, 1), "count": (0, 9, 1)}
    rc, counts, stats = counts_buffer(gpu_lib, dev.data_ptr(), len(data), 1, synth.C2_PATTERNS, [14] * len(synth.C2_PATTERNS))
    assert rc == 0 and stats.path == 1 and stats.launches == 9 + 7 and sum(counts) >= stats.matches > 0


@pytest.mark.gpu
def test_gpu_count_patterns_on_the_cuda_library(tmp_path):
    from hypergrep_b200 import count_patterns  # pylint: disable=import-outside-toplevel
    path = tmp_path / "p.log"
    path.write_bytes(synth.syslog_bytes(4 << 20, seed=3))
    got, code = count_patterns(str(path), ["sshd", "SSHD", "port [0-9]+", "zzzz"], ignore_case=True)
    assert code == 0 and got[0] == got[1] > 0 and got[2] > 0 and got[3] == 0
    assert count_patterns(str(path), ["sshd", "SSHD"], fixed_strings=True) == ([got[0], 0], 0)
