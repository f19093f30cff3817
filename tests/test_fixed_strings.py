"""Fixed strings (grep -F): gpugrep_literal_scan_file / gpugrep_literal_scan_buffer / gpugrep_check_literals, scan() / grep()
with fixed_strings and the CLI's -F.

The expected answer is the one include/gpugrep.h defines: the records of gpugrep_context_scan_* for the same set with every
byte written as \\xHH, the flags plus SINGLEMATCH and ids 0 (`escaped`), and a plain Python model of the definition
(`model_selected`: substring search in the scanned block, A-Z/a-z folded for caseless literals).  CPU tests run the host
logic on the stand-in with fixed strings (tests/mock_engine_literal), whose matcher is that definition, against the context
stand-in's regex scan of the escaped set; `gpu` tests run the CUDA engine (fast and general path) against both."""

from __future__ import annotations

import ctypes
import gzip
import os
import random
import shutil
import subprocess
import time

import numpy as np
import pytest

import parity
from gpu_api import Stats, marshal
from hypergrep_b200 import synth
from oracle_api import CALLBACK

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIT_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                  ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
_LIT_BUFFER_ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p,
                    ctypes.c_int, ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p,
                    ctypes.c_void_p]
_CTX_FILE_ARGS = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_int,
                  ctypes.c_int, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_void_p]
EDGE_TEXTS = {
    "empty": b"",
    "no_newline": b"foo bar",
    "only_newlines": b"\n\n\n\n",
    "crlf": b"foo\r\nbar foo\r\n\r\nfoo",
    "leading_nuls": b"\0\0foo\nbar\n\0foo bar\n\0\0\0\n",
    "inner_nul": b"foo\0bar\nbar\0foo\nfoo\n\0\0bar\0foo\n",
    "long_line": b"x" * 700 + b"foo" + b"y" * 300 + b"\nfoo\n",
    "split_by_buffer": b"0123456fo" + b"obar\n" + b"foobar\n" + b"ab" * 40 + b"\n",
    "high_bytes": bytes(range(256)) + b"\n" + bytes(range(255, -1, -1)) + b"\n@`[{\n",
}
EDGE_LITERALS = ([b"foo", b"bar\n", b"Oo", b"\xff\xfe", b"\x01\x02\x03", b"ab\nc", b"`", b"[{", b"abab", b"AbAbA"],
                 [0, 0, 1, 0, 0, 0, 1, 1, 1, 1])


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
    arr = (ctypes.c_char_p * max(n, 1))(*[lit if isinstance(lit, bytes) else lit.encode() for lit in literals])
    fl = (ctypes.c_uint * max(n, 1))(*(list(flags) if flags else [0] * n)) if flags is not None else None
    return arr, fl, n


def literal_scan(lib, path, literals, flags=None, buffer_size=262140, buffer_count=16, max_match_count=0, before=0, after=0, invert=False,
                 collect=True):
    entry = lib.gpugrep_literal_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _LIT_FILE_ARGS
    la, fa, n = _lits(literals, flags)
    sink, stats = _Collector(collect), Stats()
    rc = entry(path.encode(), la, fa, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def literal_scan_buffer(lib, ptr, size, location, literals, flags=None, buffer_size=262140, buffer_count=16, max_match_count=0, before=0,
                        after=0, invert=False, collect=True):
    entry = lib.gpugrep_literal_scan_buffer
    entry.restype, entry.argtypes = ctypes.c_int, _LIT_BUFFER_ARGS
    la, fa, n = _lits(literals, flags)
    sink, stats = _Collector(collect), Stats()
    rc = entry(ptr, size, location, la, fa, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert), None,
               ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def escaped(literals, flags):
    """The oracle's pattern set: every byte as \\xHH, flags | SINGLEMATCH, ids 0."""
    pats = ["".join(f"\\x{b:02x}" for b in (lit if isinstance(lit, bytes) else lit.encode())) for lit in literals]
    return pats, [(f if flags else 0) | 8 for f in (flags or [0] * len(literals))]


def context_oracle(lib, path, literals, flags=None, buffer_size=262140, buffer_count=16, max_match_count=0, before=0, after=0,
                   invert=False, collect=True):
    pats, fl = escaped(literals, flags)
    pa, fa, ia, n = marshal(pats, fl, [0] * len(pats))
    entry = lib.gpugrep_context_scan_file
    entry.restype, entry.argtypes = ctypes.c_int, _CTX_FILE_ARGS
    sink, stats = _Collector(collect), Stats()
    rc = entry(path.encode(), pa, fa, ia, n, sink.pointer(), buffer_size, buffer_count, max_match_count, before, after, int(invert),
               ctypes.byref(stats))
    return rc, sink.records, sink.batches, stats


def _fold(data: bytes) -> bytes:
    return data.translate(bytes(b | 0x20 if 65 <= b <= 90 else b for b in range(256)))


def pseudo_lines(data: bytes, buffer_size: int = 262140):
    limit = max(1, buffer_size - 1)
    pos, out = 0, []
    while pos < len(data):
        nl = data.find(b"\n", pos, pos + limit)
        end = nl + 1 if nl >= 0 else min(len(data), pos + limit)
        out.append(data[pos:end])
        pos = end
    return out


def block_of(line: bytes) -> bytes:
    body = line.lstrip(b"\0")
    cut = body.find(b"\0")
    return body if cut < 0 else body[:cut]


def model_selected(data: bytes, literals, flags=None, buffer_size: int = 262140) -> np.ndarray:
    """The definition: per pseudo-line, does its scanned block contain a literal (caseless: both sides A-Z folded)?"""
    exact = [lit for lit, f in zip(literals, flags or [0] * len(literals)) if not f & 1]
    caseless = [_fold(lit) for lit, f in zip(literals, flags or [0] * len(literals)) if f & 1]
    out = []
    for line in pseudo_lines(data, buffer_size):
        block = block_of(line)
        folded = _fold(block) if caseless else b""
        out.append(any(lit in block for lit in exact) or any(lit in folded for lit in caseless))
    return np.array(out, dtype=bool)


@pytest.fixture(scope="session")
def literal_mock_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_literal")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal.so"))


@pytest.fixture(scope="session")
def context_mock_lib() -> ctypes.CDLL:
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "mock_engine_context")], stdout=subprocess.DEVNULL)
    return ctypes.CDLL(os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_context.so"))


def random_set(rng: random.Random, count: int, lo: int = 1, hi: int = 12, alphabet: bytes = b"abcAB@`[{\n\x80\xff.") -> tuple[list, list]:
    lits = [bytes(rng.choice(alphabet) for _ in range(rng.randint(lo, hi))).replace(b"\0", b"") or b"a" for _ in range(count)]
    return lits, [rng.choice((0, 1, 2, 8, 9, 14)) for _ in range(count)]


def random_text(rng: random.Random, size: int, lits) -> bytes:
    parts = []
    while sum(map(len, parts)) < size:
        r = rng.random()
        if r < 0.3:
            parts.append(rng.choice(lits))
        elif r < 0.4:
            parts.append(b"\n")
        elif r < 0.42:
            parts.append(b"\0")
        else:
            parts.append(bytes(rng.choice(b"abcABC@`[{\x80\xff. \n") for _ in range(rng.randint(1, 20))))
    return b"".join(parts)


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_check_literals_return_codes(literal_mock_lib):
    entry = literal_mock_lib.gpugrep_check_literals
    entry.restype, entry.argtypes = ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint]

    def check(lits, flags=None):
        la, fa, n = _lits(lits, flags)
        return entry(la, fa, n)

    assert check([]) == 4
    assert check([b"ok", b""]) == 4
    assert check([b"a+b(", b"x"]) == 0
    for bit in (1, 2, 4, 8, 15):
        assert check([b"abc"], [bit]) == 0
    for bit in (16, 32, 1 << 31):
        assert check([b"abc"], [bit | 1]) == 4
    assert check([b"dup", b"dup", b"DUP"], [0, 0, 1]) == 0


def test_compile_a_million_literals(literal_mock_lib):
    rng = np.random.default_rng(5)
    lengths = rng.integers(8, 65, size=1_000_000)
    blob = rng.integers(33, 127, size=int(lengths.sum()), dtype=np.uint8).tobytes()
    offsets = np.concatenate(([0], np.cumsum(lengths)))
    lits = [blob[offsets[i]:offsets[i + 1]] for i in range(len(lengths))]
    text = ctypes.create_string_buffer(b"x\n" + lits[7] + b"\n")
    t0 = time.perf_counter()
    rc, got, _, _ = literal_scan_buffer(literal_mock_lib, ctypes.addressof(text), len(lits[7]) + 3, 0, lits)
    elapsed = time.perf_counter() - t0
    print(f"compiled and scanned 10^6 literals of 8-64 bytes in {elapsed:.1f} s")
    assert rc == 0 and [r[1] for r in got] == [1]
    assert elapsed < 60


@pytest.mark.parametrize("name", sorted(EDGE_TEXTS))
@pytest.mark.parametrize("buffer_size", [4, 9, 262140])
def test_edge_texts_against_the_oracle(name, buffer_size, literal_mock_lib, context_mock_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(EDGE_TEXTS[name])
    lits, flags = EDGE_LITERALS
    for invert, before, after in ((False, 0, 0), (True, 0, 0), (False, 1, 2)):
        want = context_oracle(context_mock_lib, str(path), lits, flags, buffer_size=buffer_size, before=before, after=after, invert=invert)
        got = literal_scan(literal_mock_lib, str(path), lits, flags, buffer_size=buffer_size, before=before, after=after, invert=invert)
        assert got[:3] == want[:3]
    selected = model_selected(EDGE_TEXTS[name], lits, flags, buffer_size)
    got = literal_scan(literal_mock_lib, str(path), lits, flags, buffer_size=buffer_size)[1]
    assert [r[1] for r in got] == list(np.flatnonzero(selected))


@pytest.mark.parametrize("seed", range(6))
def test_random_sets_limits_batches_and_context(seed, literal_mock_lib, context_mock_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")   # many segments: context windows and limits across segment bounds
    rng = random.Random(seed)
    lits, flags = random_set(rng, rng.randint(1, 40))
    data = random_text(rng, 60_000, lits)
    path = tmp_path / "r.log"
    path.write_bytes(data)
    for kw in ({}, {"max_match_count": 7, "buffer_count": 3}, {"invert": True, "max_match_count": 11}, {"before": 2, "after": 3},
               {"before": 1, "after": 0, "max_match_count": 5, "buffer_count": 4}, {"buffer_size": 17}):
        want = context_oracle(context_mock_lib, str(path), lits, flags, **kw)
        got = literal_scan(literal_mock_lib, str(path), lits, flags, **kw)
        assert got[0] == want[0] == 0 and got[1:3] == want[1:3], kw
        counted = literal_scan(literal_mock_lib, str(path), lits, flags, collect=False, **kw)
        assert counted[3].matches == want[3].matches


def test_compressed_and_sharded(literal_mock_lib, context_mock_lib, tmp_path, monkeypatch):
    text = synth.syslog_bytes(1 << 20, seed=3, lib=context_mock_lib)
    lits = [b"Failed password", b"port 22", b"SESSION", b"error:", b"\xff\xfe"]
    flags = [0, 0, 1, 0, 0]
    plain = tmp_path / "p.log"
    plain.write_bytes(text)
    want = context_oracle(context_mock_lib, str(plain), lits, flags, before=1, after=1)
    assert len(want[1]) > 100
    gz = tmp_path / "p.log.gz"
    gz.write_bytes(gzip.compress(text))
    assert literal_scan(literal_mock_lib, str(gz), lits, flags, before=1, after=1)[:2] == want[:2]
    for name, blob in parity.zstd_cases(text).items():
        path = tmp_path / f"{name}.log.zst"
        path.write_bytes(blob)
        assert literal_scan(literal_mock_lib, str(path), lits, flags, before=1, after=1)[:2] == \
            context_oracle(context_mock_lib, str(path), lits, flags, before=1, after=1)[:2], name
    monkeypatch.setenv("GPUGREP_MOCK_DEVICES", "3")
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", "100000")
    assert literal_scan(literal_mock_lib, str(plain), lits, flags, before=1, after=1)[:2] == want[:2]
    limited = context_oracle(context_mock_lib, str(plain), lits, flags, max_match_count=50, after=2, invert=True)
    assert literal_scan(literal_mock_lib, str(plain), lits, flags, max_match_count=50, after=2, invert=True)[:3] == limited[:3]


def test_older_engine_stand_ins_refuse_fixed_strings(context_mock_lib, tmp_path):
    path = tmp_path / "t.log"
    path.write_bytes(b"foo\nbar\n")
    assert literal_scan(context_mock_lib, str(path), [b"foo"])[0] == 7
    assert literal_scan(context_mock_lib, str(path), [b""])[0] == 4


@pytest.fixture()
def py_on_mock(literal_mock_lib, monkeypatch):
    from hypergrep_b200 import utils  # pylint: disable=import-outside-toplevel
    monkeypatch.setenv("GPUGREP_LIBRARY", os.path.join(ROOT, "tests", "_build", "libgpugrep_hostmock_literal.so"))
    monkeypatch.setitem(utils._state, "lib", None)  # pylint: disable=protected-access
    return utils


def test_python_keywords(py_on_mock, tmp_path):
    utils = py_on_mock
    path = tmp_path / "k.log"
    path.write_bytes(b"a.b\naxb\nA.B\n(x+\n")
    assert utils.grep(str(path), ["a.b"], fixed_strings=True) == ([(1, "a.b\n")], 0)
    assert utils.grep(str(path), ["a.b"]) == ([(1, "a.b\n"), (2, "axb\n")], 0)
    assert utils.grep(str(path), ["a.b"], fixed_strings=True, ignore_case=True, count_only=True) == (2, 0)
    assert utils.grep(str(path), ["(x+"], fixed_strings=True) == ([(4, "(x+\n")], 0)
    assert utils.grep(str(path), ["a.b"], fixed_strings=True, invert_match=True, before_context=1)[0][:2] == [(1, "a.b\n", True), (2, "axb\n", False)]
    assert utils.grep(str(path), ["a.b"], fixed_strings=True, only_matching=True) == utils.grep(str(path), [r"a\.b"], only_matching=True)
    with pytest.raises(ValueError):
        utils.scan(str(path), ["a"], lambda *_: None, ids=[1], fixed_strings=True)
    assert utils.check_compatibility(["(x+"], fixed_strings=True) == 0
    assert utils.check_compatibility(["(x+"]) == 4
    assert utils.check_compatibility(["x"], flags=[16], fixed_strings=True) == 4


_SYSTEM_GREP = shutil.which("grep")


def _cli(monkeypatch, capsys, argv):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel
    monkeypatch.setattr("sys.argv", ["hyperscanner"] + argv)
    with pytest.raises(SystemExit) as done:
        multiscanner.main()
    return done.value.code, capsys.readouterr().out


def test_cli_fixed_strings(py_on_mock, monkeypatch, capsys, tmp_path):
    from hypergrep_b200 import multiscanner  # pylint: disable=import-outside-toplevel
    assert multiscanner.parse_args(["-F", "x", "f"]).regexp == "fixed"
    with pytest.raises(SystemExit):
        multiscanner.parse_args(["-F", "-E", "x", "f"])
    path = tmp_path / "c.log"
    path.write_bytes(b"a.b\naxb\na+b(\n")
    assert _cli(monkeypatch, capsys, ["-F", "a.b", str(path)]) == (0, "a.b\n")
    assert _cli(monkeypatch, capsys, ["-E", "a.b", str(path)]) == (0, "a.b\naxb\na+b(\n")
    assert _cli(monkeypatch, capsys, ["-F", "a+b(", str(path)]) == (0, "a+b(\n")
    plist = tmp_path / "pats"
    plist.write_text("axb\na+b(\n")
    assert _cli(monkeypatch, capsys, ["-F", "-n", "-f", str(plist), str(path)]) == (0, "2:axb\n3:a+b(\n")
    code, out = _cli(monkeypatch, capsys, ["-F", "", str(path)])
    assert code == 2


@pytest.mark.skipif(_SYSTEM_GREP is None, reason="no system grep")
@pytest.mark.parametrize("seed", range(3))
def test_cli_against_system_grep(seed, py_on_mock, monkeypatch, capsys, tmp_path):
    rng = random.Random(seed)
    words = [b"alpha", b"Beta", b"gamma.x", b"de(lta", b"EPS", b"zz"]
    lines = [b" ".join(rng.choice(words + [b"filler", b"x y"]) for _ in range(rng.randint(0, 5))) for _ in range(300)]
    path = tmp_path / "s.log"
    path.write_bytes(b"\n".join(lines) + b"\n")
    other = tmp_path / "empty.log"
    other.write_bytes(b"nothing here\n")
    pats = [w.decode() for w in rng.sample(words, 2)]
    for opts in (["-c"], ["-v"], ["-n"], ["-i"], ["-A", "1", "-B", "2"], ["-l"], ["-i", "-v", "-c"]):
        files = [str(path), str(other)] if "-l" in opts else [str(path)]
        argv = ["-F"] + opts + sum((["-e", p] for p in pats), []) + files
        want = subprocess.run([_SYSTEM_GREP] + argv, capture_output=True, text=True, check=False, env={"LC_ALL": "C"})
        code, out = _cli(monkeypatch, capsys, argv)
        assert (code, out) == (want.returncode, want.stdout), opts


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _device(data: bytes):
    import torch  # pylint: disable=import-outside-toplevel
    dev = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return dev


def _gpu_compare(gpu_lib, data: bytes, lits, flags, tmp_path, kinds=("file", "host", "device"), **kw):
    """Literal scan == context scan of the escaped set (the oracle) on every input kind; returns the records."""
    path = tmp_path / "g.log"
    path.write_bytes(data)
    want = context_oracle(gpu_lib, str(path), lits, flags, **kw)
    assert want[0] == 0
    got = literal_scan(gpu_lib, str(path), lits, flags, **kw)
    assert got[:3] == want[:3]
    host = ctypes.create_string_buffer(data, len(data) + 1)
    if "host" in kinds:
        got = literal_scan_buffer(gpu_lib, ctypes.addressof(host), len(data), 0, lits, flags, **kw)
        assert got[:3] == want[:3]
    if "device" in kinds:
        dev = _device(data)
        got = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, **kw)
        assert got[:3] == want[:3]
    return want[1], got[3]


@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
def test_gpu_edges_and_alphabet(force_general, gpu_lib, tmp_path, monkeypatch):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    lits, flags = EDGE_LITERALS
    for text in EDGE_TEXTS.values():
        for buffer_size in (9, 262140):
            _gpu_compare(gpu_lib, text, lits, flags, tmp_path, buffer_size=buffer_size)
            _gpu_compare(gpu_lib, text, lits, flags, tmp_path, buffer_size=buffer_size, invert=True, before=1, after=1)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_gpu_random_sets_on_syslog(seed, gpu_lib, tmp_path):
    """Mixed caseless and exact literals, high bytes, NULs and '\\n'-ended literals planted in syslog text: fast path (the
    literals are long enough for the prefilter) and the general path of the short ones, against the oracle and the model."""
    rng = random.Random(seed)
    base = synth.syslog_bytes(8 << 20, seed=seed)
    lines = base.split(b"\n")
    lits = [bytes(rng.choice(b"abcdefghXYZ0123456789@`[{\x80\xfe ") for _ in range(rng.randint(4 if seed % 2 == 0 else 2, 24)))
            for _ in range(rng.choice((50, 2000)))]
    lits += [b"Failed password for", b"sshd[", b"\xff\xfe\xfd\xfc", b"port 22\n", b"@`[{"]
    flags = [rng.choice((0, 1, 8, 9)) for _ in lits]
    for k in range(0, len(lines), 97):
        lines[k] = lines[k] + rng.choice(lits).replace(b"\n", b"") + (b"\0tail" if k % 5 == 0 else b"")
    data = b"\n".join(lines)
    recs, stats = _gpu_compare(gpu_lib, data, lits, flags, tmp_path, buffer_count=4096)
    selected = model_selected(data, lits, flags)
    assert [r[1] for r in recs] == list(np.flatnonzero(selected))
    if seed % 2 == 0:
        assert stats.path & 1
    _gpu_compare(gpu_lib, data, lits, flags, tmp_path, kinds=("device",), buffer_count=4096, invert=True, max_match_count=5000, after=2)
    dev = _device(data)
    counted = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, flags, collect=False)
    assert counted[0] == 0 and counted[3].matches == int(selected.sum())


def _model_np(data: bytes, lits: list[bytes]) -> np.ndarray:
    """Selected lines of exact literals by a rolling hash per distinct literal length, then an exact check; the NUL cut is
    applied by replacing everything after the first NUL of a line with a byte that no literal holds."""
    lines = pseudo_lines(data)
    blocks = [block_of(line) for line in lines]
    text = b"\x01".join(blocks)
    starts = np.cumsum([0] + [len(b) + 1 for b in blocks])
    arr = np.frombuffer(text, dtype=np.uint8).astype(np.uint64)
    selected = np.zeros(len(lines), dtype=bool)
    by_len: dict[int, set] = {}
    for lit in lits:
        by_len.setdefault(len(lit), set()).add(lit)
    mul = np.uint64(1099511628211)
    for length, group in by_len.items():
        if len(arr) < length:
            continue
        h = np.zeros(len(arr) - length + 1, dtype=np.uint64)
        for k in range(length):
            h = h * mul + arr[k:len(arr) - length + 1 + k]
        targets = {}
        for lit in group:
            v = 0
            for b in lit:
                v = (v * 1099511628211 + b) & 0xFFFFFFFFFFFFFFFF
            targets.setdefault(v, []).append(lit)
        hits = np.flatnonzero(np.isin(h, np.array(list(targets), dtype=np.uint64)))
        for pos in hits:
            if text[pos:pos + length] in group:
                selected[np.searchsorted(starts, pos, side="right") - 1] = True
    return selected


@pytest.mark.gpu
@pytest.mark.parametrize("count", [100_000, 1_000_000])
def test_gpu_large_ioc_sets_against_numpy_model(count, gpu_lib):
    rng = np.random.default_rng(count)
    iocs = [f"{a}.{b}.{c}.{d}".encode() for a, b, c, d in rng.integers(1, 255, size=(count // 2, 4))]
    hexd = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)
    iocs += [rng.choice(hexd, size=32).tobytes() for _ in range(count - len(iocs))]
    data = bytearray(synth.syslog_bytes(64 << 20, seed=11))
    planted = rng.choice(len(iocs), size=2000)
    lines = bytes(data).split(b"\n")
    step = len(lines) // 2001
    for k, j in enumerate(planted):
        lines[(k + 1) * step] += b" ioc=" + iocs[j] + (b"\0x" if k % 7 == 0 else b"")
    data = b"\n".join(lines)
    want = _model_np(data, iocs)
    assert want.sum() >= 1500
    dev = _device(data)
    rc, recs, _, stats = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, buffer_count=1 << 16)
    assert rc == 0 and [r[1] for r in recs] == list(np.flatnonzero(want))
    assert stats.path & 1
    rc, _, _, stats = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, iocs, collect=False, invert=True)
    assert rc == 0 and stats.matches == len(want) - int(want.sum())


@pytest.mark.gpu
def test_gpu_shared_prefix_set(gpu_lib):
    """100k literals that share their first 16 bytes, over text full of that prefix: bounded per-hit work."""
    prefix = b"https://www.exa/"
    rng = np.random.default_rng(1)
    alnum = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    tails = {rng.choice(alnum, size=int(rng.integers(4, 20))).tobytes() for _ in range(100_000)}
    lits = [prefix + t for t in sorted(tails)]
    lines = [prefix + rng.choice(alnum, size=24).tobytes() for _ in range(300_000)]
    for k in range(0, len(lines), 1000):
        lines[k] = b"GET " + lits[(k * 7919) % len(lits)] + b" 200"
    data = b"\n".join(lines) + b"\n"
    want = _model_np(data, lits)
    dev = _device(data)
    t0 = time.perf_counter()
    rc, recs, _, _ = literal_scan_buffer(gpu_lib, dev.data_ptr(), len(data), 1, lits, buffer_count=1 << 16)
    print(f"shared-prefix scan: {time.perf_counter() - t0:.2f} s")
    assert rc == 0 and [r[1] for r in recs] == list(np.flatnonzero(want))


# The launch counts and paths of C2 regex scans (8 MiB of configs[1] syslog, device memory), read at the parent commit of
# the fixed-string stage: the stage must not change what regex scans launch.
C2_REGEX_PIN = {"plain": (0, 9, 1), "invert": (0, 15, 1), "count": (0, 9, 1)}


@pytest.mark.gpu
def test_gpu_regex_scans_keep_their_launches(gpu_lib):
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
    sink = _Collector(True)
    rc = entry(ctypes.c_void_p(dev.data_ptr()), ctypes.c_size_t(len(data)), 1, pa, fa, ia, n, sink.pointer(), 262140, 16,
               ctypes.c_ulonglong(0), None, ctypes.byref(stats))
    got["invert"] = (rc, stats.launches, stats.path)
    assert got == C2_REGEX_PIN
