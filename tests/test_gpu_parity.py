"""Parity tests proper: the CUDA engine behind the C ABI (libgpugrep.so) against the CPU oracle, on a B200."""

import ctypes

import numpy as np
import pytest

import parity
from gpu_api import scan_buffer
from hypergrep_b200 import synth
from oracle_api import scan_bytes
from test_host_logic import EDGE_TEXTS, check_only_matching

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(400))
def test_random_cases_match_oracle(seed, gpu_lib, oracle_lib):
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line: reference reads stale bytes, excluded from parity")
    parity.compare(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match)


@pytest.mark.parametrize("name", sorted(EDGE_TEXTS))
@pytest.mark.parametrize("buffer_size", [262140, 2048, 64, 8])
def test_edge_texts(name, buffer_size, gpu_lib, oracle_lib):
    for patterns in (["foo"], ["foobar"], ["foo$", "^bar"], ["o+b", "x{3}"], ["foo."]):
        parity.compare(gpu_lib, oracle_lib, EDGE_TEXTS[name], patterns, buffer_size=buffer_size)
    parity.compare(gpu_lib, oracle_lib, EDGE_TEXTS[name], ["foo", "bar", "o"], flags=[14, 14, 6], ids=[1, 2, 3], buffer_size=buffer_size)


@pytest.mark.parametrize("force_general", [False, True])
def test_multi_segment_syslog(force_general, gpu_lib, oracle_lib, monkeypatch):
    """Fast path (prefilter + verify) and general path (line table) must both equal the oracle, across segment cuts."""
    monkeypatch.setenv("GPUGREP_CHUNK_BYTES", "1")
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    data = synth.syslog_bytes(3 << 20, seed=5, lib=gpu_lib)
    assert parity.compare(gpu_lib, oracle_lib, data, synth.C1_PATTERNS) > 100
    parity.compare(gpu_lib, oracle_lib, data, synth.C2_PATTERNS)
    parity.compare(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=1000, buffer_count=7)
    parity.compare(gpu_lib, oracle_lib, data, ["(?i)error", "Port [0-9]+"], flags=[14, 15])
    parity.compare(gpu_lib, oracle_lib, data[: 1 << 20], ["ERROR", "port [0-9]+", "WARN"], flags=[14, 14, 14], ids=[3, 1, 2])
    parity.compare(gpu_lib, oracle_lib, data[: 1 << 20], ["ERROR", "ssh2$"], buffer_size=50)
    parity.compare(gpu_lib, oracle_lib, data[: 1 << 20], ["ERROR", "ssh2$"], buffer_size=1500)


def test_ioc_set_with_plants(gpu_lib, oracle_lib):
    """configs[2] shape at oracle-friendly size: 1,000 patterns, planted indicators."""
    patterns, plants = synth.c3_patterns()
    data = synth.syslog_bytes(2 << 20, seed=11, plants=plants, plant_ppm=20000, lib=gpu_lib)
    assert parity.compare(gpu_lib, oracle_lib, data, patterns) > 50


def test_caseless_template_set_on_long_lines(gpu_lib, oracle_lib):
    """configs[4] shape at oracle-friendly size: caseless patterns with alternation, bounded repeats and anchors over
    2-16 KiB JSON-ish lines (several DFA groups; lines far longer than a prefilter look-back)."""
    patterns = synth.c5_patterns(300)
    plants = ["session_10247 failed", "code=E4242abc", "REQUEST-EXPIRED-777}", "payment_555 REVOKED", "stalled xxxx31337"]
    data = synth.jsonish_bytes(3 << 20, seed=3, patterns_to_plant=plants, plant_rate=0.2)
    extra = [r"session_\d+ (?:failed|expired)", r"code=(?:E|W)\d{4}[a-f0-9]{2,6}", r"request-expired-\d+\}$", r"^\{\"ts\":\d{10},\"svc\":\"gateway",
             r"stalled x{2,8}\d+", r"payment_\d{3} revoked"]
    flags = [15] * (len(patterns) + len(extra))
    assert parity.compare(gpu_lib, oracle_lib, data, patterns + extra, flags=flags) > 3
    # the same set with distinct ids on a smaller slice (general path: events, SINGLEMATCH per id)
    small = data[: 256 << 10]
    small = small[: small.rfind(b"\n") + 1]
    parity.compare(gpu_lib, oracle_lib, small, extra, flags=[15] * len(extra), ids=list(range(len(extra))))


def test_multiscanner_over_compressed_files(gpu_lib, oracle_lib, tmp_path, monkeypatch, capsys):
    """configs[3] shape: the CLI entry (parallel_grep) over gzip + zstd (one and several frames) + plain files, one
    hyperscan() job per file (spread over the visible GPUs), counts checked against the oracle."""
    import gzip

    from hypergrep_b200 import multiscanner, utils
    from oracle_api import run_scan

    monkeypatch.setattr(utils, "_get_hyperscanner_lib", lambda: gpu_lib)
    files, expected = [], []
    for k in range(6):
        text = synth.syslog_bytes(1 << 20, seed=100 + k, lib=gpu_lib)
        kind = ["gz", "plain", "zst", "gz2", "zst2", "plain"][k]
        half = text.rfind(b"\n", 0, len(text) // 2) + 1
        blob = {"gz": gzip.compress(text, 6), "plain": text, "zst": parity.zstd_frame(text), "gz2": parity.gz_members([text[:half], text[half:]]),
                "zst2": parity.zstd_frame(text[:half]) + parity.zstd_frame(text[half:])}[kind]
        path = tmp_path / f"part{k}.log{'' if kind == 'plain' else '.' + kind[:2].replace('zs', 'zst')}"
        path.write_bytes(blob)
        files.append(str(path))
        rc, got, _ = run_scan(oracle_lib, str(path), synth.C2_PATTERNS)
        assert rc == 0
        expected.append(len(got))
    code = multiscanner.parallel_grep(files, synth.C2_PATTERNS, count_results=True, with_file_name=True)
    lines = capsys.readouterr().out.splitlines()
    assert code == 0
    assert lines == [f"{name}:{count}" for name, count in zip(files, expected)]


def test_compressed_inputs(gpu_lib, oracle_lib, tmp_path):
    text = synth.syslog_bytes(1 << 20, seed=9, lib=gpu_lib)
    half = text.rfind(b"\n", 0, len(text) // 2) + 1
    multi = tmp_path / "multi.log.gz"
    multi.write_bytes(parity.gz_members([text[:half], text[half:]]))
    parity.compare(gpu_lib, oracle_lib, None, ["ERROR"], path=str(multi))
    garbage = tmp_path / "garbage.log.gz"
    garbage.write_bytes(parity.gz_members([text[:half]]) + b"this is not gzip")
    parity.compare(gpu_lib, oracle_lib, None, ["ERROR"], path=str(garbage))
    parity.compare(gpu_lib, oracle_lib, None, ["foo"], path=str(tmp_path / "nope.txt"))
    parity.compare(gpu_lib, oracle_lib, None, ["foo"], path=str(tmp_path))
    # zstd layouts: frames back to back are read through, a skippable frame or garbage after a frame ends the data
    counts = {}
    for name, blob in parity.zstd_cases(text).items():
        path = tmp_path / f"{name}.log.zst"
        path.write_bytes(blob)
        counts[name] = parity.compare(gpu_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(path))
    assert counts["one_frame"] == counts["two_frames"] == counts["three_frames_levels"] == counts["empty_frame_then_text"] > 50
    assert 0 < counts["skippable_between"] == counts["trailing_garbage"] < counts["one_frame"]


@pytest.mark.parametrize("kind", ["gzip", "zstd"])
def test_many_members_decoded_by_several_threads(kind, gpu_lib, oracle_lib, tmp_path, monkeypatch):
    """SURVEY §8(f-1): one file of many gzip members / zstd frames decoded by helper threads from speculative starts
    (ingest_members.cpp).  Every layout gives the records of the reference's single gzgets() stream (hyperscanner.c:189-199)."""
    import gzip

    text = synth.syslog_bytes(2 << 20, seed=31, lib=gpu_lib)
    suffix = ".log.gz" if kind == "gzip" else ".log.zst"
    monkeypatch.setenv("GPUGREP_DECODE_MIN_BYTES", "0")
    for name, blob in parity.member_layout_cases(kind, text).items():
        path = tmp_path / f"{name}{suffix}"
        path.write_bytes(blob)
        counts = set()
        for threads, spacing in (("0", "1048576"), ("6", "2000"), ("3", "50000")):
            monkeypatch.setenv("GPUGREP_DECODE_THREADS", threads)
            monkeypatch.setenv("GPUGREP_DECODE_SPACING", spacing)
            counts.add(parity.compare(gpu_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(path)))
        assert len(counts) == 1 and counts.pop() > 0, (kind, name)
    # a file above the size threshold with the defaults of the machine: 40 MiB of text in 2 MiB members
    for name in ("GPUGREP_DECODE_MIN_BYTES", "GPUGREP_DECODE_THREADS", "GPUGREP_DECODE_SPACING"):
        monkeypatch.delenv(name)
    big = synth.syslog_bytes(40 << 20, seed=37, lib=gpu_lib)
    cuts = [0]
    while cuts[-1] < len(big):
        cuts.append(big.find(b"\n", min(len(big) - 1, cuts[-1] + (2 << 20))) + 1 or len(big))
    pack = (lambda d: gzip.compress(d, 1)) if kind == "gzip" else parity.zstd_frame
    path = tmp_path / f"big{suffix}"
    path.write_bytes(b"".join(pack(big[a:b]) for a, b in zip(cuts, cuts[1:])))
    assert path.stat().st_size > (4 << 20)
    assert parity.compare(gpu_lib, oracle_lib, None, synth.C2_PATTERNS, path=str(path)) > 1000


def test_buffer_entry_points_agree_with_oracle(gpu_lib, oracle_lib):
    """gpugrep_scan_buffer from pageable host memory, pinned host memory and device memory == oracle."""
    import torch

    data = synth.syslog_bytes(4 << 20, seed=21, lib=gpu_lib)
    rc, exp, _ = scan_bytes(oracle_lib, data, synth.C2_PATTERNS)
    assert rc == 0
    host = np.frombuffer(data, dtype=np.uint8)
    rc, got, st = scan_buffer(gpu_lib, host.ctypes.data, host.size, 0, synth.C2_PATTERNS)
    assert rc == 0 and got == exp
    assert st.path & 1, "the prefilter fast path should serve the C2 set"
    assert st.lines == data.count(b"\n")
    pinned = torch.from_numpy(host.copy()).pin_memory()
    rc, got, st = scan_buffer(gpu_lib, pinned.data_ptr(), pinned.numel(), 0, synth.C2_PATTERNS)
    assert rc == 0 and got == exp and st.h2d_bytes == len(data)
    dev = pinned.cuda()
    torch.cuda.synchronize()
    rc, got, st = scan_buffer(gpu_lib, dev.data_ptr(), dev.numel(), 1, synth.C2_PATTERNS)
    assert rc == 0 and got == exp and st.h2d_bytes == 0
    rc, none, st = scan_buffer(gpu_lib, dev.data_ptr(), dev.numel(), 1, synth.C2_PATTERNS, collect=False)
    assert rc == 0 and none is None and st.matches == len(exp)
    # general mode (two ids, one of them not SINGLEMATCH) on device-resident input: events + gathered lines
    pats, flags, ids = ["ERROR", "port [0-9]+", "o"], [14, 14, 6], [3, 1, 2]
    small = data[: 256 << 10]
    small = small[: small.rfind(b"\n") + 1]
    rc, exp2, _ = scan_bytes(oracle_lib, small, pats, flags=flags, ids=ids)
    dev2 = torch.frombuffer(bytearray(small), dtype=torch.uint8).cuda()
    rc, got2, st = scan_buffer(gpu_lib, dev2.data_ptr(), dev2.numel(), 1, pats, flags, ids)
    assert rc == 0 and got2 == exp2


def test_large_scan_properties(gpu_lib):
    """Size-independent properties at 1 GiB (the oracle would need minutes): independent counts and shard invariance."""
    import torch

    size = 1 << 30
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    lines = synth.fill_syslog(host.numpy(), seed=1234, lib=gpu_lib)
    dev = host.cuda()
    torch.cuda.synchronize()
    rc, _, st = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, collect=False)
    assert rc == 0
    assert st.lines == lines == int((dev == 10).sum().item())
    # 'ERROR' only ever appears as the level field, once per line: occurrences == matching lines
    view = host.numpy()
    e = np.flatnonzero(view[:-4] == ord("E"))
    occurrences = int(np.count_nonzero((view[e + 1] == ord("R")) & (view[e + 2] == ord("R")) & (view[e + 3] == ord("O")) & (view[e + 4] == ord("R"))))
    assert st.matches == occurrences
    # shard invariance: 4 newline-aligned byte ranges, line numbers rebased by a prefix sum of shard line counts
    gpu_lib.gpugrep_shard_begin.restype = ctypes.c_size_t
    gpu_lib.gpugrep_shard_begin.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint, ctypes.c_uint]
    cuts = [gpu_lib.gpugrep_shard_begin(host.data_ptr(), size, r, 4) for r in range(5)]
    assert cuts[0] == 0 and cuts[4] == size
    rc, whole, _ = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C2_PATTERNS, max_match_count=0)
    merged, base = [], 0
    for r in range(4):
        # shards start at arbitrary byte offsets: they are read from (pinned) host memory, as a rank would do
        rc, part, pst = scan_buffer(gpu_lib, host.data_ptr() + cuts[r], cuts[r + 1] - cuts[r], 0, synth.C2_PATTERNS)
        assert rc == 0
        merged += [(i, ln + base, text) for (i, ln, text) in part]
        base += pst.lines
    assert base == lines and merged == whole


@pytest.mark.parametrize("seed", range(200, 240))
def test_nfa_fallback_random_cases(seed, gpu_lib, oracle_lib, monkeypatch):
    """Every pattern forced through the bit-parallel NFA fallback (DFA state budget of 3): same reports as the oracle."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "3")
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = parity.random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    parity.compare(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match)


def test_nfa_fallback_for_exploding_patterns(gpu_lib, oracle_lib):
    """Patterns whose DFA is exponential (a gap of n arbitrary bytes) take the NFA path next to ordinary DFA patterns."""
    text = synth.syslog_bytes(256 << 10, seed=13, lib=gpu_lib)
    patterns = [r"e.{60}d\b", r"ERROR", r"\bport .{40,80}x"]
    assert parity.compare(gpu_lib, oracle_lib, text, patterns) > 10
    parity.compare(gpu_lib, oracle_lib, text[: 64 << 10], patterns, flags=[14, 14, 6], ids=[1, 2, 3])


def test_nfa_patterns_ride_the_fast_path(gpu_lib, oracle_lib, monkeypatch):
    """A pattern whose DFA explodes but which has a literal factor (`session .{150}closed`) no longer sends the whole set down
    the general path: its grams mark candidates like any other, and the lines of those candidates are checked by the NFA
    simulation.  Lines with NUL bytes are re-checked with the NFA patterns as well."""
    import random

    import torch

    rng = random.Random(5)
    text = bytearray(synth.syslog_bytes(1 << 20, seed=17, lib=gpu_lib))
    lines = bytes(text).split(b"\n")
    out = []
    for k, line in enumerate(lines):
        roll = rng.random()
        if roll < 0.02:
            filler = bytes(rng.choice(b"abcdefghij ") for _ in range(rng.choice([149, 150, 151, 200])))
            line = line[:40] + b" session " + filler + b"closed " + line[40:]
        elif roll < 0.03:
            line = line[:20] + b"\0session " + b"x" * 150 + b"closed"       # behind a NUL: must not count
        elif roll < 0.04:
            line = b"\0\0" + line[:30] + b" session " + b"y" * 150 + b"closed"  # leading NULs are stripped: counts
        out.append(line)
    data = b"\n".join(out)
    patterns = [r"session .{150}closed", "ERROR", r"port [0-9]+"]
    assert parity.compare(gpu_lib, oracle_lib, data, patterns) > 100
    assert parity.compare(gpu_lib, oracle_lib, data, [r"session .{150}closed"]) > 10
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    rc, _, st = scan_buffer(gpu_lib, dev.data_ptr(), dev.numel(), 1, patterns, collect=False)
    assert rc == 0 and st.path == 1, "expected the fast path only"
    monkeypatch.setenv("GPUGREP_NFA_GENERAL", "1")
    rc, _, st2 = scan_buffer(gpu_lib, dev.data_ptr(), dev.numel(), 1, patterns, collect=False)
    assert rc == 0 and (st2.path & 2) and st2.matches == st.matches


def test_cli_in_fresh_processes(gpu_lib, oracle_lib, tmp_path):
    """The `hyperscanner` command line end to end, in fresh interpreters: default thread pool and --mp (fork AFTER the
    parent's compile check, which therefore must not have touched CUDA)."""
    import os
    import subprocess
    import sys

    from oracle_api import run_scan

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files, expected = [], []
    for k in range(3):
        text = synth.syslog_bytes(512 << 10, seed=300 + k, lib=gpu_lib)
        path = tmp_path / f"cli{k}.log"
        path.write_bytes(text)
        files.append(str(path))
        rc, got, _ = run_scan(oracle_lib, str(path), ["Failed password", "port [0-9]+"])
        expected.append(len(got))
    env = dict(os.environ, PYTHONPATH=root)
    for extra in ([], ["--mp"]):
        cmd = [sys.executable, "-m", "hypergrep_b200.multiscanner", "-E", "-c", "-e", "Failed password", "-e", "port [0-9]+"] + extra + files
        proc = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300, check=False)
        assert proc.returncode == 0, proc.stdout + proc.stderr
        assert proc.stdout.splitlines() == [f"{name}:{count}" for name, count in zip(files, expected)]
    # -n output of one file equals the oracle's (1-based numbers, lines with their text)
    rc, got, _ = run_scan(oracle_lib, files[0], ["Failed password"])
    proc = subprocess.run([sys.executable, "-m", "hypergrep_b200.multiscanner", "-n", "Failed password", files[0]], env=env,
                          capture_output=True, text=True, timeout=300, check=False)
    assert proc.returncode == 0
    assert proc.stdout == "".join(f"{ln + 1}:{line.decode()}" for (_i, ln, line) in got)


def test_default_buffer_boundary_lines(gpu_lib, oracle_lib):
    """Lines of exactly buffer_size-2, -1, 0, +1 bytes around the default gzgets buffer (262,140): the pseudo-line split
    (SURVEY.md §8a-2 rule 1) with matches on both sides of every cut, between ordinary lines."""
    limit = 262140 - 1
    parts = [b"foo first\n"]
    for total in (limit - 1, limit, limit + 1, limit + 2, 2 * limit, 2 * limit + 5):
        body = bytearray(b"x" * (total - 1))
        body[10:13] = b"foo"
        body[limit - 2:limit + 1] = b"foo" if len(body) > limit + 1 else body[limit - 2:limit + 1]   # straddles the first cut
        if len(body) > limit + 20:
            body[limit + 5:limit + 8] = b"foo"
        parts.append(bytes(body) + b"\n")
        parts.append(b"bar between\n")
    parts.append(b"foo last")
    data = b"".join(parts)
    assert parity.compare(gpu_lib, oracle_lib, data, ["foo"]) >= 8
    parity.compare(gpu_lib, oracle_lib, data, ["foo", "bar"], flags=[14, 6], ids=[1, 2])
    parity.compare(gpu_lib, oracle_lib, data, ["o{2}$", "^x+foo"])


@pytest.mark.parametrize("switch", ["", "GPUGREP_NO_REPROBE=1", "GPUGREP_NO_MIXED_STRIDE=1", "GPUGREP_NO_TUNE=1", "GPUGREP_FILTER=exact",
                                    "GPUGREP_MAX_DFA_STATES=300", "GPUGREP_VERIFY=v1", "GPUGREP_NFA_GENERAL=1", "GPUGREP_NO_EXT_CONFIRM=1"])
def test_every_optimisation_switch_gives_the_same_result(switch, gpu_lib, oracle_lib, monkeypatch):
    """Each fast-path optimisation can be turned off (INTEGRATION.md): the result never changes.  The pattern sets carry
    a switch-specific extra literal so that no cached database or gram table of another variant is reused.
    GPUGREP_MAX_DFA_STATES=300 splits the sets into many DFA groups (group gating in the verification kernel)."""
    if switch:
        name, value = switch.split("=")
        monkeypatch.setenv(name, value)
    tag = "zq" + "".join(ch for ch in switch if ch.isalnum())[-12:] + "qz"
    patterns, plants = synth.c3_patterns()
    data = synth.syslog_bytes(2 << 20, seed=21, plants=plants + ["ERROR"], plant_ppm=20000, lib=gpu_lib)
    assert parity.compare(gpu_lib, oracle_lib, data, patterns[:200] + [tag]) > 10                 # multi-group, large gram set
    assert parity.compare(gpu_lib, oracle_lib, data, ["ERROR", "connection reset by peer", tag]) > 10   # mixed sampling
    assert parity.compare(gpu_lib, oracle_lib, data, synth.C2_PATTERNS + [tag]) > 100
    parity.compare(gpu_lib, oracle_lib, data, ["(?i)error", "Port [0-9]+", tag], flags=[14, 15, 14])


def test_long_lines_with_nuls_take_the_cooperative_searches(gpu_lib, oracle_lib):
    """Lines of 0.3-6 KiB (longer than the per-thread bound of the emit kernel, so their extents are finished by the
    whole warp), some with NUL bytes before or after the match: the strip / cut rule (hyperscanner.c:205-217) decides
    whether the line counts, and the has-NUL hint must survive the hand-over between the two searches."""
    import random
    rng = random.Random(99)
    words = ["alpha", "bravo", "charlie", "delta", "echo", "foxtrot", "golf", "hotel", "india", "juliett"]
    lines = []
    for k in range(400):
        target = rng.choice([40, 300, 900, 2500, 6000])
        parts = []
        size = 0
        while size < target:
            w = rng.choice(words) + str(rng.randint(0, 999))
            parts.append(w)
            size += len(w) + 1
        if rng.random() < 0.5:
            parts.insert(rng.randint(0, len(parts)), "needle-in-haystack")
        text = " ".join(parts)
        roll = rng.random()
        if roll < 0.25:   # a NUL somewhere: a match behind it must not count, one in front of it must
            at = rng.randint(0, len(text))
            text = text[:at] + "\0" + text[at:]
        elif roll < 0.35:
            text = "\0\0" + text   # leading NULs are stripped
        lines.append(text)
    data = ("\n".join(lines) + "\n").encode("latin1")
    assert parity.compare(gpu_lib, oracle_lib, data, ["needle-in-haystack"]) > 50
    parity.compare(gpu_lib, oracle_lib, data, ["needle-in-haystack", "juliett9[0-9]{2}$", "^alpha1"])


def test_fast_path_capacity_overflow_falls_back(gpu_lib, oracle_lib):
    """A text in which more than half of all 16-byte chunks hold a gram of the set overflows the candidate list of the
    fast path; a text of very short matching lines overflows its record buffer.  Both segments are redone on the
    general path (stats.path bit 1) with identical results."""
    from gpu_api import scan_buffer as scan
    import torch

    dense = (b"abcdabcdabcdabcd" * 40 + b"\n") * 3000 + b"tail without the gram\n"
    short = b"abcd\n" * 200000
    for data in (dense, short):
        assert parity.compare(gpu_lib, oracle_lib, data, ["abcd"]) > 1000
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        rc, _, st = scan(gpu_lib, dev.data_ptr(), dev.numel(), 1, ["abcd"], collect=False)
        assert rc == 0 and (st.path & 2), "expected the general-path fallback"


@pytest.mark.parametrize("patterns", [["^GET "], ["^abcd"], ["^foo:"], ["^.abcdefg"], [r"\AGET /index"], ["^GET ", "POST /submit"],
                                      [r"^\s*warn: disk"], ["(?i)^get /INDEX"]])
def test_anchored_match_at_every_line_start_alignment(patterns, gpu_lib, oracle_lib, monkeypatch):
    """Regression (round-1 advisor finding): the local verification walk starts `lookback` bytes before the candidate chunk,
    rounded down to a word.  A line that starts exactly there has its '\\n' one byte BEFORE the window; the walk must
    still enter in the start-of-line state, or ^ / \\A matches are lost for about one line start in sixteen."""
    from test_compiler import anchored_alignment_text

    heads = {"^GET ": b"GET ", "^abcd": b"abcd", "^foo:": b"foo:", "^.abcdefg": b"Zabcdefg", r"\AGET /index": b"GET",
             r"^\s*warn: disk": b"  warn: disk", "(?i)^get /INDEX": b"GET"}
    data = anchored_alignment_text(heads[patterns[0]])
    flags = [14] * len(patterns)
    assert parity.compare(gpu_lib, oracle_lib, data, patterns, flags=flags) >= 64
    # the same text behind a long filler, so that the walks do not start at offset 0 of the segment, and with tiny segments
    assert parity.compare(gpu_lib, oracle_lib, b"filler line\n" * 1000 + data, patterns, flags=flags) >= 64
    monkeypatch.setenv("GPUGREP_NO_REPROBE", "1")
    assert parity.compare(gpu_lib, oracle_lib, data * 3, patterns + ["zqanchorqz"], flags=flags + [14]) >= 192


def _oracle_records_threaded(oracle_lib, data: bytes, patterns, flags, threads: int):
    """(line number, line bytes) of every oracle result over `data`, the text cut into newline-aligned shards that run
    on `threads` host threads (the 10,000-pattern alternation costs the oracle about a second per MiB on one core)."""
    import threading

    n = len(patterns)
    pa = (ctypes.c_char_p * n)(*[p.encode() for p in patterns])
    fa = (ctypes.c_uint * n)(*flags)
    ia = (ctypes.c_uint * n)(*([0] * n))
    oracle_lib.oracle_lines_buffer.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                                               ctypes.c_int, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_void_p]
    bounds = [0]
    for t in range(1, threads):
        cut = data.find(b"\n", len(data) * t // threads)
        bounds.append(max(bounds[-1], cut + 1 if cut >= 0 else len(data)))
    bounds.append(len(data))
    found, counts = [None] * threads, [0] * threads

    def work(t: int) -> None:
        shard = data[bounds[t]:bounds[t + 1]]
        cap = shard.count(b"\n") + 8
        out = np.zeros(cap, dtype=np.uint64)
        m, ln = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        rc = oracle_lib.oracle_lines_buffer(shard, len(shard), pa, fa, ia, n, 262140, out.ctypes.data, cap, ctypes.byref(m), ctypes.byref(ln))
        assert rc == 0 and m.value <= cap
        found[t], counts[t] = out[: m.value], ln.value

    pool = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for th in pool:
        th.start()
    for th in pool:
        th.join()
    lines = data.split(b"\n")
    records, base = [], 0
    for t in range(threads):
        records += [(int(v) + base, lines[int(v) + base] + b"\n") for v in found[t]]
        base += counts[t]
    return records


def test_ten_thousand_caseless_patterns_full_set(gpu_lib, oracle_lib):
    """configs[4] at its named size: ALL 10,000 caseless template patterns (4 DFA groups, group gating, a candidate
    list close to its capacity) over 64 MiB of 2-16 KiB JSON-ish lines, records compared with the oracle (every matched
    line number and its bytes).  The oracle runs sharded over the host cores."""
    import os

    patterns = synth.c5_patterns(10000)
    flags = [15] * len(patterns)
    plants = ["session_10247 failed", "code=E4242abc", "REQUEST-EXPIRED-777}", "payment_555 REVOKED", "stalled xxxx31337"]
    planted = [p for p in patterns if p.startswith("session_")][:40]
    plants += [p.split(" ")[0] + " " + p.split("(?:")[1].split("|")[0] for p in planted]   # literal instances of real set members
    sample = synth.jsonish_bytes(8 << 20, seed=7, patterns_to_plant=plants, plant_rate=0.3)
    data = sample * 8   # 64 MiB: the generator is pure Python; the repeats still cross every segment / tile boundary differently
    expected = _oracle_records_threaded(oracle_lib, data, patterns, flags, max(2, min(32, os.cpu_count() or 2)))
    assert len(expected) > 200
    host = np.frombuffer(data, dtype=np.uint8)
    rc, got, st = scan_buffer(gpu_lib, host.ctypes.data, host.size, 0, patterns, flags=flags, buffer_count=4096)
    assert rc == 0
    assert [(ln, text) for (_i, ln, text) in got] == expected
    assert st.lines == data.count(b"\n")


def test_one_input_over_all_gpus(gpu_lib, oracle_lib, monkeypatch, tmp_path):
    """$GPUGREP_DEVICES=all: one file / one host buffer split into a newline-aligned range per GPU, merged on the calling
    thread (prefix sum of the shard line counts, ordered callbacks, max_match_count cut).  Needs two GPUs."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    monkeypatch.setenv("GPUGREP_DEVICES", "all")
    monkeypatch.setenv("GPUGREP_MIN_SHARD_BYTES", str(1 << 20))
    data = synth.syslog_bytes(48 << 20, seed=31)
    assert parity.compare(gpu_lib, oracle_lib, data, synth.C2_PATTERNS) > 10000
    parity.compare(gpu_lib, oracle_lib, data, synth.C2_PATTERNS, max_match_count=5000, buffer_count=7)
    parity.compare(gpu_lib, oracle_lib, data[: 4 << 20], ["ERROR", "port [0-9]+", "o"], flags=[14, 14, 6], ids=[3, 1, 2])
    # a large pinned buffer: the sharded result equals the single-device result record for record
    size = 1 << 30
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    lines = synth.fill_syslog(host.numpy(), seed=1234)
    rc, sharded, st = scan_buffer(gpu_lib, host.data_ptr(), size, 0, synth.C2_PATTERNS, buffer_count=4096)
    assert rc == 0 and st.lines == lines and st.segments >= 2
    monkeypatch.delenv("GPUGREP_DEVICES")
    rc, single, st1 = scan_buffer(gpu_lib, host.data_ptr(), size, 0, synth.C2_PATTERNS, buffer_count=4096)
    assert rc == 0 and single == sharded and st1.lines == lines


def test_text_drift_retunes_the_prefilter(gpu_lib, oracle_lib, monkeypatch):
    """The prefilter windows are tuned on the head of the input.  When the text changes character later on (syslog lines
    first, then access-log lines in which `zqxjk=` is on every line), the segments of the second half flag far more
    chunks than the sample promised; the windows are then chosen again with text of the drifting region (`500 w` instead
    of `zqxj`).  Results never change (the filter is a superset filter) - the candidate count does."""
    import random

    import torch

    monkeypatch.setenv("GPUGREP_CHUNK_MB", "4")
    first = synth.syslog_bytes(16 << 20, seed=41)
    rng = random.Random(43)
    lines = []
    size = 0
    while size < (16 << 20):
        code = 500 if rng.random() < 0.01 else rng.choice([200, 200, 200, 204, 301, 404])
        line = f"ts={rng.randint(1_600_000_000, 1_800_000_000)} zqxjk={code} {'wvfgh' if code == 500 else 'gateway'} unavailable bytes={rng.randint(0, 99999)} path=/api/v{rng.randint(1, 3)}/items/{rng.randint(0, 10 ** 6)}\n"
        lines.append(line)
        size += len(line)
    data = first + "".join(lines).encode()
    patterns = synth.C2_PATTERNS + ["zqxjk=500 wvfgh"]   # no window of it occurs in the syslog half: the tuner cannot know that `zqxjk=` will be on every line later
    assert parity.compare(gpu_lib, oracle_lib, data, patterns) > 1000
    host = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    rc, _, tuned = scan_buffer(gpu_lib, host.data_ptr(), host.numel(), 0, patterns, collect=False)
    monkeypatch.setenv("GPUGREP_NO_RETUNE", "1")
    rc2, _, fixed = scan_buffer(gpu_lib, host.data_ptr(), host.numel(), 0, patterns, collect=False)
    assert rc == 0 and rc2 == 0 and tuned.matches == fixed.matches and tuned.path == 1
    print(f"candidates with re-tuning {tuned.candidates}, without {fixed.candidates}")
    assert tuned.candidates < fixed.candidates


def test_long_line_costs_one_piece_not_the_segment(gpu_lib):
    """A line too long for the fast path (an aligned 64 KiB without a newline) used to send its whole device-resident segment - up to
    2 GiB - down the general path.  Now the segment is scanned again in 64 MiB pieces and only the piece that holds the
    line takes the general path; the result is the same as ever."""
    import torch

    size = 192 << 20
    host = torch.empty(size, dtype=torch.uint8).pin_memory()
    synth.fill_syslog(host.numpy(), seed=77)
    view = host.numpy()
    start = 100 << 20
    while view[start - 1] != 10:
        start += 1
    view[start:start + (300 << 10)] = ord("x")   # one line of more than 300 KiB: longer than the gzgets buffer, it is split into pseudo-lines
    dev = host.cuda()
    torch.cuda.synchronize()
    rc, _, st = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, collect=False)
    assert rc == 0
    e = np.flatnonzero(view[:-4] == ord("E"))
    occurrences = int(np.count_nonzero((view[e + 1] == ord("R")) & (view[e + 2] == ord("R")) & (view[e + 3] == ord("O")) & (view[e + 4] == ord("R"))))
    # (the long line is two pseudo-lines: 262,139 bytes, then the rest)
    assert st.matches == occurrences and st.lines == int(np.count_nonzero(view == 10)) + 1
    assert st.split_segments == 1 and st.path == 3, (st.split_segments, st.path)
    # records too (line numbers and bytes), against the same scan from host memory in small segments
    rc, dev_records, _ = scan_buffer(gpu_lib, dev.data_ptr(), size, 1, synth.C1_PATTERNS, buffer_count=4096)
    rc2, host_records, st2 = scan_buffer(gpu_lib, host.data_ptr(), size, 0, synth.C1_PATTERNS, buffer_count=4096)
    assert rc == 0 and rc2 == 0 and dev_records == host_records and st2.split_segments == 0


def test_only_matching_spans_from_match_ends(gpu_lib, tmp_path, monkeypatch):
    """SURVEY §8(f-4): `grep -o` spans from the device's match END offsets (gpugrep_match_ends) == re.finditer over every
    matched line (reference utils.py:205-212), for fixed-width patterns; everything else keeps the reference's way."""
    check_only_matching(gpu_lib, tmp_path, monkeypatch)


def test_device_text_reads_stay_inside_the_buffer():
    """Memory safety of caller-owned device text (GPUGREP_LOC_DEVICE, include/gpugrep.h): the kernels read nothing before
    `data` and nothing past data + round_up(size, 16).  compute-sanitizer is closed on the GPU pool, so the text is placed
    flush against UNMAPPED virtual pages (cuMemMap) and every kernel path is run over it in a subprocess: a stray read
    is an illegal-address fault there (tests/guarded_device_scan.py)."""
    import os
    import subprocess
    import sys

    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "guarded_device_scan.py")
    done = subprocess.run([sys.executable, script], capture_output=True, text=True, timeout=900, check=False)
    assert done.returncode == 0, done.stdout[-2000:] + done.stderr[-2000:]
    assert "guarded scans ok" in done.stdout


def test_match_ends_from_host_and_device_memory(gpu_lib):
    """gpugrep_match_ends on the GPU: every (line, id, end) of fixed-width patterns equals what Python's re finds with an
    overlapping search, for host memory and for a device-resident buffer."""
    import re

    import torch

    from hypergrep_b200 import utils

    text = synth.syslog_bytes(3 << 20, seed=53, lib=gpu_lib)
    patterns = ["ERROR", "port [0-9]{5}", r"\d\d:\d\d:\d\d", "ss"]
    expected = []
    for number, line in enumerate(text.split(b"\n")[:-1]):
        row = []
        for pid, pattern in enumerate(patterns):
            for m in re.finditer(b"(?=(" + pattern.encode() + b"))", line):
                row.append((m.end(1), pid))
        expected += [(number, pid, end) for end, pid in sorted(row)]
    pa, fa, ia = utils.prepare_patterns(patterns, flags=[0] * len(patterns), ids=list(range(len(patterns))))
    entry = gpu_lib.gpugrep_match_ends
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                      ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    host = np.frombuffer(text, dtype=np.uint8)
    dev = torch.from_numpy(host.copy()).cuda()
    torch.cuda.synchronize()
    for pointer, location in ((host.ctypes.data, 0), (dev.data_ptr(), 1)):
        out = (utils._MatchEnd * (len(expected) + 16))()
        found = ctypes.c_size_t()
        assert entry(pointer, len(text), location, pa, fa, ia, len(patterns), 262140, out, len(expected) + 16, ctypes.byref(found), None) == 0
        assert found.value == len(expected)
        got = [(out[k].line_number, out[k].id, out[k].end) for k in range(found.value)]
        assert got == expected, location
