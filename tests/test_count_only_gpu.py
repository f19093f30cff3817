"""Count-only scans on the fast path (k_emit_nlm<*, true> -> k_count_keys) and the streaming kernel's per-segment NUL flag
(Totals::flags bit 3, gpugrep_stats.nul_segments).

For every case the count-only `matches` equal the number of records the records path delivers and the oracle's, the
inverted count-only `matches` equal `lines - matches`, and the number of segments flagged with a NUL byte equals the CPU
model's (any NUL in [0, n) of the segment).  Inputs come from host, pinned and device memory.
"""

from __future__ import annotations

import numpy as np
import pytest

import fast_path_cases as fpc
from dfa_sim import CompiledDb
from gpu_api import scan_buffer
from hypergrep_b200 import synth
from k1_model import K1Tables, stream_sweep_bytes
from oracle_api import scan_bytes
from test_fast_path_gpu import _all_grams, _k1_sizes, _on_device, _same_records, _tuned, k1_text
from test_invert_match import invert_scan_buffer

pytestmark = pytest.mark.gpu

HOST, DEVICE = 0, 1
C3_PATTERNS, C3_PLANTS = synth.c3_patterns()
NFA_PATTERNS = [r"session .{150}closed", "ERROR", r"port [0-9]+"]


def k1_has_nul(data) -> bool:
    """Model of Totals::flags bit 3 for a segment of len(data) bytes: some byte in [0, n) is NUL (the zero padding past n
    is not)."""
    return b"\0" in bytes(data)


def nul_segments(st) -> int:
    """gpugrep_stats.nul_segments (the test helpers' Stats structure calls the field `reserved`)."""
    return st.reserved


@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    assert module.cuda.is_available()
    return module


def check(lib, oracle, torch, data: bytes, patterns, flags=None, label: str = "", want_path: int = 1, expected=None) -> int:
    """Records, count-only and inverted count-only from host, pinned and device memory agree with the oracle (or
    `expected`); one segment, flagged iff the text holds a NUL."""
    if expected is None:
        rc, expected, _ = scan_bytes(oracle, data, patterns, flags=flags)
        assert rc == 0
    host = np.frombuffer(data, dtype=np.uint8)
    pinned = torch.from_numpy(host.copy()).pin_memory()
    dev, dptr = _on_device(torch, data)
    for what, ptr, loc in (("host", host.ctypes.data, HOST), ("pinned", pinned.data_ptr(), HOST), ("device", dptr, DEVICE)):
        at = f"{label} {what}"
        rc, got, st = scan_buffer(lib, ptr, len(data), loc, patterns, flags)
        assert rc == 0, at
        _same_records(got, expected, at)
        assert st.path == want_path, f"{at}: path {st.path}"
        rc, _, counted = scan_buffer(lib, ptr, len(data), loc, patterns, flags, collect=False)
        assert rc == 0 and counted.path == want_path, at
        assert counted.matches == len(expected), f"{at}: counted {counted.matches}, records {len(expected)}"
        assert counted.segments == 1 and nul_segments(counted) == k1_has_nul(data), f"{at}: nul_segments {nul_segments(counted)}"
        rc, _, _, inv = invert_scan_buffer(lib, ptr, len(data), loc, patterns, flags, collect=None)
        assert rc == 0 and inv.matches == counted.lines - len(expected), at
    del dev, pinned
    return len(expected)


def _lines_text(seed: int, size: int = 1 << 20) -> bytearray:
    return bytearray(synth.syslog_bytes(size, seed=seed))


def test_nul_free_syslog_text(gpu_lib, oracle_lib, torch):
    """configs[1] text (no NUL) with the C2 set: many matched lines, several candidate chunks per line."""
    data = bytes(_lines_text(5, 4 << 20))
    assert check(gpu_lib, oracle_lib, torch, data, synth.C2_PATTERNS, label="c2") > 1000


@pytest.mark.parametrize("where", ["matched_line_before", "matched_line_after", "unmatched_line", "first_chunk",
                                   "last_partial_chunk", "last_byte"])
def test_nul_placements(where, gpu_lib, oracle_lib, torch):
    """One NUL byte: in a matched line in front of and behind its matches (the exact re-check decides), in a line no pattern
    matches, in the first 16-byte chunk, in the last partial chunk and as the last byte before n."""
    buf = _lines_text(9)
    del buf[len(buf) - 7:]   # n % 16 != 0: the last chunk is partial
    rc, records, _ = scan_bytes(oracle_lib, bytes(buf), synth.C2_PATTERNS)
    assert rc == 0 and records
    starts = [0] + [k + 1 for k, b in enumerate(bytes(buf)) if b == 10]
    matched = {ln for _, ln, _ in records}
    m = records[len(records) // 2][1]
    u = next(k for k in range(len(starts) - 1) if k not in matched)
    at = {"matched_line_before": starts[m] + 1, "matched_line_after": starts[m + 1] - 2, "unmatched_line": (starts[u] + starts[u + 1]) // 2,
          "first_chunk": 3, "last_partial_chunk": len(buf) - 3, "last_byte": len(buf) - 1}[where]
    assert 0 < at < len(buf) and buf[at] != 10
    buf[at] = 0
    check(gpu_lib, oracle_lib, torch, bytes(buf), synth.C2_PATTERNS, label=where)


@pytest.mark.parametrize("rem", range(16))
def test_every_length_mod_16(rem, gpu_lib, oracle_lib, torch):
    """n % 16 from 0 to 15 (the zero padding past n and the device bytes after n are not text), with and without a NUL
    in the last line."""
    buf = _lines_text(20 + rem, 256 << 10)
    n = len(buf) // 16 * 16 - 16 + rem
    for nul in (False, True):
        data = bytearray(buf[:n])
        if nul:
            data[n - 1 - (rem % 3)] = 0
        check(gpu_lib, oracle_lib, torch, bytes(data), synth.C2_PATTERNS, label=f"n%16={rem} nul={nul}")


@pytest.mark.parametrize("nul", [False, True])
def test_long_lines_with_a_late_nul(nul, gpu_lib, oracle_lib, torch):
    """Matched lines of 600 B, 3 KiB and 20 KiB (past the per-thread NUL scan bound and the warp scan's 2 KiB step), each
    marked by several candidate chunks, with a NUL 5 bytes before their end; and short lines between them."""
    out = []
    for k, length in enumerate((600, 3000, 20000) * 4):
        body = bytearray(b"x%d " % k + b"Failed password for root " * (length // 25))
        if nul and k % 2 == 0:
            body[-5] = 0
        out += [bytes(body), b"port 22 ok %d" % k, b"nothing here"]
    data = b"\n".join(out) + b"\n"
    assert check(gpu_lib, oracle_lib, torch, data, synth.C2_PATTERNS, label=f"nul={nul}") >= 12


def test_c3_set_with_confirm_and_local_verification(gpu_lib, oracle_lib, torch):
    """configs[2] shape (1,000 IOC patterns: k_confirm + k_verify_local), with and without NULs in planted lines."""
    data = bytearray(synth.syslog_bytes(2 << 20, seed=11, plants=C3_PLANTS, plant_ppm=20000))
    assert check(gpu_lib, oracle_lib, torch, bytes(data), C3_PATTERNS, label="c3") > 50
    for k, plant in enumerate(C3_PLANTS[:40]):
        pos = data.find(plant.encode())
        if pos > 0:
            data[pos + (len(plant) + 2 if k % 2 else -2)] = 0   # behind the match, or in front of it
    assert check(gpu_lib, oracle_lib, torch, bytes(data), C3_PATTERNS, label="c3 nul") > 50


def test_nfa_fallback_set(gpu_lib, oracle_lib, torch):
    """NFA-fallback patterns on the fast path (k_verify_local<true>): lines with NULs re-checked with the NFA simulation."""
    import random  # pylint: disable=import-outside-toplevel

    rng = random.Random(5)
    lines = synth.syslog_bytes(1 << 20, seed=17).split(b"\n")
    out = []
    for line in lines:
        roll = rng.random()
        if roll < 0.02:
            line = line[:40] + b" session " + b"abc " * 37 + b"ab" + b"closed " + line[40:]
        elif roll < 0.03:
            line = line[:20] + b"\0session " + b"x" * 150 + b"closed"
        elif roll < 0.04:
            line = b"\0\0" + line[:30] + b" session " + b"y" * 150 + b"closed"
        out.append(line)
    check(gpu_lib, oracle_lib, torch, b"\n".join(out), NFA_PATTERNS, label="nfa")


def test_nul_flag_is_per_segment(gpu_lib, oracle_lib, torch, monkeypatch):
    """Device input cut into 8 MiB segments (and host input into 8 MiB chunks): a NUL in the second segment only flags that
    segment, and the counts of every segment stay exact."""
    buf = _lines_text(31, 40 << 20)
    nul_at = (8 << 20) + (3 << 20)
    while buf[nul_at] == 10:
        nul_at += 1
    buf[nul_at] = 0
    data = bytes(buf)
    rc, expected, _ = scan_bytes(oracle_lib, data, synth.C2_PATTERNS)
    assert rc == 0
    monkeypatch.setenv("GPUGREP_DEVICE_SEGMENT_MB", "8")
    monkeypatch.setenv("GPUGREP_CHUNK_MB", "8")
    dev, ptr = _on_device(torch, data)
    for loc, p in ((DEVICE, ptr), (HOST, np.frombuffer(data, dtype=np.uint8).ctypes.data)):
        rc, got, st = scan_buffer(gpu_lib, p, len(data), loc, synth.C2_PATTERNS)
        assert rc == 0
        _same_records(got, expected, f"loc={loc}")
        rc, _, counted = scan_buffer(gpu_lib, p, len(data), loc, synth.C2_PATTERNS, collect=False)
        assert rc == 0 and counted.matches == len(expected) and counted.path == 1
        assert counted.segments >= 5 and nul_segments(counted) == 1, (counted.segments, nul_segments(counted))
    del dev


def test_nul_in_the_second_of_three_2gib_segments(gpu_lib, oracle_lib, torch):
    """4.5 GiB of device text in the default 2 GiB segments; a rare literal planted in all three, a NUL only in the second
    (in front of one plant, behind another).  Only lines that hold the literal can match, so the oracle scans just those."""
    sample = torch.frombuffer(bytearray(synth.syslog_bytes(16 << 20, seed=3)), dtype=torch.uint8).cuda()
    size = (9 << 29) + 12345
    dev = sample.repeat(-(-size // sample.numel()))[:size].contiguous()
    dev[-1] = 10
    plant = b"kqzzplantedqk"
    planted = []
    for k, pos in enumerate([1 << 20, (1 << 30) + 77, (5 << 29) + 333, (5 << 29) + 4444, (3 << 30) + 55, (4 << 30) + 999]):
        host = dev[pos:pos + 4096].cpu().numpy().tobytes()
        s = host.find(b"\n") + 1
        e = host.find(b"\n", s)
        line = bytearray(host[s:e])
        line[5:5 + len(plant)] = plant
        if k == 3:
            line[2] = 0          # in front of the plant: the re-check drops the line
        if k == 2:
            line[-3] = 0         # behind the plant: still a match
        dev[pos + s:pos + e] = torch.frombuffer(bytearray(line), dtype=torch.uint8).cuda()
        planted.append(bytes(line))
    torch.cuda.synchronize()
    rc, expected, _ = scan_bytes(oracle_lib, b"\n".join(planted) + b"\n", [plant.decode()])
    assert rc == 0 and len(expected) == 5
    rc, got, st = scan_buffer(gpu_lib, dev.data_ptr(), size, DEVICE, [plant.decode()])
    assert rc == 0 and len(got) == 5 and st.path == 1
    rc, _, counted = scan_buffer(gpu_lib, dev.data_ptr(), size, DEVICE, [plant.decode()], collect=False)
    assert rc == 0 and counted.matches == 5 and counted.segments == 3 and nul_segments(counted) == 1
    del dev, sample
    torch.cuda.empty_cache()


@pytest.mark.parametrize("config", fpc.K1_CONFIGS, ids=[c[0] for c in fpc.K1_CONFIGS])
def test_k1_nul_flag_matches_the_model(config, gpu_lib, torch, sms):
    """The streaming-kernel inputs of test_fast_path_gpu (every instantiation, sizes around chunk, block, group and sweep
    ends, a gram of the set or a newline in the device bytes after n), with a NUL at a seeded position or none: the flag
    equals the model's.  The zero bytes past n in the device allocation never count."""
    name, pats, flags, env, inst = config
    tuned = "GPUGREP_NO_TUNE" not in env
    with fpc.environment(env):
        tables0 = K1Tables(CompiledDb(gpu_lib, pats, flags))
        exact = inst[0] == 1
        grams = _all_grams(pats, tables0.fold) if tuned else tables0.grams
        sweep = stream_sweep_bytes(K1Tables(_tuned(gpu_lib, pats, flags, b"q" * 8192)) if tuned else tables0, sms, exact)
        rng = np.random.default_rng(sum(map(ord, name)))
        for i, n in enumerate(_k1_sizes(sweep, False)):
            data = bytearray(k1_text(n, grams, seed=sum(map(ord, name)) * 100 + i))
            if i % 3:
                data[int(rng.integers(0, n)) if i % 3 == 1 else n - 1] = 0
            data = bytes(data)
            g = int(grams[i % grams.size]).to_bytes(4, "little")
            for loc, tail in ((DEVICE, b""), (DEVICE, b"\n" + g * 8), (HOST, b"")):
                keep, ptr = _on_device(torch, data, tail) if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
                rc, _, st = scan_buffer(gpu_lib, ptr, n, loc, pats, flags, collect=False)
                assert rc == 0
                assert nul_segments(st) == k1_has_nul(data), f"{name} n={n} loc={loc} tail={tail[:2]!r}"
                del keep


@pytest.fixture(scope="module")
def sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count
