"""The fast path on the GPU (k_stream -> scan -> k_list_candidates -> [k_confirm] -> k_verify_* -> k_tile_offsets -> k_emit_nlm ->
k_dedupe_records) against exact references:
  a. the candidate chunks and newlines of the streaming kernel against its CPU model (tests/k1_model.py), for every
     instantiation, at sizes around chunk, block, group and grid-sweep ends, from host, device and unaligned device memory;
  b. random factor sets on texts built to stay on the fast path, records against the oracle, under every switch;
  c. the capacity bounds and the long-line check of the fast path at their boundaries.
"""

from __future__ import annotations

import numpy as np
import pytest

import fast_path_cases as fpc
from dfa_sim import CompiledDb
from gpu_api import scan_buffer
from k1_model import K1Tables, has_newline_free_super_block, k1_candidates, stream_sweep_bytes, super_block_bytes
from oracle_api import run_scan, scan_bytes
from test_invert_match import compare_invert

pytestmark = pytest.mark.gpu

DEVICE = 1
HOST = 0


@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    assert module.cuda.is_available()
    return module


@pytest.fixture(scope="module")
def sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _on_device(torch, data: bytes, tail: bytes = b"", shift: int = 0):
    """A device allocation holding `tail` right after the data (and `shift` bytes in front of it); returns (tensor, pointer)."""
    t = torch.zeros(shift + len(data) + len(tail) + 64, dtype=torch.uint8, device="cuda")
    if data or tail:
        t[shift:shift + len(data) + len(tail)] = torch.frombuffer(bytearray(data + tail), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t, t.data_ptr() + shift


def _same_records(got, expected, label: str) -> None:
    """The records equal the oracle's; a difference is reported by its first record (pytest's own report of two long lists
    costs minutes and memory)."""
    if got != expected:
        k = next((k for k, (a, b) in enumerate(zip(got, expected)) if a != b), min(len(got), len(expected)))
        pytest.fail(f"{label}: {len(got)} records, oracle {len(expected)}; first difference at {k}: "
                    f"{got[k] if k < len(got) else None} vs {expected[k] if k < len(expected) else None}", pytrace=False)


# ---- a. K1 candidates are exact ----------------------------------------------------------------------------------------------

def _gram_bytes(g: int) -> bytes:
    return int(g).to_bytes(4, "little")


def k1_text(n: int, grams: np.ndarray, seed: int, background: np.ndarray = fpc.BACKGROUND) -> bytes:
    """Background that no gram of the set occurs in, lines of 20-300 bytes, and grams of the set planted one per 16-byte
    chunk at most: one per 512-byte block at offset 53*j + 509 (every offset mod 512 and mod 16 over 512 blocks) and one in
    the last six bytes of each block (grams that run into the next block, the next group of four, the next warp's step)."""
    r = np.random.default_rng(seed)
    buf = background[r.integers(0, background.size, n)]
    nl = np.cumsum(r.integers(20, 300, n // 20 + 2))
    buf[nl[nl < n]] = 10
    j = np.arange((n + 511) // 512, dtype=np.int64)
    at = np.concatenate([j * 512 + (53 * j + 509) % 512, j * 512 + 506 + j % 6])
    at = np.sort(at[(at + 4 <= n) & (r.random(at.size) < 0.8)])
    keep = np.ones(at.size, dtype=bool)
    keep[1:] = np.diff(at) >= 24
    at = at[keep]
    pick = grams[r.integers(0, grams.size, at.size)]
    for k in range(4):
        buf[at + k] = ((pick >> np.uint32(8 * k)) & np.uint32(0xFF)).astype(np.uint8)
    return buf.tobytes()


def _k1_sizes(sweep: int, big: bool) -> list[int]:
    sizes = [1, 15, 16, 17, 511, 512, 513, 2047, 2048, 2049, 3 * 2048 - 3, 4 * 2048 + 2, 9 * 2048 + 511, 32 * 2048 + 1, sweep - 5, sweep + 13]
    if big:
        sizes += [2 * sweep + 517, (64 << 20) + 13]
    return sizes


@pytest.mark.parametrize("config", fpc.K1_CONFIGS, ids=[c[0] for c in fpc.K1_CONFIGS])
def test_k1_candidates_and_lines_are_exact(config, gpu_lib, torch, sms):
    """stats.candidates == the model's candidate chunks and stats.lines == its newlines (+1 for a last line without one), for
    the instantiation this pattern set selects.  The bytes after n in the same device allocation are a newline or complete a
    gram of the set planted at n - 3: neither may count.  The untuned configurations run with GPUGREP_NO_TUNE (the
    database's own table); the tuned ones re-tune the model's database on the same head the scan tunes on."""
    name, pats, flags, env, inst = config
    tuned = "GPUGREP_NO_TUNE" not in env
    with fpc.environment(env):
        base = CompiledDb(gpu_lib, pats, flags)
        assert base.rc == 0
        tables0 = K1Tables(base)
        assert fpc.instantiation(tables0, env) == inst
        exact = inst[0] == 1
        # a tuned table takes the windows that are rarest in the text: plant every 4-gram of the (literal) patterns
        grams = _all_grams(pats, tables0.fold) if tuned else tables0.grams
        sweep = stream_sweep_bytes(K1Tables(_tuned(gpu_lib, pats, flags, b"q" * 8192)) if tuned else tables0, sms, exact)
        assert 4 << 20 < sweep < 32 << 20
        big = name in ("m2_s1", "m1_s2_fold", "mixed", "tuned_s4")
        for i, n in enumerate(_k1_sizes(sweep, big)):
            data = bytearray(k1_text(n, grams, seed=sum(map(ord, name)) * 100 + i))
            g = _gram_bytes(grams[i % grams.size])
            if n >= 3:
                data[n - 3:] = g[:3]
            data = bytes(data)
            tables = K1Tables(_tuned(gpu_lib, pats, flags, data[: 512 << 10])) if tuned and n >= 4096 else tables0
            newlines, chunks = k1_candidates(data, tables, exact)
            want_lines = newlines + (data[-1] != 10)
            runs = [("device, gram completed after n", DEVICE, g[3:] + b"\n" + g * 8, 0), ("device, newline after n", DEVICE, b"\n" + g * 8, 0)]
            if n < (32 << 20):
                runs += [("host", HOST, b"", 0), ("device, unaligned", DEVICE, b"\n" + g * 8, 3)]
            for what, loc, tail, shift in runs:
                if loc == HOST:
                    host = np.frombuffer(data, dtype=np.uint8)
                    rc, _, st = scan_buffer(gpu_lib, host.ctypes.data, n, HOST, pats, flags, collect=False)
                else:
                    keep, ptr = _on_device(torch, data, tail, shift)
                    rc, _, st = scan_buffer(gpu_lib, ptr, n, DEVICE, pats, flags, collect=False)
                    del keep
                assert rc == 0
                label = f"{name} n={n} {what}"
                assert st.path == 1, label
                assert st.lines == want_lines, label
                assert st.candidates == chunks.size, f"{label}: {st.candidates} candidates, model {chunks.size}"


def _all_grams(patterns, fold: bool) -> np.ndarray:
    out = {int.from_bytes(p[k:k + 4].encode(), "little") | (0x20202020 if fold else 0) for p in patterns for k in range(len(p) - 3)}
    return np.array(sorted(out), dtype=np.uint32)


def _tuned(lib, pats, flags, head: bytes) -> CompiledDb:
    db = CompiledDb(lib, pats, flags)
    db.retune(head)
    return db


# ---- b. random factor sets, records against the oracle --------------------------------------------------------------------

N_FAST_CASES = 40


@pytest.mark.parametrize("seed", range(N_FAST_CASES))
def test_random_factor_sets_match_the_oracle(seed, gpu_lib, oracle_lib, torch, tmp_path):
    """Records, return codes and batches of file, host, pinned and device input == the oracle's, for a random factor set
    (fast_path_cases.fast_case) under the default settings and one switch.  The path bits, the candidate count (K1 model),
    and - from the launch count - whether k_confirm ran must be what the engine's rules predict; a count-only scan counts the
    records; an inverted scan selects the complement."""
    case = fpc.fast_case(seed)
    data, bs = case["data"], case["buffer_size"]
    path = tmp_path / "case.log"
    path.write_bytes(data)
    rc, expected, exp_batches = run_scan(oracle_lib, str(path), case["patterns"], case["flags"], case["ids"], buffer_size=bs)
    assert rc == 0
    host = np.frombuffer(data, dtype=np.uint8)
    pinned = torch.from_numpy(host.copy()).pin_memory()
    dev = pinned.cuda()
    torch.cuda.synchronize()
    for switch in ("", case["switch"]):
        env = fpc.switch_env(switch)
        pats, flags, ids = fpc.tagged(case, switch) if switch else (case["patterns"], case["flags"], case["ids"])
        pred = fpc.predict(gpu_lib, pats, flags, ids, env, data, bs)
        label = f"seed {seed} [{switch or 'default'}] {pred.get('inst')} {pred.get('verify')}"
        with fpc.environment(env):
            rc, got, batches = run_scan(gpu_lib, str(path), pats, flags, ids, buffer_size=bs)
            assert rc == 0, label
            _same_records(got, expected, label)
            assert batches == exp_batches, label
            for what, ptr, loc in (("host", host.ctypes.data, HOST), ("pinned", pinned.data_ptr(), HOST), ("device", dev.data_ptr(), DEVICE)):
                rc, got, st = scan_buffer(gpu_lib, ptr, len(data), loc, pats, flags, ids, buffer_size=bs)
                assert rc == 0, f"{label} {what}"
                _same_records(got, expected, f"{label} {what}")
                assert st.path == pred["path"], f"{label} {what}: path {st.path}"
                if pred["fast"]:
                    _, chunks = k1_candidates(data, pred["tables"], pred["inst"][0] == 1)
                    assert st.candidates == chunks.size, f"{label} {what}"
            rc, _, st = scan_buffer(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids, collect=False, buffer_size=bs)
            assert rc == 0 and st.matches == len(expected), label
            if st.path == 1:
                assert st.segments == 1 and st.launches == 9 + pred["confirm"], f"{label}: {st.launches} launches"
            if not switch and len(data) <= (1 << 20):
                compare_invert(gpu_lib, oracle_lib, data, pats, flags, ids, buffer_size=bs, tmp_dir=str(tmp_path))


def test_ineligible_cases_take_the_general_path(gpu_lib, oracle_lib, torch):
    """An NFA pattern under GPUGREP_FILTER=exact (NFA sets need the bloom mode with its confirmation table) and a buffer_size
    below 4096 cannot use the fast path: the general path serves them, with the oracle's records."""
    data = b"".join(b"qq %d alphabet %s bravados qq\n" % (k, b"x" * (k % 170)) for k in range(3000))
    for pats, bs, env in (([r"alphabet .{150}bravados", "kilogram"], 262140, {"GPUGREP_FILTER": "exact"}), (["alphabet", "kqsmallbufkq"], 4095, {})):
        rc, expected, _ = scan_bytes(oracle_lib, data, pats, buffer_size=bs)
        pred = fpc.predict(gpu_lib, pats, None, None, env, data, bs)
        assert not pred["fast"] and expected
        dev, ptr = _on_device(torch, data)
        with fpc.environment(env):
            rc, got, st = scan_buffer(gpu_lib, ptr, len(data), DEVICE, pats, buffer_size=bs)
        assert rc == 0
        _same_records(got, expected, str(pats))
        assert st.path == 2 and st.candidates == 0
        del dev


# ---- c. boundaries ------------------------------------------------------------------------------------------------------------

CAP_PATTERN = ["ABCDEFGHIJ"]


def _capacity_text(target: int, lines: int, tables: K1Tables) -> bytes:
    """64-byte lines; a few of them match, and the 7-byte window "ABCDEFG" (which flags its chunk without matching) is
    planted at chunk starts until the model counts exactly `target` candidate chunks."""
    buf = bytearray((b"q" * 63 + b"\n") * lines)
    for k in range(0, lines, 97):
        buf[k * 64 + 20:k * 64 + 30] = b"ABCDEFGHIJ"
    _, chunks = k1_candidates(bytes(buf), tables)
    taken = set(chunks.tolist())
    free = [c for c in range(len(buf) // 16) if c * 16 % 64 != 48 and c not in taken]
    need = target - chunks.size
    assert 0 <= need <= len(free)
    for c in free[:need]:
        buf[c * 16:c * 16 + 7] = b"ABCDEFG"
    data = bytes(buf)
    assert k1_candidates(data, tables)[1].size == target
    return data


def test_candidate_capacity_boundary(gpu_lib, oracle_lib, torch):
    """Exactly cand_cap = n/32 + 4096 candidate chunks stay on the fast path; one more falls back to the general path.
    Records equal the oracle's both times."""
    with fpc.environment({"GPUGREP_NO_TUNE": "1"}):
        tables = K1Tables(CompiledDb(gpu_lib, CAP_PATTERN))
        for extra, want_path in ((0, 1), (1, 2)):
            n = 16384 * 64
            data = _capacity_text(n // 32 + 4096 + extra, 16384, tables)
            rc, expected, _ = scan_bytes(oracle_lib, data, CAP_PATTERN)
            dev, ptr = _on_device(torch, data)
            rc, got, st = scan_buffer(gpu_lib, ptr, n, DEVICE, CAP_PATTERN)
            assert rc == 0 and len(expected) > 100
            _same_records(got, expected, f"cand_cap + {extra}")
            assert st.candidates == n // 32 + 4096 + extra
            assert st.path == want_path, f"{extra}: path {st.path}"
            del dev


@pytest.mark.parametrize("nul", [False, True])
def test_one_line_over_several_emit_tiles(nul, gpu_lib, oracle_lib, torch, tmp_path):
    """One matched line whose ~1,600 candidate chunks fill several emit tiles of 512 candidates, between short matched lines:
    one record for it (the repeats across tiles are dropped), and none when a NUL in front of every match fails the exact
    re-check.  A count-only scan counts the valid records; the inverted scan is the complement."""
    long_line = b"qq" + (b"ABCDEFGHIJqqqqqq" * 1600) + b"\n"
    if nul:
        long_line = b"qq\0" + long_line[3:]
    short = b"".join(b"q%04d ABCDEFGHIJ\n" % k for k in range(40))
    data = short + b"qqq\n" * 7 + long_line + short + long_line[:-1] + b"tail\n" + short
    rc, expected, _ = scan_bytes(oracle_lib, data, CAP_PATTERN)
    assert len(expected) == 120 + (0 if nul else 2)
    for loc in (HOST, DEVICE):
        keep, ptr = _on_device(torch, data) if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
        rc, got, st = scan_buffer(gpu_lib, ptr, len(data), loc, CAP_PATTERN)
        assert rc == 0
        _same_records(got, expected, f"nul={nul} loc={loc}")
        assert st.path == 1 and st.candidates > 3200
        rc, _, st = scan_buffer(gpu_lib, ptr, len(data), loc, CAP_PATTERN, collect=False)
        assert rc == 0 and st.matches == len(expected)
        del keep
    compare_invert(gpu_lib, oracle_lib, data, CAP_PATTERN, tmp_dir=str(tmp_path))


@pytest.mark.parametrize("buffer_size", [4096, 8192, 16384, 65536, 262140])
def test_long_lines_around_the_super_block_size(buffer_size, gpu_lib, oracle_lib, torch):
    """Lines of super - 1, super and 2 * super - 1 bytes and of buffer_size - 2 .. buffer_size bytes, at several alignments,
    with matches near their start, middle and end, between short matched lines.  A segment with an aligned newline-free
    super-block takes the general path; every other one stays on the fast path (which never splits a line into pseudo-lines:
    that is what the check protects).  Host and device input; records == the oracle's."""
    s = super_block_bytes(buffer_size)
    for length in (s - 1, s, 2 * s - 1, buffer_size - 2, buffer_size - 1, buffer_size):
        for lead in (0, 7, 1000):
            body = bytearray(b"q" * length)
            for at in (3, length // 2, length - 12):
                body[at:at + 10] = b"ABCDEFGHIJ"
            data = b"q" * lead + b"\n" + b"ABCDEFGHIJ 1\n" * 5 + bytes(body) + b"\nABCDEFGHIJ 2\nqq\n"
            rc, expected, _ = scan_bytes(oracle_lib, data, CAP_PATTERN, buffer_size=buffer_size)
            want_path = 2 if has_newline_free_super_block(data, s) else 1
            for loc in (HOST, DEVICE):
                keep, ptr = _on_device(torch, data) if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
                rc, got, st = scan_buffer(gpu_lib, ptr, len(data), loc, CAP_PATTERN, buffer_size=buffer_size)
                label = f"bs={buffer_size} line={length} lead={lead} loc={loc}"
                assert rc == 0, label
                _same_records(got, expected, label)
                assert st.path == want_path, f"{label}: path {st.path}"
                del keep


def test_record_capacity_boundary(gpu_lib, oracle_lib, torch):
    """Short matched lines whose record count crosses rec_cap = n/48 + 4096 (the fast path falls back above it): records ==
    the oracle's on both sides, and the sweep really crosses the bound."""
    paths = set()
    for lines in (4000, 4600, 5000, 5400, 6000, 8000):
        data = b"ABCDEFGHIJ\n" * lines
        rc, expected, _ = scan_bytes(oracle_lib, data, CAP_PATTERN)
        dev, ptr = _on_device(torch, data)
        rc, got, st = scan_buffer(gpu_lib, ptr, len(data), DEVICE, CAP_PATTERN)
        assert rc == 0 and len(expected) == lines
        _same_records(got, expected, f"{lines} lines")
        rc, _, counted = scan_buffer(gpu_lib, ptr, len(data), DEVICE, CAP_PATTERN, collect=False)
        assert rc == 0 and counted.matches == lines
        paths.add(st.path)
        del dev
    assert paths == {1, 2}, paths
