"""Every scan path over the whole byte alphabet (tests/byte_cases.py): high bytes, control bytes, every escape form, POSIX
classes and the non-letters whose bit-5 partner is another byte, against the oracle.

The device code works on bytes arithmetically: the streaming kernel folds every byte with 0x20 under FOLD, the newline
count and the NUL flag are SWAR tests whose top-bit terms are exact only for bytes >= 0x80, the verification walks index
byte tables and a 255-entry class map, the NFA splits bytes into word / other.  A bug that shows only on bytes >= 0x80 or on
a bit-5 pair that is not a letter pair would pass every test whose text is ASCII.

CPU tests: the compiled tables (tests/dfa_sim.py) and the host logic (mock engine) against the oracle, accept/reject of
the escape forms, the fast-path model.  GPU tests (`-m gpu`): random cases on both paths and on the NFA, factor sets on
the fast path from every kind of input, the streaming kernel's candidates / lines / NUL flag on high-byte text, the
boundary of the shared-memory class table, and NFA patterns of up to 4096 positions.
"""

from __future__ import annotations

import random

import numpy as np
import pytest

import byte_cases as bc
import fast_path_cases as fpc
import parity
from dfa_sim import CompiledDb, fast_path_matched_line_starts, split_pseudo_lines
from gpu_api import scan_buffer
from k1_model import K1Tables, k1_candidates, stream_sweep_bytes
from oracle_api import check, run_scan, scan_bytes
from test_context_lines import compare_context
from test_count_only_gpu import k1_has_nul, nul_segments
from test_fast_path_gpu import _k1_sizes, _on_device, _same_records, k1_text
from test_invert_match import compare_invert

HOST, DEVICE = 0, 1
N_RANDOM = 150
N_FAST = 40


@pytest.fixture(scope="module")
def torch():
    import torch as module  # pylint: disable=import-outside-toplevel

    assert module.cuda.is_available()
    return module


@pytest.fixture(scope="module")
def sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- CPU: the compiler against the oracle ------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(N_RANDOM))
def test_tables_match_oracle(seed, gpu_lib, oracle_lib):
    """The DFA tables, walked by dfa_sim, give the oracle's per-line reports; the prefilter is a superset filter."""
    patterns, flags, ids, buffer_size, data, _, _ = bc.byte_random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    db = CompiledDb(gpu_lib, patterns, flags, ids)
    assert (db.rc == 0) == (check(oracle_lib, patterns, flags, ids) == 0), (patterns, db.error)
    if db.rc:
        return
    _, got, _ = scan_bytes(oracle_lib, data, patterns, flags=flags, ids=ids, buffer_size=buffer_size)
    expected = [(i, ln) for (i, ln, _line) in got]
    mine = []
    for ln, pl in enumerate(split_pseudo_lines(data, buffer_size)):
        reports = db.line_reports(pl)
        mine += [(rid, ln) for rid in reports]
        assert not reports or db.prefilter_hits(db.block_of(pl)), "prefilter must be a superset filter"
    assert mine == expected, patterns


ESCAPES_ACCEPTED = [rb"\xff", rb"\x{ff}", rb"\x{0ff}", rb"\x{C9}", rb"\x", rb"\x7", rb"\xzz", rb"\o{377}", rb"\o{0}", rb"\0", rb"\012", rb"\0129",
                    rb"\08", rb"\ca", rb"\cA", rb"\c ", rb"\c~", rb"\c{", rb"\c\xe9", rb"\e\a\f\r\t", rb"\h\H\v\V\N\W\S\D", rb"\N{2}", rb"a\N{0}b",
                    rb"[\h]", rb"[\v]", rb"[\e]", rb"[\b]x", rb"[\cA]", rb"[\7]", rb"[\18]", rb"[\8]", rb"[\9a]", rb"[\80]", rb"[\08]",
                    rb"[\0-\x7f]", rb"[^\x00-\x7f]", rb"[\x7e-\x81]", rb"[@-\x60]", rb"[Z-a]", rb"[\xc0-\xdf]", rb"[%-\x{ff}]", rb"[\e-z]",
                    rb"[\d-]", rb"[-\d]", rb"[\d\-z]", rb"[[:digit:]-]", rb"[%--]", rb"[[:^ascii:]]", rb"[[:punct:]]", rb"[[:cntrl:]]x",
                    rb"[[:print:]]", rb"[[:graph:]]", rb"[[:xdigit:]]", rb"[[:word:]]", rb"[[:^print:]]", b"\xe9", b"\xc3\xa9", b"[\xe9-\xff]",
                    rb"(?i)\xc9", rb"(?i)[@]", rb"\_", rb"\@", b"\\Q\xe9\\E", rb"[\Q]\E]", rb"(?x)a # \xe9"]
ESCAPES_REJECTED = [rb"\x{100}", rb"\x{}", rb"\o{400}", rb"\o{7777}", rb"\o{}", rb"\o", b"\\c\xe9", rb"\c", rb"\c\\", rb"[\c]", b"\\c\t", b"\\c\x7f",
                    b"\\c\x1f", rb"\N{U+41}", rb"\N{x}", rb"\N{", rb"[\N]", rb"\8", rb"[a-\d]", rb"[\d-z]", rb"[\h-a]", rb"[a-\h]", rb"[\w-\]]",
                    rb"[a-\e]", rb"[[:digit:]-z]", rb"[a-[:digit:]]", b"[\xff-\xe9]", rb"[z-a]", rb"[[:foo:]]", rb"[[.a.]]", rb"[[=a=]]",
                    rb"\u0041", rb"\U", rb"\L", rb"\l", rb"\y", b"a\\"]


def test_escape_forms_accept_reject(gpu_lib, oracle_lib):
    """Accept/reject of every escape form, with the code-point limits of a byte engine (no UTF mode), against check()."""
    for pattern in ESCAPES_ACCEPTED:
        assert check(oracle_lib, [pattern]) == 0, pattern
        assert CompiledDb(gpu_lib, [pattern]).rc == 0, pattern
    for pattern in ESCAPES_REJECTED:
        assert check(oracle_lib, [pattern]) == 4, pattern
        assert CompiledDb(gpu_lib, [pattern]).rc == 4, pattern


def _reports(lib, pattern: bytes, lines: list[bytes]) -> list[bool]:
    db = CompiledDb(lib, [pattern])
    assert db.rc == 0, pattern
    return [bool(db.line_reports(line)) for line in lines]


def _oracle_reports(oracle, pattern: bytes, lines: list[bytes]) -> list[bool]:
    _, got, _ = scan_bytes(oracle, b"".join(lines), [pattern])
    hit = {ln for _, ln, _ in got}
    return [k in hit for k in range(len(lines))]


def test_digit_8_and_9_in_a_class_are_the_digits(gpu_lib, oracle_lib):
    """Regression: `[\\8]` and `[\\9]` were rejected; PCRE2 reads the digits themselves inside a class (outside one they are
    back-references, rejected by both)."""
    lines = [b"8x\n", b"9x\n", b"\x08x\n", b"\x38x\n", b"ax\n", b"x\n"]
    for pattern in (rb"[\8]x", rb"[\9a]x", rb"[\80]x"):
        assert _reports(gpu_lib, pattern, lines) == _oracle_reports(oracle_lib, pattern, lines), pattern


def test_c_escape_needs_a_printable_character(gpu_lib, oracle_lib):
    """Regression: `\\c` followed by a tab, 0x7F or another control character was accepted; PCRE2 rejects it (\\c must be
    followed by a printable ASCII character).  The printable ones map to X ^ 0x40."""
    for x in list(range(0, 32)) + [127]:
        if x in (0, 10):
            continue
        pattern = b"\\c" + bytes([x])
        assert check(oracle_lib, [pattern]) == 4 and CompiledDb(gpu_lib, [pattern]).rc == 4, pattern
    lines = [bytes([b]) + b"\n" for b in range(1, 128) if b != 10]
    for x in b" ~{?@`[_z":
        pattern = b"\\c" + bytes([x]) + b"|\\x{41}\\c" + bytes([x])
        assert _reports(gpu_lib, pattern, lines) == _oracle_reports(oracle_lib, pattern, lines), pattern


def test_class_escapes_bound_no_range(gpu_lib, oracle_lib):
    """Regression: `[a-\\d]`, `[\\d-z]`, `[a-[:digit:]]` and `[[:digit:]-z]` were read with a literal '-'; PCRE2 rejects them
    ("invalid range in character class").  A '-' last in the class or after a single-byte escape stays legal."""
    for pattern in (rb"[a-\d]", rb"[\d-z]", rb"[a-\h]", rb"[a-[:digit:]]", rb"[[:digit:]-z]"):
        assert CompiledDb(gpu_lib, [pattern]).rc == 4 and check(oracle_lib, [pattern]) == 4, pattern
    lines = [bytes([b]) + b"q\n" for b in range(1, 256) if b != 10]
    for pattern in (rb"[\d-]q", rb"[[:digit:]-]q", rb"[\e-z]q", rb"[\x7e-\x81-]q", rb"[a-\x{ff}]q"):
        assert _reports(gpu_lib, pattern, lines) == _oracle_reports(oracle_lib, pattern, lines), pattern


def test_n_escape_with_a_brace(gpu_lib, oracle_lib):
    """Regression: `\\N{U+41}` was read as \\N followed by literal text; without UTF mode PCRE2 rejects it, and a '{' after
    \\N must open a quantifier."""
    lines = [b"ab\n", b"a\xffb\n", b"a\xff\x80b\n", b"a\nb", b"a\x00b\n"]
    for pattern in (rb"a\N{1}b", rb"a\N{1,2}b", rb"a\N{0}b"):
        assert _reports(gpu_lib, pattern, lines) == _oracle_reports(oracle_lib, pattern, lines), pattern


def _plant_lines(rng: random.Random, pieces: list[bytes], caseless: bool) -> bytes:
    lines = []
    for _ in range(40):
        text = bc.byte_text(rng, 1, max_len=50).rstrip(b"\n")
        if rng.random() < 0.6:
            piece = rng.choice(pieces)
            if caseless:
                piece = bc.flip_case(piece, rng)
                piece = (bc.flip_bit5(piece, rng) or piece) if rng.random() < 0.4 else piece
            at = rng.randint(0, len(text))
            text = text[:at] + piece + text[at:]
        if rng.random() < 0.1:
            at = rng.randint(0, len(text))
            text = text[:at] + b"\0" + text[at:]
        lines.append(text)
    return b"\n".join(lines) + (b"\n" if rng.random() < 0.7 else b"")


@pytest.mark.parametrize("seed", range(60))
def test_fast_path_model_is_exact(seed, gpu_lib):
    """The fast-path algorithm modelled on the CPU (gram hits, local walk with look-back, mid-line entry states, NUL
    re-check) finds exactly the lines the full walk finds, on byte texts with UTF-8 and punctuation factors, bit-5 near
    misses included."""
    rng = random.Random(seed)
    k = rng.choice([1, 2, 4])
    made = [bc.byte_factor_pattern(rng) for _ in range(k)]
    caseless = rng.random() < 0.5
    db = CompiledDb(gpu_lib, [p for p, _ in made], [15 if caseless else rng.choice([14, 10])] * k, [0] * k)
    assert db.rc == 0, db.error
    if not db.info.prefilter:
        pytest.skip("no usable factor")
    data = _plant_lines(rng, [pc for _, pcs in made for pc in pcs], caseless)
    if parity.has_all_nul_pseudo_line(data, 262140):
        pytest.skip("all-NUL pseudo-line")
    if rng.random() < 0.5:
        db.retune(data[: max(8, len(data) // 2)])
    truth, pos = set(), 0
    for pl in split_pseudo_lines(data, 262140):
        if db.line_reports(pl):
            truth.add(pos)
        pos += len(pl)
    assert fast_path_matched_line_starts(db, data) == truth


@pytest.mark.parametrize("budget", ["", "3"])
@pytest.mark.parametrize("seed", range(60))
def test_host_logic_matches_oracle(seed, budget, hostmock_lib, oracle_lib, monkeypatch):
    """Host logic (segments, batches, limits) and the compiler on the mock engine, at the default DFA budget and with every
    pattern on the NFA (GPUGREP_MAX_DFA_STATES=3)."""
    if budget:
        monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", budget)
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = bc.byte_random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    parity.compare(hostmock_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match)


# ---- the shared-memory class table: 253 and 254 byte classes ------------------------------------------------------------------

def class_table_set(classes: int) -> list[bytes]:
    """One-group pattern sets whose DFA has `classes` byte classes: eight patterns `kqjw<k>xy[S_k]zz` in which S_k holds the
    bytes of a subset U whose index has bit k set, so that every byte of U has a column of its own (a few states, far under
    the shared-memory budget).  The size of U is searched once per library; see test_class_table_boundary_sets."""
    chosen = [b for b in range(1, 256) if b not in b"\nkqjwxyz01234567"]
    return [b"kqjw%dxy[" % k + b"".join(b"\\x%02x" % b for j, b in enumerate(chosen[:classes]) if (j + 1) >> k & 1) + b"]zz" for k in range(8)]


def _class_count(lib, size: int) -> tuple[int, int]:
    db = CompiledDb(lib, class_table_set(size))
    assert db.rc == 0 and db.info.groups == 1
    return db.groups[0][0].classes, db.groups[0][0].states


def class_table_sizes(lib) -> dict:
    """{253: |U|, 254: |U|}: the subset sizes that give exactly 253 and 254 classes (ncls = classes + 2 = 255 and 256)."""
    out = {}
    for size in range(225, 245):
        classes, _ = _class_count(lib, size)
        if classes in (253, 254):
            out.setdefault(classes, size)
    return out


def class_table_text(seed: int) -> bytes:
    """Every byte in every position of the lines, and the patterns' words with each byte after their class."""
    rng = random.Random(seed)
    lines = []
    for k in range(8):
        for b in range(1, 256):
            if b == 10:
                continue
            lines.append(b"kqjw%dxy" % k + bytes([b]) + b"zz" + bytes(rng.randrange(1, 256) for _ in range(rng.randint(0, 12))).replace(b"\n", b"\x8a"))
    body = bytes(b for b in range(1, 256) if b != 10)
    lines += [body, body[::-1], body[7:] + body[:7]]
    rng.shuffle(lines)
    return b"\n".join(lines) + b"\n"


def test_class_table_boundary_sets(gpu_lib):
    """The sets exist: one group, 253 and 254 classes, few states; predict serves the first with k_verify_smem and the
    second with k_verify_local."""
    sizes = class_table_sizes(gpu_lib)
    assert set(sizes) == {253, 254}, sizes
    data = class_table_text(1)
    for classes, want in ((253, "smem"), (254, "local")):
        got, states = _class_count(gpu_lib, sizes[classes])
        assert got == classes and states < 100
        pred = fpc.predict(gpu_lib, class_table_set(sizes[classes]), None, None, {"GPUGREP_NO_TUNE": "1"}, data, 262140)
        assert pred["fast"] and pred["path"] == 1 and pred["verify"] == want, (classes, pred.get("verify"))


# ---- wide NFA patterns -------------------------------------------------------------------------------------------------------
NFA_POSITIONS = [31, 32, 33, 64, 65, 1000, 4096]


def wide_nfa_literal(positions: int, seed: int) -> tuple[bytes, bytes]:
    """(pattern, one text it matches): `positions` single-byte items, mostly high bytes written as escapes, every 7th a
    small class; no repeat keeps many positions active at once."""
    rng = random.Random(seed)
    pattern, text = [], bytearray()
    for k in range(positions):
        if k % 7 == 3:
            pattern.append(rb"[\xc0-\xdf]")
            text.append(rng.randrange(0xC0, 0xE0))
        else:
            b = rng.choice([0x80, 0x85, 0xA0, 0xC9, 0xE9, 0xFF, 0x8A, 0x81, ord("@"), ord("`"), ord("q")])
            pattern.append(bc.escaped(b, rng))
            text.append(b)
    return b"".join(pattern), bytes(text)


def wide_nfa_text(pattern_text: bytes, seed: int, prefix: bytes = b"") -> bytes:
    """Lines of high bytes with planted matches and one-byte-off near misses (a byte changed in bit 5, or the last byte
    dropped)."""
    rng = random.Random(seed)
    lines = []
    for k in range(60):
        filler = bytes(rng.choice(bc.K1_BACKGROUND.tolist()) for _ in range(rng.randint(0, 40)))
        roll = k % 4
        if roll == 0:
            body = prefix + pattern_text
        elif roll == 1:
            at = rng.randrange(len(pattern_text))
            body = prefix + pattern_text[:at] + bytes([pattern_text[at] ^ 0x20]) + pattern_text[at + 1:]
        elif roll == 2:
            body = prefix + pattern_text[:-1]
        else:
            body = b""
        lines.append(filler + body + filler[::-1])
    return b"\n".join(lines) + b"\n"


def test_nfa_position_limit_on_the_cpu(gpu_lib, oracle_lib, monkeypatch):
    """With the DFA budget at 3 states every wide pattern is an NFA of exactly its item count; 4097 positions exceed the
    simulation's limit (DESIGN.md §2) and are rejected with 4."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "3")
    for positions in NFA_POSITIONS:
        pattern, _ = wide_nfa_literal(positions, positions)
        db = CompiledDb(gpu_lib, [pattern])
        assert db.rc == 0 and db.info.groups == 0, (positions, db.error)
        assert check(oracle_lib, [pattern]) == 0
    pattern, _ = wide_nfa_literal(4097, 4097)
    assert CompiledDb(gpu_lib, [pattern]).rc == 4


# ---- coverage of the byte-alphabet cases -----------------------------------------------------------------------------------

def coverage(lib) -> dict:
    """What the byte-alphabet GPU cases reach, from the engine's launch rules (fast_path_cases.predict) on the compiled
    tables: k_stream instantiations, k_confirm with and without extended confirmation, the verification kernels, the
    general path and the NFA word counts."""
    reached = {"k_stream": set(), "random k_stream": set(), "verify": set(), "k_confirm": set(), "general path": 0, "nfa words": set()}
    for name, pats, flags, env, inst in bc.K1_BYTE_CONFIGS:
        with fpc.environment(env):
            got = fpc.instantiation(K1Tables(CompiledDb(lib, pats, flags)), env)
        assert got == inst, (name, got)
        reached["k_stream"].add(got)
    for seed in range(N_FAST):
        case = bc.byte_fast_case(seed)
        for switch in ("", case["switch"]):
            pats, flags, ids = fpc.tagged(case, switch) if switch else (case["patterns"], case["flags"], case["ids"])
            env = fpc.switch_env(switch)
            p = fpc.predict(lib, pats, flags, ids, env, case["data"], case["buffer_size"])
            if not p["fast"]:
                reached["general path"] += 1
                continue
            reached["k_stream"].add(p["inst"])
            reached["random k_stream"].add(p["inst"])
            reached["verify"].add(p["verify"])
            if p["confirm"]:
                ext = "grams with extended confirmation" in p["db"].prefilter_note and env.get("GPUGREP_NO_EXT_CONFIRM") != "1"
                reached["k_confirm"].add("extended" if ext else "plain")
    sizes = class_table_sizes(lib)
    for classes in (253, 254):
        p = fpc.predict(lib, class_table_set(sizes[classes]), None, None, {"GPUGREP_NO_TUNE": "1"}, class_table_text(1), 262140)
        reached["verify"].add(p["verify"])
    for seed in range(N_RANDOM):
        patterns, flags, ids, buffer_size, data, _, _ = bc.byte_random_case(seed)
        db = CompiledDb(lib, patterns, flags, ids)
        if db.rc == 0 and not (db.info.simple and db.info.prefilter and buffer_size >= 4096):
            reached["general path"] += 1
    reached["nfa words"] = {(p + 31) // 32 for p in NFA_POSITIONS}
    return reached


def test_byte_cases_cover_every_kernel(gpu_lib):
    """Every k_stream instantiation (the folded ones included), k_confirm with extended confirmation, k_verify_smem,
    k_verify_local plain and WITH_NFA, the general path and NFA patterns of 1, 2, 3, 32 and 128 words are reached by some
    byte-alphabet case.  Prints the coverage table."""
    reached = coverage(gpu_lib)
    print("\nbyte-alphabet coverage")
    for (mode, stride, fold, odd) in sorted(fpc.ALL_INSTANTIATIONS):
        print(f"  k_stream MODE={mode} STRIDE={stride} FOLD={int(fold)} NODD={odd}: {'yes' if (mode, stride, fold, odd) in reached['k_stream'] else 'no'}")
    print(f"  k_confirm: {sorted(reached['k_confirm'])}")
    print(f"  verification: {sorted(reached['verify'])}")
    print(f"  general path: {reached['general path']} cases")
    print(f"  NFA words: {sorted(reached['nfa words'])}")
    assert reached["k_stream"] == fpc.ALL_INSTANTIATIONS, sorted(fpc.ALL_INSTANTIATIONS - reached["k_stream"])
    folded_by_random_cases = {p for p in reached["random k_stream"] if p[2]}
    assert folded_by_random_cases == {i for i in fpc.ALL_INSTANTIATIONS if i[2]}, sorted(folded_by_random_cases)
    assert "extended" in reached["k_confirm"]
    assert {"smem", "local"} <= reached["verify"] and any(v.startswith("local_nfa") for v in reached["verify"]), reached["verify"]
    assert reached["general path"] >= 50
    assert {1, 2, 3, 32, 128} <= reached["nfa words"]


def test_byte_fast_cases_stay_on_the_fast_path(gpu_lib):
    """Most byte factor sets are served by the fast path (a case that drifted to the general path would test nothing new)."""
    fast = 0
    for seed in range(N_FAST):
        case = bc.byte_fast_case(seed)
        p = fpc.predict(gpu_lib, case["patterns"], case["flags"], case["ids"], {}, case["data"], case["buffer_size"])
        fast += p["fast"] and p["path"] == 1
    assert fast >= 0.8 * N_FAST, fast


# ---- GPU ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("force_general", [False, True])
@pytest.mark.parametrize("seed", range(N_RANDOM))
def test_gpu_random_cases_match_oracle(seed, force_general, gpu_lib, oracle_lib, monkeypatch):
    if force_general:
        monkeypatch.setenv("GPUGREP_FORCE_GENERAL", "1")
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = bc.byte_random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    parity.compare(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(500, 540))
def test_gpu_nfa_random_cases_match_oracle(seed, gpu_lib, oracle_lib, monkeypatch):
    """Every pattern on the bit-parallel NFA (GPUGREP_MAX_DFA_STATES=3): reach rows of high bytes, word/other kinds."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "3")
    patterns, flags, ids, buffer_size, data, buffer_count, max_match = bc.byte_random_case(seed)
    if parity.has_all_nul_pseudo_line(data, buffer_size):
        pytest.skip("all-NUL pseudo-line")
    parity.compare(gpu_lib, oracle_lib, data, patterns, flags, ids, buffer_size, buffer_count, max_match)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(N_FAST))
def test_gpu_byte_factor_sets_match_the_oracle(seed, gpu_lib, oracle_lib, torch, tmp_path):
    """Records, return codes and batches of file, host, pinned and device input == the oracle's; path and candidate count
    (which pins the k_stream instantiation) == the model's; count-only counts the records; the inverted scan and -B2 -A3
    agree with the oracle."""
    case = bc.byte_fast_case(seed)
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
                    assert st.candidates == chunks.size, f"{label} {what}: {st.candidates} candidates, model {chunks.size}"
            rc, _, st = scan_buffer(gpu_lib, dev.data_ptr(), len(data), DEVICE, pats, flags, ids, collect=False, buffer_size=bs)
            assert rc == 0 and st.matches == len(expected), label
            if st.path == 1:
                assert st.segments == 1 and st.launches == 9 + pred["confirm"], f"{label}: {st.launches} launches"
            if not switch:
                small = data[: data.rfind(b"\n", 0, 1 << 19) + 1] if len(data) > (1 << 19) else data
                compare_invert(gpu_lib, oracle_lib, small, pats, flags, ids, buffer_size=bs, tmp_dir=str(tmp_path))
                compare_context(gpu_lib, oracle_lib, small, pats, flags, ids, buffer_size=bs, before=2, after=3, tmp_dir=str(tmp_path))


@pytest.mark.gpu
@pytest.mark.parametrize("config", bc.K1_BYTE_CONFIGS, ids=[c[0] for c in bc.K1_BYTE_CONFIGS])
def test_gpu_k1_folded_high_byte_grams(config, gpu_lib, torch, sms):
    """The streaming kernel's candidates, lines and NUL flag == the model's for the folded configurations, on a background of
    high bytes and bit-5 partners with the grams planted once as they are and once with their non-letters' bit 5 cleared
    (0xC9 for 0xE9, '@' for '`'): hits only because every byte is folded.  Sizes around chunk, block, group and sweep ends;
    a NUL at a seeded place, at the end, or none."""
    name, pats, flags, env, inst = config
    with fpc.environment(env):
        tables = K1Tables(CompiledDb(gpu_lib, pats, flags))
        assert fpc.instantiation(tables, env) == inst
        exact = inst[0] == 1
        grams = bc.bit5_variants(tables.grams, sum(map(ord, name)))
        sweep = stream_sweep_bytes(tables, sms, exact)
        rng = np.random.default_rng(sum(map(ord, name)))
        for i, n in enumerate(_k1_sizes(sweep, False)):
            data = bytearray(k1_text(n, grams, seed=sum(map(ord, name)) * 100 + i, background=bc.K1_BACKGROUND))
            if i % 3:
                data[int(rng.integers(0, n)) if i % 3 == 1 else n - 1] = 0
            data = bytes(data)
            newlines, chunks = k1_candidates(data, tables, exact)
            want_lines = newlines + (data[-1] != 10)
            for what, loc in (("device", DEVICE), ("host", HOST)):
                keep, ptr = _on_device(torch, data, b"\x8a" + data[:8]) if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
                rc, _, st = scan_buffer(gpu_lib, ptr, n, loc, pats, flags, collect=False)
                label = f"{name} n={n} {what}"
                assert rc == 0 and st.path == 1, label
                assert st.lines == want_lines, f"{label}: {st.lines} lines, model {want_lines}"
                assert st.candidates == chunks.size, f"{label}: {st.candidates} candidates, model {chunks.size}"
                assert nul_segments(st) == k1_has_nul(data), f"{label}: nul_segments {nul_segments(st)}"
                del keep


@pytest.mark.gpu
def test_gpu_swar_near_misses_are_neither_newlines_nor_nuls(gpu_lib, oracle_lib, torch):
    """A NUL-free text dense in 0x80, 0x81 and 0x8A: no NUL flag, the exact line count, the oracle's records and count."""
    pats = [rb"\x8a\x0a|\x81\x80\x8a", "kqnearmissqk"]
    for n in (4096 + 5, 1 << 20, (8 << 20) + 3):
        data = bc.swar_near_miss_text(n, n)
        rc, expected, _ = scan_bytes(oracle_lib, data, pats)
        assert rc == 0 and expected
        for loc in (DEVICE, HOST):
            keep, ptr = _on_device(torch, data, b"\x8a\x80") if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
            rc, _, st = scan_buffer(gpu_lib, ptr, n, loc, pats, collect=False)
            assert rc == 0 and nul_segments(st) == 0, (n, loc)
            assert st.lines == data.count(b"\n") + (data[-1] != 10), (n, loc, st.lines)
            assert st.matches == len(expected), (n, loc)
            rc, got, _ = scan_buffer(gpu_lib, ptr, n, loc, pats)
            _same_records(got, expected, f"n={n} loc={loc}")
            del keep


@pytest.mark.gpu
@pytest.mark.parametrize("classes,verify", [(253, "smem"), (254, "local")])
def test_gpu_class_table_boundary(classes, verify, gpu_lib, oracle_lib, torch, tmp_path):
    """253 classes (ncls 255) are served by k_verify_smem, 254 (ncls 256, one more than the 8-bit class map holds) by
    k_verify_local: both give the oracle's records on text that uses every byte, on the fast and the general path."""
    size = class_table_sizes(gpu_lib)[classes]
    pats = class_table_set(size)
    data = class_table_text(classes)
    env = {"GPUGREP_NO_TUNE": "1"}
    pred = fpc.predict(gpu_lib, pats, None, None, env, data, 262140)
    assert pred["verify"] == verify and pred["path"] == 1
    rc, expected, _ = scan_bytes(oracle_lib, data, pats)
    assert rc == 0 and len(expected) > 8 * 100
    with fpc.environment(env):
        for loc in (DEVICE, HOST):
            keep, ptr = _on_device(torch, data) if loc == DEVICE else (None, np.frombuffer(data, dtype=np.uint8).ctypes.data)
            rc, got, st = scan_buffer(gpu_lib, ptr, len(data), loc, pats)
            assert rc == 0 and st.path == 1
            _same_records(got, expected, f"{classes} classes loc={loc}")
            del keep
        parity.compare(gpu_lib, oracle_lib, data, pats, buffer_size=64)
        compare_invert(gpu_lib, oracle_lib, data, pats, tmp_dir=str(tmp_path))


@pytest.mark.gpu
@pytest.mark.parametrize("positions", NFA_POSITIONS)
def test_gpu_wide_nfa_patterns(positions, gpu_lib, oracle_lib, torch, monkeypatch):
    """NFA patterns of 31 .. 4096 positions (1 .. 128 words) with planted matches and one-byte-off near misses in byte text:
    both paths at the default buffer_size, the general path at buffer_size 2048, and the fast path with NFA verification
    when a literal factor leads the pattern."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "3")
    for prefix in (b"", b"kq\xe9factor"):   # the literal prefix is part of the position count
        pattern, text = wide_nfa_literal(positions - len(prefix), positions)
        pats = [prefix + pattern, b"kqwidenfaqk"] if prefix else [pattern]
        data = wide_nfa_text(text, positions, prefix)
        matched = parity.compare(gpu_lib, oracle_lib, data, pats)
        assert matched >= 15   # the planted matches (a dropped last byte can be supplied by the filler behind it)
        assert parity.compare(gpu_lib, oracle_lib, data, pats, buffer_size=2048) == (matched if positions < 2000 else 0)
        if prefix:
            pred = fpc.predict(gpu_lib, pats, None, None, {}, data, 262140)
            assert pred["fast"] and pred["nfa"] >= 1 and pred["verify"].startswith("local_nfa"), pred.get("verify")
            dev, ptr = _on_device(torch, data)
            rc, got, st = scan_buffer(gpu_lib, ptr, len(data), DEVICE, pats)
            assert rc == 0 and st.path == pred["path"] and len(got) == matched
            del dev


@pytest.mark.gpu
def test_gpu_nfa_position_limit(gpu_lib, oracle_lib, tmp_path, monkeypatch):
    """4097 positions: 4 from check_patterns and from hyperscan (DESIGN.md §2), on the GPU build."""
    monkeypatch.setenv("GPUGREP_MAX_DFA_STATES", "3")
    pattern, text = wide_nfa_literal(4097, 4097)
    assert check(gpu_lib, [pattern]) == 4
    path = tmp_path / "t.log"
    path.write_bytes(text + b"\n")
    rc, got, _ = run_scan(gpu_lib, str(path), [pattern])
    assert rc == 4 and got == []
