"""Inputs for the match-event tests (tests/test_match_events_gpu.py, and a CPU subset in tests/test_match_events_cpu.py):
random general-mode cases - several ids, SINGLEMATCH mixed with patterns that report every end - and pattern sets that
compile to an exact number of DFA groups, with the oracle's match ends to compare with (oracle_ends_buffer).
"""

from __future__ import annotations

import ctypes
import random

import numpy as np

import byte_cases
import fast_path_cases as fpc
from dfa_sim import CompiledDb
from oracle_api import check
from regex_gen import gen_regex

BUFFER_SIZES = [262140, 4096, 257, 64, 9]
BUFFER_COUNTS = [1, 7, 16]
CASELESS, SINGLEMATCH = 1, 8


class MatchEnd(ctypes.Structure):
    """gpugrep_match_end (include/gpugrep.h); oracle_ends_buffer writes the same layout."""

    _fields_ = [("line_number", ctypes.c_ulonglong), ("id", ctypes.c_uint), ("end", ctypes.c_uint)]


def _marshal(patterns, flags, ids):
    n = len(patterns)
    pa = (ctypes.c_char_p * n)(*[p if isinstance(p, bytes) else p.encode("latin1") for p in patterns])
    return pa, (ctypes.c_uint * n)(*flags), (ctypes.c_uint * n)(*ids), n


def ends_entry(lib, name: str = "gpugrep_match_ends"):
    entry = getattr(lib, name)
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                      ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
    return entry


def match_ends(lib, ptr: int, size: int, location: int, patterns, flags, ids, buffer_size: int, capacity: int | None = None,
               stats=None):
    """gpugrep_match_ends -> (rc, [(line, id, end)] of the stored records, count found).  capacity None: room for all
    (a first call with out = NULL counts them)."""
    pa, fa, ia, n = _marshal(patterns, flags, ids)
    entry = ends_entry(lib)
    found = ctypes.c_size_t()
    if capacity is None:
        rc = entry(ptr, size, location, pa, fa, ia, n, buffer_size, None, 0, ctypes.byref(found), None)
        if rc:
            return rc, [], 0
        capacity = found.value
    out = (MatchEnd * max(1, capacity))()
    rc = entry(ptr, size, location, pa, fa, ia, n, buffer_size, out, capacity, ctypes.byref(found),
               ctypes.byref(stats) if stats is not None else None)
    stored = min(capacity, found.value)
    return rc, [(out[k].line_number, out[k].id, out[k].end) for k in range(stored)], found.value


def oracle_ends(oracle, data: bytes, patterns, flags, ids, buffer_size: int, capacity: int | None = None):
    """oracle_ends_buffer -> (rc, [(line, id, end)], count found); the same contract as match_ends."""
    pa, fa, ia, n = _marshal(patterns, flags, ids)
    entry = oracle.oracle_ends_buffer
    entry.restype = ctypes.c_int
    entry.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, ctypes.c_int,
                      ctypes.c_void_p, ctypes.c_ulonglong, ctypes.POINTER(ctypes.c_ulonglong)]
    found = ctypes.c_ulonglong()
    if capacity is None:
        rc = entry(data, len(data), pa, fa, ia, n, buffer_size, None, 0, ctypes.byref(found))
        if rc:
            return rc, [], 0
        capacity = found.value
    out = (MatchEnd * max(1, capacity))()
    rc = entry(data, len(data), pa, fa, ia, n, buffer_size, out, capacity, ctypes.byref(found))
    stored = min(capacity, found.value)
    return rc, [(out[k].line_number, out[k].id, out[k].end) for k in range(stored)], found.value


# ---- random general-mode cases -------------------------------------------------------------------------------------------

def _gap_pattern(rng: random.Random) -> tuple[bytes, bytes]:
    """A literal, a gap of 60-100 arbitrary bytes, a literal: too many DFA states for the default budget, so it becomes an
    NFA fallback.  Returns (pattern, an instance of it)."""
    a, b = fpc.words(rng.randrange(1 << 30), 2, rng.choice([4, 5]))
    gap = rng.choice([60, 80, 100])
    filler = "".join(rng.choice("qjxz0189 _") for _ in range(gap))
    return f"{a}.{{{gap}}}{b}".encode(), (a + filler + b).encode()


def _draw_patterns(rng: random.Random, oracle, k: int) -> tuple[list[bytes], list[bytes]]:
    """k patterns the oracle accepts, from the three generators of the suite plus gap patterns; and literal pieces to plant."""
    patterns, pieces = [], []
    while len(patterns) < k:
        roll = rng.random()
        if roll < 0.35:
            pattern, piece = gen_regex(rng).encode(), []
        elif roll < 0.7:
            text, lits = fpc.fast_factor_pattern(rng)
            if "{1" in text and " ." in text:   # its gap patterns are 100-150 wide: kept for _gap_pattern's narrower ones
                continue
            pattern, piece = text.encode(), [p.encode() for p in lits]
        elif roll < 0.9:
            pattern, piece = byte_cases.byte_regex(rng), []
        else:
            pattern, lit = _gap_pattern(rng)
            piece = [lit]
        if pattern in patterns or check(oracle, [pattern], flags=[0], ids=[0]) != 0:
            continue
        patterns.append(pattern)
        pieces += piece
    return patterns, pieces


def _text(rng: random.Random, nrng: np.random.Generator, size: int, buffer_size: int, pieces: list[bytes], nul_rate: float) -> bytes:
    """Mostly short lines over a small alphabet (letters the generators use, a few high and control bytes), literal pieces
    planted about every 300 bytes, a few lines longer than buffer_size when it is small."""
    alphabet = np.frombuffer(b"abcABxX _1.\t-" + bytes(rng.sample(range(1, 256), 12)).replace(b"\n", b"y"), dtype=np.uint8)
    lengths = np.where(nrng.random(size // 12 + 16) < 0.9, nrng.integers(0, 24, size // 12 + 16), nrng.integers(24, 120, size // 12 + 16))
    ends = np.cumsum(lengths + 1)
    ends = ends[ends <= size]
    size = int(ends[-1])
    buf = alphabet[nrng.integers(0, alphabet.size, size)]
    buf[ends - 1] = 10
    for p in np.sort(nrng.integers(0, max(1, size - 200), max(1, size // 300))).tolist():
        if not pieces:
            break
        piece = rng.choice(pieces)
        if rng.random() < 0.3:
            piece = piece.swapcase()
        buf[p:p + len(piece)] = np.frombuffer(piece, dtype=np.uint8)[: size - p]
    if nul_rate:
        buf[nrng.random(size) < nul_rate] = 0
    data = bytearray(buf.tobytes())
    if buffer_size <= 4096:
        # lines longer than a pseudo-line: the engine splits them (run_general's split branch); kept few, since the oracle's
        # cost grows with the square of the pseudo-line length
        for _ in range(rng.randint(2, 5)):
            at = data.find(b"\n", rng.randrange(len(data)))
            if at >= 0:
                long = bytes(alphabet[nrng.integers(0, alphabet.size, rng.randint(buffer_size, min(3 * buffer_size + 7, 9000)))])
                data[at + 1:at + 1] = long.replace(b"\n", b"y") + b"\n"
    if rng.random() < 0.3:
        data = data.rstrip(b"\n") + b"q"   # no final newline
    return fpc._no_all_nul_pseudo_lines(bytes(data), buffer_size)  # pylint: disable=protected-access


def event_case(seed: int, oracle, size: int | None = None) -> dict:
    """One random general-mode case: 3-6 patterns with shared or distinct ids, SINGLEMATCH per id mixed with patterns that
    report every end, some CASELESS; a text of 1-6 MiB (or `size` bytes); buffer_size and buffer_count; and max_match_count
    of 0, 1 or "mid" (the test puts the limit inside a line with several reports)."""
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    k = rng.choice([3, 4, 5, 6])
    patterns, pieces = _draw_patterns(rng, oracle, k)
    id_mode = ["shared", "distinct", "mixed"][seed % 3]
    if id_mode == "shared":
        ids = [rng.randint(0, 1) for _ in range(k)]
    elif id_mode == "distinct":
        ids = list(range(10, 10 + k))
    else:
        ids = [rng.randint(0, k // 2) for _ in range(k)]
    singlematch = {i: rng.random() < 0.4 for i in set(ids)}   # patterns sharing an id agree on SINGLEMATCH
    singlematch[ids[0]] = False                                 # never all SINGLEMATCH with one id (that is simple mode)
    flags = [(SINGLEMATCH if singlematch[i] else 0) | (CASELESS if rng.random() < 0.3 else 0) | rng.choice([0, 0, 2, 4, 6]) for i in ids]
    buffer_size = BUFFER_SIZES[seed % len(BUFFER_SIZES)]
    if size is None:
        size = rng.choice([1 << 20, 1 << 20, 2 << 20, 3 << 20, 6 << 20])
    data = _text(rng, nrng, size, buffer_size, pieces, rng.choice([0.0, 0.0, 0.002]))
    return {"seed": seed, "patterns": patterns, "flags": flags, "ids": ids, "buffer_size": buffer_size, "data": data,
            "buffer_count": BUFFER_COUNTS[(seed // len(BUFFER_SIZES)) % len(BUFFER_COUNTS)], "max_match": [0, 1, "mid"][seed % 3 if seed % 4 else 0]}


def mid_line_limit(records) -> int:
    """A max_match_count that is reached by a report that is not the last one of its line (0 if no line has two)."""
    for k in range(1, len(records)):
        if records[k][1] == records[k - 1][1]:
            return k   # records k-1 and k share a line: the limit falls on k-1, and k still comes
    return 0


# ---- sets of an exact number of DFA groups ------------------------------------------------------------------------------

GAP_PATTERNS = ["alpha .{30}omega", "kilo.{20}gram"]


def many_group_set(lib, k: int, mode: str, extra_nfa: int = 0) -> dict:
    """k eight-letter words plus 2-4 gap patterns (NFA fallbacks), and the DFA state budget at which the words compile to
    exactly k groups - one word each.  mode "simple": every pattern SINGLEMATCH with id 0; "general": distinct ids, every
    other word without SINGLEMATCH.  Returns patterns, flags, ids, budget, groups, the number of NFA patterns and `member`:
    which pattern sits in groups 0, 31, 32, 63, 64 and k - 1 (the ones below k).  Groups keep pattern order (database.cpp
    build_groups), NFA fallbacks leave it; the members are read from the compiled database, not assumed."""
    words = fpc.words(7, k, 8)
    gaps = GAP_PATTERNS + ["charlie.{40}delta", "echo.{25}foxtrot"][:extra_nfa]
    patterns = words + gaps
    n = len(patterns)
    if mode == "simple":
        flags, ids = [14] * n, [0] * n
    else:
        flags = [14 if i % 2 else 6 for i in range(n)]
        ids = list(range(1, n + 1))
    for budget in (12, 14, 16, 18, 20):
        with fpc.environment({"GPUGREP_MAX_DFA_STATES": str(budget)}):
            db = CompiledDb(lib, patterns, flags, ids)
        if db.rc == 0 and db.info.groups == k:
            break
    else:
        raise AssertionError(f"no budget gives {k} groups")
    members = [g[0].members for g in db.groups]
    nfa = n - sum(members)
    assert nfa == len(gaps) and members == [1] * k, (members, nfa)
    return {"patterns": patterns, "flags": flags, "ids": ids, "budget": budget, "groups": db.info.groups, "nfa": nfa,
            "simple": bool(db.info.simple), "member": {g: words[g] for g in (0, 31, 32, 63, 64, k - 1) if g < k}, "gaps": gaps}


def many_group_text(groups: dict, seed: int, size: int = 1 << 20) -> bytes:
    """Background lines (bytes no pattern uses) with plants, each on a line of its own: the members of the groups that
    many_group_set names and an instance of every gap pattern, each starting at every offset mod 16; and lines with a word and the start
    of a gap pattern's instance in the same 16-byte chunk.  So some lines are matched by the group-31 member alone, others
    by an NFA pattern alone."""
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    background = fpc.BACKGROUND
    instances = {"alpha .{30}omega": "alpha " + "x" * 30 + "omega", "kilo.{20}gram": "kilo" + "q" * 20 + "gram",
                 "charlie.{40}delta": "charlie" + "z" * 40 + "delta", "echo.{25}foxtrot": "echo" + "0" * 25 + "foxtrot"}
    plants = [w.encode() for w in groups["member"].values()] + [instances[g].encode() for g in groups["gaps"]]
    word = groups["member"][0].encode()
    both = b"kilo" + word + b"q" * 12 + b"gram"   # the word lies inside the NFA instance's gap, in the chunk of "kilo"
    lines = []
    total = 0
    while total < size:
        line = bytes(background[nrng.integers(0, background.size, rng.randint(20, 160))])
        lines.append(line)
        total += len(line) + 1
    out = bytearray()
    plant_at = set(rng.sample(range(len(lines)), min(len(lines), 16 * (len(plants) + 1))))
    queue = [(p, r) for p in plants + [both] for r in range(16)]
    for i, line in enumerate(lines):
        if i in plant_at and queue:
            piece, r = queue.pop()
            pad = (r - (len(out) + 3)) % 16 + 3   # the plant starts at a byte offset == r mod 16
            line = line[:pad] + piece + line[pad + len(piece):]
        out += line + b"\n"
    assert not queue
    return bytes(out)
