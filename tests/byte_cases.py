"""Inputs over the whole byte alphabet (tests/test_byte_alphabet.py, tools/fuzz_gpu.py `bytes`): patterns built from high
bytes, control bytes, every escape form the parser takes, POSIX classes and the punctuation pairs that differ only in
bit 5; texts of bytes 1-255 weighted towards the edges of those classes and towards the near-misses of the SWAR tests.

The patterns are bytes (a raw byte >= 0x80 stands for itself; a str would reach the C side UTF-8 encoded).  The oracle
has no UTF mode, uses the C-locale tables of PCRE2 and folds ASCII letters only: `(?i)\\xc9` matches 0xC9, never 0xE9.
"""

from __future__ import annotations

import random

import numpy as np

import fast_path_cases as fpc
from k1_model import super_block_bytes
from regex_gen import ANCHORS

_META = set(b"\\^$.|?*+()[]{}")


def escaped(b: int, rng: random.Random | None = None) -> bytes:
    """One byte as a pattern atom that matches exactly that byte: raw (meta characters behind a backslash) or one of the
    escape forms \\xHH, \\x{HH}, \\o{ooo}, \\0oo, \\cX and the named escapes."""
    forms = ["hex"]
    if rng is None:
        return b"\\x%02x" % b
    if b not in (0, 10) and (b < 0x80 or rng.random() < 0.5):
        forms.append("raw")
    forms += ["hexbrace", "octbrace"]
    if b < 0o100:
        forms.append("oct0")
    if (b < 0x20 or b == 0x7F) and b != 0x1C:
        forms.append("ctrl")   # \cX: X is printable (PCRE2 rejects a control character after \c)
    named = {27: b"\\e", 7: b"\\a", 12: b"\\f", 13: b"\\r", 9: b"\\t"}
    if b in named:
        forms.append("named")
    form = rng.choice(forms)
    if form == "raw":
        return (b"\\" if b in _META else b"") + bytes([b])
    if form == "hexbrace":
        return b"\\x{%x}" % b if rng.random() < 0.5 else b"\\x{%02X}" % b
    if form == "octbrace":
        return b"\\o{%o}" % b
    if form == "oct0":
        return b"\\0%02o" % b   # always two digits: a following octal digit must not extend the escape
    if form == "ctrl":
        x = b ^ 0x40
        return b"\\c" + bytes([x | 0x20 if 0x41 <= x <= 0x5A and rng.random() < 0.5 else x])   # \ca == \cA
    if form == "named":
        return named[b]
    return b"\\x%02x" % b if rng.random() < 0.5 else b"\\x%02X" % b


HIGH = [0x80, 0x85, 0xA0, 0xC9, 0xE9, 0xFF, 0x8A, 0xC3, 0xA9, 0x89]
CONTROL = [0x01, 0x0B, 0x0C, 0x0D, 0x1B, 0x7F, 0x09]
# the pairs that differ only in bit 5 without being letters, and letters that do
BIT5 = [ord(c) for c in "@`[{\\|]}^~"] + [0xC9, 0xE9, 0xC0, 0xE0, ord("a"), ord("A"), ord("e"), ord("E")]
UTF8 = [b"\xc3\xa9", b"\xc3\x89", b"\xe2\x80\x94", b"\xc3\xbc"]
CLASSES = [rb"\h", rb"\H", rb"\v", rb"\V", rb"\N", rb"\W", rb"\S", rb"\D", rb"\w", rb"\s", rb".",
           rb"[\x7e-\x81]", rb"[\x7f-\x80]", rb"[@-\x60]", rb"[Z-a]", rb"[\xc0-\xdf]", rb"[^\x00-\x7f]", rb"[\x80-\xff]", rb"[^\x80-\xbf]",
           rb"[\x00-\x1f]", rb"[\xa0\x85]", rb"[\h\v]", rb"[^\h]", rb"[\x{c9}\o{351}]", rb"[\e\cA-\cZ]", rb"[\1\7]", rb"[\8\9]",
           rb"[[:^ascii:]]", rb"[[:ascii:]]", rb"[[:punct:]]", rb"[[:cntrl:]]", rb"[[:print:]]", rb"[[:graph:]]", rb"[[:xdigit:]]",
           rb"[^[:print:]]", rb"[[:^graph:]]", rb"[[:alpha:]\xe9]", rb"[@`]", rb"[\[{]", rb"[\\|]", rb"[\]}]", rb"[\^~]"]
INLINE = [b"(?i)", b"(?-i)", b"(?s)", b"(?i-s)"]


def _atom(rng: random.Random) -> bytes:
    r = rng.random()
    if r < 0.22:
        return escaped(rng.choice(HIGH), rng)
    if r < 0.32:
        return escaped(rng.choice(CONTROL), rng)
    if r < 0.52:
        return escaped(rng.choice(BIT5), rng)
    if r < 0.6:
        return b"".join(escaped(b, rng) for b in rng.choice(UTF8))
    if r < 0.9:
        return rng.choice(CLASSES)
    return rng.choice(INLINE)


def byte_regex(rng: random.Random, depth: int = 0) -> bytes:
    """regex_gen.gen_regex over byte atoms: sequences, alternation, repeats, anchors, inline (?i) / (?-i) / (?s) and
    (?i:...) groups."""
    r = rng.random()
    if depth > 3 or r < 0.35:
        return b"".join(_atom(rng) for _ in range(rng.randint(1, 4)))
    if r < 0.5:
        return byte_regex(rng, depth + 1) + byte_regex(rng, depth + 1)
    if r < 0.65:
        opener = rng.choice([b"(?:", b"(?:", b"(?i:", b"(?-i:", b"(?s:"])
        return opener + byte_regex(rng, depth + 1) + b"|" + byte_regex(rng, depth + 1) + b")"
    if r < 0.85:
        q = rng.choice([b"?", b"*", b"+", b"{2}", b"{1,3}", b"{2,}", b"{0,2}", b"+?", b"*?"])
        return b"(" + byte_regex(rng, depth + 1) + b")" + q
    if r < 0.95:
        return rng.choice(ANCHORS).encode() + byte_regex(rng, depth + 1)
    return byte_regex(rng, depth + 1) + rng.choice([b"$", b"\\b", b"\\z", b"\\Z", b"\\B"])


# text bytes: the edges of the classes above, the bit-5 partners, and the near-misses of the SWAR tests next to '\n' and NUL
EDGES = [0x1F, 0x20, 0x7E, 0x7F, 0x80, 0x84, 0x85, 0x9F, 0xA0, 0xBF, 0xC0, 0xDF, 0xE0, 0xFF]
NEAR_MISSES = [0x8A, 0x8D, 0x80, 0x81]


def byte_text(rng: random.Random, lines: int, max_len: int = 24, nul_rate: float = 0.0) -> bytes:
    """Lines of bytes 1-255 without '\\n' (NUL at `nul_rate`); 0x8A, 0x8D, 0x80 and 0x81 often stand right before and
    after a newline or a NUL."""
    pools = [EDGES, BIT5, HIGH, CONTROL, NEAR_MISSES, list(range(1, 10)) + list(range(11, 256))]
    weights = [3, 3, 3, 1, 2, 2]
    out = bytearray()
    for _ in range(lines):
        for _ in range(rng.randint(0, max_len)):
            if nul_rate and rng.random() < nul_rate:
                out.append(0)
                if rng.random() < 0.5:
                    out.append(rng.choice(NEAR_MISSES))
            elif rng.random() < 0.12:
                out += rng.choice(UTF8)
            else:
                out.append(rng.choice(rng.choices(pools, weights)[0]))
        if rng.random() < 0.3:
            out.append(rng.choice(NEAR_MISSES))
        out.append(10)
        if rng.random() < 0.3:
            out.append(rng.choice(NEAR_MISSES))
    if rng.random() < 0.3 and out:
        out.pop()
    return bytes(out)


def byte_random_case(seed: int):
    """parity.random_case over the byte alphabet: the same modes, flags, buffer sizes, buffer counts and limits."""
    rng = random.Random(seed)
    k = rng.choice([1, 1, 1, 2, 3, 5])
    patterns = [byte_regex(rng) for _ in range(k)]
    mode = rng.choice(["simple", "simple", "ids", "nosm", "mixed"])
    base = rng.choice([14, 14, 14, 10, 12, 8, 15, 14])
    flags = [base] * k
    if mode == "simple":
        ids = [rng.choice([0, 7])] * k
    elif mode == "ids":
        ids = [rng.randint(0, 2) for _ in range(k)]
    elif mode == "nosm":
        flags = [f & ~8 for f in flags]
        ids = [rng.randint(0, 1) for _ in range(k)]
    else:
        ids = list(range(k))
        flags = [f & ~8 if i % 2 else f for i, f in enumerate(flags)]
    buffer_size = rng.choice([262140, 262140, 64, 9, 5])
    data = byte_text(rng, rng.choice([0, 1, 30, 200]), nul_rate=rng.choice([0, 0, 0.05]))
    buffer_count = rng.choice([16, 1, 3])
    max_match = rng.choice([0, 0, 0, 1, 4])
    return patterns, flags, ids, buffer_size, data, buffer_count, max_match


# ---- factor sets on the fast path ------------------------------------------------------------------------------------------
# stems of UTF-8 words and punctuation; the background never contains one of their bytes
STEMS = [b"caf\xc3\xa9s", b"\xc3\x89t\xc3\xa9_x", b"na\xc3\xafve!", b"[warn]{x}", b"@user`q`", b"pipe|b\\c", b"hat^tilde~",
         b"\xc2\xa0nbsp\xc2\xa0", b"r\xc3\xa9sum\xc3\xa9", b"stra\xc3\x9fe", b"\xe2\x80\x94dash", b"\x1b[31mred", b"\xe9t\xe9@\xc9T",
         b"\xff\xfebom\xfd", b"ma\xc3\xb1ana", b"gr\xc3\xbc\xc3\x9fe{}"]
_STEM_BYTES = {b for s in STEMS for b in s}
BACKGROUND = np.array([b for b in range(0x80, 0x100) if b not in _STEM_BYTES and b ^ 0x20 not in _STEM_BYTES and b not in (0x8A,)]
                      + [0x8A] * 8 + [0x20] * 8, dtype=np.uint8)


def pattern_of(literal: bytes, rng: random.Random | None = None) -> bytes:
    return b"".join(escaped(b, rng) for b in literal)


def _is_letter(b: int) -> bool:
    return 0x41 <= b <= 0x5A or 0x61 <= b <= 0x7A


def flip_case(piece: bytes, rng: random.Random) -> bytes:
    """Letters in random case: a caseless pattern still matches."""
    return bytes(b ^ 0x20 if _is_letter(b) and rng.random() < 0.5 else b for b in piece)


def flip_bit5(piece: bytes, rng: random.Random) -> bytes | None:
    """One non-letter byte with bit 5 flipped (0xE9 <-> 0xC9, '@' <-> '`', '[' <-> '{'): the folded prefilter and the
    extended confirmation let it through, no pattern matches it.  None if the piece has no such byte."""
    at = [k for k, b in enumerate(piece) if not _is_letter(b) and b not in (0x0A, 0x2A) and (b ^ 0x20) not in (0, 10)]
    if not at:
        return None
    k = rng.choice(at)
    return piece[:k] + bytes([piece[k] ^ 0x20]) + piece[k + 1:]


def _core(rng: random.Random) -> bytes:
    core = rng.choice(STEMS)[: rng.choice([4, 5, 6, 7, 8, 9])]
    if rng.random() < 0.2:
        core += rng.choice([b" ", b"\xa0", b"-"]) + rng.choice(STEMS)[: rng.randint(2, 5)]
    return core


PRE = [b"", b"", b"", b"^", rb"\b", rb"[\x80-\xff]", rb"\W", b".*", rb"[^\x00-\x7f]{1,3}", rb"\h", b"[[:punct:]]", rb"(?:\xe9|\xc9)", rb"\B"]
SUF = [b"", b"", b"", b"$", rb"\b", rb"[\x80-\xbf]", rb"\v", rb"\S?", rb".\xff", rb"[^\xa0]", rb"[[:^ascii:]]{1,2}", rb"\N", rb"[@-\x60]"]


def byte_factor_pattern(rng: random.Random) -> tuple[bytes, list[bytes]]:
    """(pattern, literal pieces that a match needs), as fast_path_cases.fast_factor_pattern builds them."""
    roll = rng.random()
    if roll < 0.08:
        a, b = _core(rng), _core(rng)
        gap = rng.choice([100, 150])
        return pattern_of(a, rng) + b".{%d}" % gap + pattern_of(b, rng), [a + bytes(rng.choice(BACKGROUND.tolist()) for _ in range(gap)) + b]
    if roll < 0.25:
        a, b = _core(rng), _core(rng)
        body, pieces = b"(?:" + pattern_of(a, rng) + b"|" + pattern_of(b, rng) + b")", [a, b]
    else:
        a = _core(rng)
        body, pieces = pattern_of(a, rng), [a]
    return rng.choice(PRE) + body + rng.choice(SUF), pieces


def byte_words(seed: int, count: int, length: int) -> list[bytes]:
    """Distinct words of ASCII letters with one or two bytes that are not letters (high bytes and punctuation with a bit-5
    partner) at random places: a caseless set of them folds to far fewer grams, like fast_path_cases.words."""
    rng = random.Random(seed)
    others = [0xE9, 0xC9, 0xE0, 0xFC, 0xDC, 0xA0, 0x80, 0xBF, ord("@"), ord("`"), ord("["), ord("{"), ord("~"), ord("^"), ord("|"), ord("\\")]
    out = set()
    while len(out) < count:
        w = [ord(rng.choice(fpc.LETTERS)) for _ in range(length)]
        for _ in range(rng.choice([1, 1, 2])):
            w[rng.randrange(length)] = rng.choice(others)
        if sum(map(_is_letter, w)) >= 2:
            out.add(bytes(w))
    return sorted(out)


def byte_fast_case(seed: int) -> dict:
    """fast_path_cases.fast_case over the byte alphabet: UTF-8 and punctuation factors planted at every alignment in a
    background of high bytes that never holds one of their bytes.  Caseless cases plant letters in random case (these
    match) and, as often, pieces with one non-letter flipped in bit 5 (these must not match: the prefilter folds them)."""
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    sm_id = rng.choice([0, 7])
    caseless = rng.random() < 0.4
    if seed % 4 == 0:   # a large caseless set: folded tables, stride 1, 2, 4 and mixed sampling in turn
        kind = (seed // 4) % 4
        words = byte_words(seed, 300, 4) if kind == 0 else byte_words(seed, 200, 5) if kind == 1 else byte_words(seed, 100, 8) if kind == 2 \
            else byte_words(seed, 1, 5) + byte_words(seed + 1, 120, 9)
        pats = [pattern_of(w, rng) for w in words]
        pieces = [[w] for w in words]
        flags = [15] * len(pats)
        caseless = True
    else:
        k = rng.choice([1, 2, 3, 4, 6])
        made = [byte_factor_pattern(rng) for _ in range(k)]
        pats = [p for p, _ in made]
        pieces = [pc for _, pc in made]
        flags = [rng.choice([15, 15, 11]) if caseless else rng.choice([14, 14, 10, 12, 8]) for _ in pats]
    buffer_size = fpc.BUFFER_SIZES[seed % len(fpc.BUFFER_SIZES)]
    size = rng.choice([256 << 10, 512 << 10, 1 << 20, 2 << 20])
    longest = min(16384, super_block_bytes(buffer_size))
    kinds = nrng.choice(4, size=size // 40 + 16, p=[0.3, 0.3, 0.37, 0.03])
    lengths = np.where(kinds == 0, nrng.integers(1, 16, kinds.size),
                       np.where(kinds == 1, nrng.integers(8, 72, kinds.size),
                                np.where(kinds == 2, nrng.integers(60, 400, kinds.size), nrng.integers(2048, longest + 1, kinds.size))))
    ends = np.cumsum(lengths)
    ends = ends[ends <= size]
    size = int(ends[-1]) if ends.size else size
    buf = BACKGROUND[nrng.integers(0, BACKGROUND.size, size)]
    buf[ends - 1] = 10
    nplants = max(4, size // 700)
    at = np.sort(nrng.integers(0, max(1, size - 300), nplants))
    for p in at.tolist():
        piece = rng.choice(rng.choice(pieces))
        if caseless:
            piece = flip_case(piece, rng)
            if rng.random() < 0.5:
                piece = flip_bit5(piece, rng) or piece
        ctx = rng.choice([b"", b" ", b"\xa0", b"_", b"7", b"\xe9", b"\n", b"\x85"])
        blob = ctx + piece + rng.choice([b"", b" ", b"\xff", b"9", b"\x80", b"x", b"\n", b"\xa0 "])
        if rng.random() < 0.02:
            blob = b"\0" + blob if rng.random() < 0.5 else blob + b"\0"
        buf[p:p + len(blob)] = np.frombuffer(blob, dtype=np.uint8)[: size - p]
    if rng.random() < 0.25:
        buf[-1] = 0xA0   # no final newline
    data = fpc._no_all_nul_pseudo_lines(buf.tobytes(), buffer_size)   # pylint: disable=protected-access
    return {"seed": seed, "patterns": pats, "flags": flags, "ids": [sm_id] * len(pats), "buffer_size": buffer_size, "data": data,
            "switch": "GPUGREP_FILTER=exact" if seed % 4 == 0 and (seed // 16) % 2 else
            fpc.SWITCHES[(seed // len(fpc.BUFFER_SIZES)) % len(fpc.SWITCHES)] if seed % 2 else fpc.SWITCHES[seed % len(fpc.SWITCHES)],
            "general_ok": False}


# ---- folded K1 configurations ------------------------------------------------------------------------------------------------
def _k1_byte_configs():
    """Sets of high-byte and punctuation factors for every instantiation of k_stream (stride 4, 2, 1 and mixed sampling; bloom
    and exact mode), the folded ones from caseless sets of byte_words, in the layout of fast_path_cases.K1_CONFIGS."""
    plain = {4: [b"r\xc3\xa9seau d\xc3\xa9faut", b"\xe2\x80\x94@\xc9T\xc9[x]"], 2: [b"\xe9t\xe9@!", b"\xc9T\xc9`?", b"[\xff]{}", b"\x1b[31m", b"\xa0\x85|~x"],
             1: [b"\xe9t\xe9\xff", b"\xc3\x89`{~\x80"]}
    folded = {4: byte_words(41, 80, 8), 2: byte_words(81, 160, 5), 1: byte_words(151, 320, 4)}
    mixed_plain = [b"\xe9t\xe9@!", b"r\xc3\xa9seau d\xc3\xa9faut", b"\xe2\x80\x94@\xc9T\xc9[x]"]
    mixed = byte_words(3, 1, 5) + byte_words(4, 200, 9)
    out = []
    for exact in (False, True):
        env = {"GPUGREP_NO_TUNE": "1"}
        if exact:
            env["GPUGREP_FILTER"] = "exact"
        mode = 1 if exact else 2
        for stride in (4, 2, 1):
            out.append((f"bytes_m{mode}_s{stride}", plain[stride], 14, env, (mode, stride, False, 0)))
            out.append((f"bytes_m{mode}_s{stride}_fold", folded[stride], 15, env, (mode, stride, True, 0)))
    out.append(("bytes_mixed", mixed_plain, 14, {"GPUGREP_NO_TUNE": "1"}, (2, 4, False, 2)))
    out.append(("bytes_mixed_fold", mixed, 15, {"GPUGREP_NO_TUNE": "1"}, (2, 4, True, 2)))
    return [(name, [pattern_of(w) for w in words] + [f"kq{name.replace('_', 'q')}kq".encode()], [flag] * (len(words) + 1), env, inst)
            for name, words, flag, env, inst in out]


K1_BYTE_CONFIGS = _k1_byte_configs()


def bit5_variants(grams: np.ndarray, seed: int) -> np.ndarray:
    """Every gram once as it is and once with each non-letter byte's bit 5 cleared and each letter in random case: bytes
    that are hits only because the streaming kernel folds every byte (0xC9 for 0xE9, '@' for '`', '[' for '{')."""
    r = np.random.default_rng(seed)
    g = grams.astype(np.uint32)
    b = np.stack([(g >> np.uint32(8 * k)) & np.uint32(0xFF) for k in range(4)])
    letter = ((b | np.uint32(0x20)) >= 0x61) & ((b | np.uint32(0x20)) <= 0x7A)
    flip = np.where(letter, r.random(b.shape) < 0.5, (b & np.uint32(0x20)) != 0)
    flip &= ~(((b & ~np.uint32(0x20)) == 0) | ((b & ~np.uint32(0x20)) == 0x0A))   # never produce NUL or '\n'
    b2 = np.where(flip, b & ~np.uint32(0x20), b)
    varied = b2[0] | (b2[1] << np.uint32(8)) | (b2[2] << np.uint32(16)) | (b2[3] << np.uint32(24))
    return np.concatenate([g, varied.astype(np.uint32)])


# K1 background: high bytes with a bit-5 partner among the grams' non-letters, and the SWAR near-misses; no letters, so no
# 4 bytes of it fold into a gram (every gram has a letter)
K1_BACKGROUND = np.array([0xC9, 0xC0, 0xDC, 0x80, 0x81, 0x8A, 0x8D, 0x9F, 0xA0, 0xBF, 0x9F, 0xFF, 0x40, 0x5B, 0x7E, 0x20], dtype=np.uint8)


def swar_near_miss_text(n: int, seed: int) -> bytes:
    """NUL-free lines dense in 0x80, 0x81 and 0x8A (0x8A - 0x80 == '\\n', 0x80 - 0x80 == NUL): the newline count and the NUL
    flag must not see them."""
    r = np.random.default_rng(seed)
    buf = np.array([0x80, 0x81, 0x8A, 0x8A, 0x8D, 0x80], dtype=np.uint8)[r.integers(0, 6, n)]
    nl = np.cumsum(r.integers(3, 200, n // 3 + 2))
    buf[nl[nl < n]] = 10
    return buf.tobytes()
