"""Synthetic workloads of BASELINE.json (SURVEY.md §8d): seeded syslog-shaped text and the pattern sets.

Used by bench.py, __graft_entry__.smoke() and the tests.  The text generator itself is native
(``gpugrep_synth_syslog`` in libgpugrep_synth.so, csrc/synth.cpp - a library of its own, so that a process which must
not load the product, like ``bench.py --impl reference``, can still produce the corpus) so that 10 GiB can be produced
in seconds; this module only holds the pattern sets and the ctypes glue.  Nothing here is on the scan path.
"""

from __future__ import annotations

import ctypes
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np

BLOCK_BYTES = 16 << 20  # generation granularity: block k is generated from seed + k


_SYNTH_LIB: ctypes.CDLL | None = None


def _lib() -> ctypes.CDLL:
    global _SYNTH_LIB  # pylint: disable=global-statement
    if _SYNTH_LIB is None:
        _SYNTH_LIB = ctypes.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libgpugrep_synth.so"))
    return _SYNTH_LIB


def _bind(lib: ctypes.CDLL) -> ctypes.CDLL:
    lib.gpugrep_synth_syslog.restype = ctypes.c_size_t
    lib.gpugrep_synth_syslog.argtypes = [
        ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_uint, ctypes.c_uint,
    ]
    return lib


def fill_syslog(out: np.ndarray, seed: int = 1234, plants: list[str] | None = None, plant_ppm: int = 0,
                threads: int = 0, lib: ctypes.CDLL | None = None) -> int:
    """Fill a uint8 array with synthetic syslog text; returns the number of lines.  Deterministic in (seed, size).
    `lib` is accepted for older call sites and ignored: the generator lives in libgpugrep_synth.so."""
    assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
    del lib
    lib = _bind(_lib())
    plant_array = None
    count = 0
    if plants:
        encoded = [p.encode() for p in plants]
        plant_array = (ctypes.c_char_p * len(encoded))(*encoded)
        count = len(encoded)
    base = out.ctypes.data
    size = out.size
    blocks = [(k, off, min(BLOCK_BYTES, size - off)) for k, off in enumerate(range(0, size, BLOCK_BYTES))]

    def work(item: tuple[int, int, int]) -> int:
        k, off, length = item
        return lib.gpugrep_synth_syslog(seed + k, base + off, length, plant_array, count, plant_ppm)

    threads = threads or min(64, os.cpu_count() or 8)
    if len(blocks) <= 1 or threads <= 1:
        return sum(work(b) for b in blocks)
    with ThreadPoolExecutor(max_workers=threads) as pool:
        return sum(pool.map(work, blocks))


def syslog_bytes(size: int, seed: int = 1234, plants: list[str] | None = None, plant_ppm: int = 0,
                 lib: ctypes.CDLL | None = None) -> bytes:
    out = np.empty(size, dtype=np.uint8)
    fill_syslog(out, seed, plants, plant_ppm, lib=lib)
    return out.tobytes()


# ---- BASELINE.json configs[0]: one literal ----
C1_PATTERNS = ["ERROR"]

# ---- BASELINE.json configs[1]: 32 mixed patterns = 20 literals (8-20 bytes) + 12 character-class patterns ----
C2_LITERALS = [
    "Failed password for", "invalid user", "segfault at", "Out of memory", "Kill process", "sacrifice child",
    "nf_conntrack: table", "dropping packet", "authentication fail", "bad certificate", "TLS handshake error",
    "disk quota exceeded", "SYN flooding", "Sending cookies", "I/O error, dev", "nil pointer", "panic: runtime error",
    "goroutine", "op 0x1:(WRITE)", "tty=ssh ruser=",
]
C2_CLASSES = [
    r"[Ff]ailed password", r"port [0-9]+", r"id=[0-9a-f]{12}", r"host0[0-4][0-9] kernel", r"error [0-9]+ in lib\w+\.so",
    r"score [0-9]{1,4}", r"rhost=10\.[0-9]+\.[0-9]+\.[0-9]+", r"/dev/sd[a-f][1-4]", r"sector [0-9]{6,}",
    r"user=(root|admin)", r"HTTP/1\.1 404 [0-9]{5}B", r"dur=499[0-9]ms",
]
C2_PATTERNS = C2_LITERALS + C2_CLASSES


def c3_patterns(seed: int = 77) -> tuple[list[str], list[str]]:
    """configs[2]: 1,000 IOC-style patterns = 950 literals (hex digests, domains, paths; 6-24 bytes) + 50 class patterns.

    Returns (patterns, plant strings): the plants are literal indicators the generator injects at ~0.1 % of lines.
    """
    rng = random.Random(seed)
    tlds = ["com", "net", "org", "ru", "cn", "io", "info", "biz", "xyz", "top"]
    syll = ["ka", "zu", "mo", "ri", "ta", "ne", "lo", "vi", "xa", "qu", "be", "do", "fi", "gu", "hy", "jo"]
    literals: set[str] = set()
    while len(literals) < 950:
        kind = rng.random()
        if kind < 0.4:
            literals.add("".join(rng.choice("0123456789abcdef") for _ in range(rng.choice([16, 20, 24]))))
        elif kind < 0.75:
            name = "".join(rng.choice(syll) for _ in range(rng.randint(2, 4)))
            literals.add(f"{name}{rng.randint(0, 99)}.{rng.choice(tlds)}")
        else:
            parts = ["".join(rng.choice(syll) for _ in range(rng.randint(1, 2))) for _ in range(rng.randint(2, 3))]
            literals.add(("/" + "/".join(parts) + rng.choice([".sh", ".php", ".dll", ".bin", ""]))[:24])
    lits = sorted(literals)
    rng.shuffle(lits)
    escaped = [lit.replace(".", r"\.") for lit in lits]
    classes = []
    for k in range(50):
        which = k % 5
        if which == 0:
            classes.append(rf"10\.{rng.randint(0, 255)}\.\d{{1,3}}\.\d{{1,3}} beacon")
        elif which == 1:
            classes.append(rf"/tmp/\.[a-z]{{4,8}}{rng.randint(10, 99)}")
        elif which == 2:
            classes.append(rf"cmd=[A-Za-z0-9+/]{{16,}}{rng.choice('QRSTUVWX')}==")
        elif which == 3:
            classes.append(rf"{rng.choice(syll)}{rng.choice(syll)}[0-9]{{2,4}}\.onion")
        else:
            classes.append(rf"User-Agent: [a-z]+bot/{rng.randint(1, 9)}\.[0-9]")
    return escaped + classes, lits


def c5_patterns(count: int = 10000, seed: int = 99) -> list[str]:
    """configs[4]: caseless patterns with alternation, bounded repeats and anchors, generated from templates."""
    rng = random.Random(seed)
    nouns = ["session", "request", "payment", "invoice", "shipment", "account", "device", "cluster", "tenant", "gateway",
             "pipeline", "worker", "volume", "replica", "ledger", "wallet", "sensor", "router", "tunnel", "broker"]
    verbs = ["failed", "rejected", "expired", "revoked", "stalled", "aborted", "degraded", "throttled", "poisoned", "orphaned"]
    out: set[str] = set()
    while len(out) < count:
        kind = rng.randrange(6)
        noun, verb = rng.choice(nouns), rng.choice(verbs)
        num = rng.randint(100, 99999)
        if kind == 0:
            out.add(rf"{noun}_{num} (?:{verb}|{rng.choice(verbs)}|{rng.choice(verbs)})")
        elif kind == 1:
            out.add(rf"\"{noun}Id\":\"[a-z]{{3,12}}{num}\"")
        elif kind == 2:
            out.add(rf"^\{{\"ts\":\d{{10}},\"svc\":\"{noun}{num % 1000}\"")
        elif kind == 3:
            out.add(rf"{verb} x{{2,8}}{num}")
        elif kind == 4:
            out.add(rf"code=(?:E|W){num}[a-f0-9]{{2,6}}")
        else:
            out.add(rf"{noun}-{verb}-{num}\}}$")
    return sorted(out)


def jsonish_bytes(size: int, seed: int = 4321, patterns_to_plant: list[str] | None = None, plant_rate: float = 0.02) -> bytes:
    """configs[4] text: long JSON-ish lines (2-16 KiB each).  `patterns_to_plant` are literal strings sprinkled into
    about `plant_rate` of the lines.  Pure Python: meant for parity-test sizes, not for the 10 GiB bench."""
    rng = random.Random(seed)
    nouns = ["session", "request", "payment", "invoice", "shipment", "account", "device", "cluster", "tenant", "gateway"]
    out = bytearray()
    while len(out) < size:
        fields = [f'{{"ts":{rng.randint(1_600_000_000, 1_800_000_000)},"svc":"{rng.choice(nouns)}{rng.randint(0, 999)}"']
        target = rng.randint(2048, 16384)
        length = len(fields[0])
        while length < target:
            key = f'{rng.choice(nouns)}{rng.choice(["Id", "State", "Code", "Note"])}'
            kind = rng.random()
            if kind < 0.4:
                value = '"' + "".join(rng.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(rng.randint(3, 12))) + str(rng.randint(100, 99999)) + '"'
            elif kind < 0.7:
                value = str(rng.randint(0, 10 ** 9))
            else:
                value = '"' + " ".join(rng.choice(nouns) for _ in range(rng.randint(1, 6))) + '"'
            field = f'"{key}":{value}'
            if patterns_to_plant and rng.random() < plant_rate / 8:
                field += ',"evt":"' + rng.choice(patterns_to_plant) + '"'
            fields.append(field)
            length += len(field) + 1
        out += (",".join(fields) + "}\n").encode()
    return bytes(out[:size].rsplit(b"\n", 1)[0] + b"\n")


_FILLER = [b"session", b"opened", b"upstream", b"handler", b"timeout", b"pending", b"device", b"req=3ec9805d", b"dur=424ms", b"pod"]
_ERROR_WORDS = [b"errors", b"xerror", b"error_1", b"terrorize", b"errorless", b"Aerror"]


def dense_reject_bytes(lines: int, seed: int = 1) -> tuple[bytes, list[int]]:
    """A text for whole-word scans of `error` in which nearly every selected line is rejected: every line (about 230 bytes)
    holds `error` inside two longer words, and one line in 97 also holds it as a word.  Returns the text and the numbers
    (0-based) of those lines.  The lines are long enough that the fast path keeps its candidate and record capacity."""
    rng = random.Random(seed)
    out, words = [], []
    for k in range(lines):
        parts = [rng.choice(_FILLER) for _ in range(rng.randint(22, 30))]
        for _ in range(2):
            parts.insert(rng.randint(0, len(parts)), rng.choice(_ERROR_WORDS))
        if k % 97 == 5:
            parts.insert(rng.randint(0, len(parts)), rng.choice([b"error", b"(error)", b"error:", b"-error-"]))
            words.append(k)
        out.append(b" ".join(parts))
    return b"\n".join(out) + b"\n", words
