"""Inputs for the fast-path tests (tests/test_k1_model.py on CPU, tests/test_fast_path_gpu.py on the GPU): pattern sets that
select every instantiation of the streaming kernel, random factor sets with texts built to stay on the fast path, and
what the engine's launch rules (engine.cu slot_submit, engine_upload_prefilter) predict for them from the compiled tables.
"""

from __future__ import annotations

import contextlib
import os
import random

import numpy as np

import parity
from dfa_sim import CompiledDb
from k1_model import K1Tables, has_newline_free_super_block, super_block_bytes

# pattern letters; background text never uses them, so that gram hits come from planted factors (and bloom collisions)
LETTERS = "abcdefghiklmnoprstuvwy"
BACKGROUND = np.frombuffer(b"qjxzQJXZ0123456789  .,:;=/-", dtype=np.uint8)


@contextlib.contextmanager
def environment(env: dict):
    """Set $GPUGREP_* switches for the duration (the compiler and the engine read them on every call)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def words(seed: int, count: int, length: int) -> list[str]:
    rng = random.Random(seed)
    out = set()
    while len(out) < count:
        out.add("".join(rng.choice(LETTERS) for _ in range(length)))
    return sorted(out)


# ---- the instantiations of k_stream ----------------------------------------------------------------------------------------
# (mode, stride, fold, odd compares): mode 1 = exact table (GPUGREP_FILTER=exact), 2 = bloom bitmap (launch_stream_m)
ALL_INSTANTIATIONS = {(m, s, f, 0) for m in (1, 2) for s in (4, 2, 1) for f in (False, True)} | {(2, 4, False, 2), (2, 4, True, 2)}


def _k1_configs():
    plain = {4: ["connection refused", "segfault at"], 2: ["ERROR", "WARN:", "FATAL", "PANIC", "ALERT"], 1: ["abcd", "wxyz12"]}
    # caseless sets large enough that folding shrinks them more than 3x (prefilter.cpp build_uniform)
    folded = {4: words(40, 40, 8), 2: words(80, 80, 5), 1: words(150, 150, 4)}
    mixed = ["ERROR", "connection reset by peer", "segfault at"]
    mixed_folded = words(1, 1, 5) + words(2, 80, 9)
    out = []
    for exact in (False, True):
        env = {"GPUGREP_NO_TUNE": "1"}
        if exact:
            env["GPUGREP_FILTER"] = "exact"
        mode = 1 if exact else 2
        for stride in (4, 2, 1):
            out.append((f"m{mode}_s{stride}", plain[stride], [14] * len(plain[stride]), env, (mode, stride, False, 0)))
            out.append((f"m{mode}_s{stride}_fold", folded[stride], [15] * len(folded[stride]), env, (mode, stride, True, 0)))
    out.append(("mixed", mixed, [14] * 3, {"GPUGREP_NO_TUNE": "1"}, (2, 4, False, 2)))
    out.append(("mixed_fold", mixed_folded, [15] * len(mixed_folded), {"GPUGREP_NO_TUNE": "1"}, (2, 4, True, 2)))
    # the production case: tables tuned on the head of the input (2^20 bits, multiplier chosen against the sample)
    out.append(("tuned_s4", ["connection refused", "segfault at", "kernel panic"], [14] * 3, {}, (2, 4, False, 0)))
    out.append(("tuned_mixed_fold", mixed_folded, [15] * len(mixed_folded), {}, (2, 4, True, 2)))
    # every configuration compiles a pattern set of its own: the engine caches tables per database and sample, not per switch
    return [(name, pats + [f"kq{name.replace('_', 'q')}kq"], flags + [flags[0]], env, inst) for name, pats, flags, env, inst in out]


K1_CONFIGS = _k1_configs()


def instantiation(tables: K1Tables, env: dict) -> tuple:
    """The k_stream template arguments the engine launches for these tables (engine_upload_prefilter, launch_stream_m)."""
    exact = env.get("GPUGREP_FILTER") == "exact" and tables.exact_mode_possible()
    nodd = min(len(tables.odd), 2)
    return (1 if exact else 2, tables.stride, tables.fold, nodd if not exact else 0)


# ---- random factor sets on the fast path -----------------------------------------------------------------------------------
STEMS = ["alphabet", "bravados", "charlie7", "deltoids", "echoing_", "foxtrots", "golfball", "hotelier", "indiana_", "kilogram",
         "limerick", "mikado_w", "november", "operetta", "papayas_", "rebounds"]
BUFFER_SIZES = [4096, 4097, 8191, 8192, 16384, 65536, 262139, 262140, 1 << 20]
SWITCHES = ["", "GPUGREP_VERIFY=v1", "GPUGREP_NO_REPROBE=1", "GPUGREP_MAX_DFA_STATES=60", "GPUGREP_FILTER=exact", "GPUGREP_NO_MIXED_STRIDE=1",
            "GPUGREP_NO_EXT_CONFIRM=1"]


def _core(rng: random.Random) -> str:
    core = rng.choice(STEMS)[: rng.choice([4, 5, 6, 7, 8])]
    if rng.random() < 0.25:
        core += rng.choice([" ", "_", "-"]) + rng.choice(STEMS)[: rng.randint(2, 5)]
    return core


def fast_factor_pattern(rng: random.Random) -> tuple[str, list[str]]:
    """(pattern, literal pieces that a match needs): classes around a literal, \\b, ^ / $, alternated factors, gaps that
    exceed the DFA budget (NFA fallback)."""
    roll = rng.random()
    if roll < 0.08:
        a, b = _core(rng), _core(rng)
        gap = rng.choice([100, 150])
        return f"{a} .{{{gap}}}{b}", [a + " " + "".join(rng.choice("qjxz0189 ") for _ in range(gap)) + b]
    if roll < 0.25:
        a, b = _core(rng), _core(rng)
        body, pieces = f"(?:{a}|{b})", [a, b]
    else:
        a = _core(rng)
        body, pieces = a, [a]
    pre = rng.choice(["", "", "", "^", r"\b", "[a-z]", r"\w+", ".*", "[0-9]{1,3}", "(?:x|y_)", "[ -]", r"\s"])
    suf = rng.choice(["", "", "", "$", r"\b", "[0-9]", r"\s", "s?", ".x", "[^a]", r"\d{1,2}", "[A-Z]"])
    return pre + body.replace(" ", "[ ]") + suf, pieces


def fast_case(seed: int) -> dict:
    """One random fast-path case: a factor set, a text of 0.5-8 MiB with the factors planted at every alignment, a
    buffer_size, and a switch for the second run."""
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    sm_id = rng.choice([0, 7])
    caseless = rng.random() < 0.3
    if rng.random() < 0.1:   # a large caseless set: folded tables
        pats = words(seed, 300, rng.choice([6, 8, 9]))
        pieces = [[w] for w in pats]
        flags = [15] * len(pats)
    else:
        k = rng.choice([1, 2, 3, 4, 6])
        made = [fast_factor_pattern(rng) for _ in range(k)]
        pats = [p for p, _ in made]
        pieces = [pc for _, pc in made]
        flags = [rng.choice([15, 15, 11]) if caseless else rng.choice([14, 14, 10, 12, 8]) for _ in pats]
    buffer_size = BUFFER_SIZES[seed % len(BUFFER_SIZES)]
    general_ok = rng.random() < 0.15   # some texts also get lines that are too long for the fast path
    size = rng.choice([512 << 10, 512 << 10, 1 << 20, 1 << 20, 2 << 20, 4 << 20, 8 << 20])
    longest = 16384 if general_ok else min(16384, super_block_bytes(buffer_size))
    # line lengths: under 16 bytes, about the look-back, ordinary, long
    kinds = nrng.choice(4, size=size // 40 + 16, p=[0.3, 0.3, 0.37, 0.03])
    lengths = np.where(kinds == 0, nrng.integers(1, 16, kinds.size),
                       np.where(kinds == 1, nrng.integers(8, 72, kinds.size),
                                np.where(kinds == 2, nrng.integers(60, 400, kinds.size), nrng.integers(2048, longest + 1, kinds.size))))
    ends = np.cumsum(lengths)
    ends = ends[ends <= size]
    size = int(ends[-1]) if ends.size else size
    buf = BACKGROUND[nrng.integers(0, BACKGROUND.size, size)]
    buf[ends - 1] = 10
    # plants: one every ~700 bytes at random offsets (every alignment), in random case for caseless patterns
    nplants = max(4, size // 700)
    at = np.sort(nrng.integers(0, max(1, size - 300), nplants))
    for p in at.tolist():
        piece = rng.choice(rng.choice(pieces))
        if caseless or flags[0] & 1:
            piece = "".join(ch.upper() if rng.random() < 0.5 else ch for ch in piece)
        ctx = rng.choice(["", " ", "x", "_", "7", "A", "\n"])
        blob = (ctx + piece + rng.choice(["", " ", "s", "9", "Q", "x", "\n", "b "])).encode("latin1")
        if rng.random() < 0.02:   # a NUL before or after the plant
            blob = b"\0" + blob if rng.random() < 0.5 else blob + b"\0"
        buf[p:p + len(blob)] = np.frombuffer(blob, dtype=np.uint8)[: size - p]
    if rng.random() < 0.25:
        buf[-1] = ord("q")   # no final newline
    data = _no_all_nul_pseudo_lines(buf.tobytes(), buffer_size)
    return {"seed": seed, "patterns": pats, "flags": flags, "ids": [sm_id] * len(pats), "buffer_size": buffer_size, "data": data,
            "switch": SWITCHES[(seed // len(BUFFER_SIZES)) % len(SWITCHES)] if seed % 2 else SWITCHES[seed % len(SWITCHES)],
            "general_ok": general_ok}


def _no_all_nul_pseudo_lines(data: bytes, buffer_size: int) -> bytes:
    """The reference reads stale buffer bytes for a pseudo-line made only of NULs (parity.has_all_nul_pseudo_line): such
    lines get a visible byte."""
    if not parity.has_all_nul_pseudo_line(data, buffer_size):
        return data
    out = bytearray(data)
    pos, lim = 0, buffer_size - 1
    while pos < len(out):
        nl = out.find(b"\n", pos, pos + lim)
        end = nl + 1 if nl >= 0 else min(len(out), pos + lim)
        if out[pos] == 0 and not bytes(out[pos:end]).strip(b"\0"):
            out[pos] = ord("q")
        pos = end
    return bytes(out)


def tagged(case: dict, switch: str) -> tuple[list, list, list]:
    """The case's pattern set plus one literal that never occurs in the text, unique to `switch` (the engine caches
    tables per database, so each switch must compile a set of its own)."""
    tag = "kq" + "".join(ch for ch in switch if ch.isalnum()).lower()[-14:] + "qk"
    assert tag.encode() not in case["data"].lower()
    return case["patterns"] + [tag], case["flags"] + [case["flags"][0]], case["ids"] + [case["ids"][0]]


def switch_env(switch: str) -> dict:
    if not switch:
        return {}
    name, value = switch.split("=")
    return {name: value}


def predict(lib, patterns, flags, ids, env: dict, data: bytes, buffer_size: int) -> dict:
    """What the engine does with this case (slot_submit): fast path or not, the k_stream instantiation, whether k_confirm
    runs, and which verification kernel."""
    with environment(env):
        db = CompiledDb(lib, patterns, flags, ids)
        assert db.rc == 0, (patterns, db.error)
        info = db.info
        nfa = info.patterns - sum(g[0].members for g in db.groups)
        out = {"db": db, "nfa": nfa, "groups": info.groups, "simple": bool(info.simple), "prefilter": bool(info.prefilter)}
        if not (info.simple and info.prefilter and super_block_bytes(buffer_size)):
            out.update(fast=False, path=2)
            return out
        if len(data) >= 4096 and "GPUGREP_NO_TUNE" not in env:
            db.retune(data[: 512 << 10])
        tables = K1Tables(db)
    inst = instantiation(tables, env)
    fast = nfa == 0 or inst[0] == 2
    out.update(tables=tables, inst=inst, fast=fast)
    if not fast:
        out["path"] = 2
        return out
    bloom_false_rate = info.prefilter_grams * (16.0 / tables.stride) / (1 << tables.log2_bits)
    want_reprobe = info.groups >= 2 or bloom_false_rate > 0.005 or nfa > 0
    confirm = inst[0] == 2 and want_reprobe and (nfa > 0 or "GPUGREP_NO_REPROBE" not in env)
    lookback = info.prefilter_lookback
    smem_table = False
    if info.groups == 1:
        gi = db.groups[0][0]
        ctab = gi.states * (gi.classes + 2) * 2
        smem_table = gi.classes + 2 <= 255 and (ctab + 15) // 16 * 16 + (gi.states + 15) // 16 * 16 <= 112 << 10
    if env.get("GPUGREP_VERIFY") != "v1" and smem_table and not confirm and lookback <= 64:
        verify = "smem"
    else:
        verify = ("local_nfa" if nfa else "local") + ("+confirm" if confirm else "")
    out.update(confirm=confirm, verify=verify,
               path=2 if has_newline_free_super_block(data, super_block_bytes(buffer_size)) else 1)
    return out
