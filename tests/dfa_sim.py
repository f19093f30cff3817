"""Test-only CPU walker for the tables the pattern compiler emits (never used by the product).

It loads a compiled database through the introspection entry points of include/gpugrep.h and walks the DFA
groups over pseudo-lines with the same rules the CUDA kernels implement, so the compiler can be checked against
the oracle on a machine without a GPU.
"""

from __future__ import annotations

import ctypes
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class DbInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint) for n in (
        "patterns", "groups", "simple", "simple_id", "prefilter", "prefilter_stride", "prefilter_fold",
        "prefilter_log2_bits", "prefilter_grams", "prefilter_min_factor", "prefilter_lookback", "total_states", "reserved")]


class GroupInfo(ctypes.Structure):
    _fields_ = [("states", ctypes.c_uint), ("classes", ctypes.c_uint), ("stride", ctypes.c_uint),
                ("first_accept", ctypes.c_uint), ("sink_match", ctypes.c_int), ("dead", ctypes.c_int),
                ("accept_sets", ctypes.c_uint), ("members", ctypes.c_uint), ("entry_mid_other", ctypes.c_uint),
                ("entry_mid_word", ctypes.c_uint), ("idle_end", ctypes.c_uint), ("reserved", ctypes.c_uint)]


def marshal(patterns, flags=None, ids=None):
    n = len(patterns)
    flags = list(flags) if flags else [14] * n
    ids = list(ids) if ids else [0] * n
    pa = (ctypes.c_char_p * n)(*[p if isinstance(p, bytes) else p.encode() for p in patterns])
    fa = (ctypes.c_uint * n)(*flags)
    ia = (ctypes.c_uint * n)(*ids)
    return pa, fa, ia, n


class CompiledDb:
    def __init__(self, lib: ctypes.CDLL, patterns, flags=None, ids=None):
        self.lib = lib
        lib.gpugrep_db_compile.restype = ctypes.c_void_p
        lib.gpugrep_last_error.restype = ctypes.c_char_p
        lib.gpugrep_db_prefilter_note.restype = ctypes.c_char_p
        lib.gpugrep_db_prefilter_note.argtypes = [ctypes.c_void_p]
        lib.gpugrep_db_copy_prefilter.restype = ctypes.c_size_t
        pa, fa, ia, n = marshal(patterns, flags, ids)
        rc = ctypes.c_int(0)
        self.handle = lib.gpugrep_db_compile(pa, fa, ia, n, ctypes.byref(rc))
        self.rc = rc.value
        self.error = lib.gpugrep_last_error().decode()
        self.groups = []
        self.depths = []   # per group: depth[state] (see automata.hpp)
        if not self.handle:
            return
        h = ctypes.c_void_p(self.handle)
        self.info = DbInfo()
        lib.gpugrep_db_get_info(h, ctypes.byref(self.info))
        for g in range(self.info.groups):
            gi = GroupInfo()
            lib.gpugrep_db_get_group(h, g, ctypes.byref(gi))
            cls = np.zeros(256, dtype=np.uint8)
            trans = np.zeros(gi.states * gi.stride, dtype=np.uint32)
            acc = np.zeros(gi.states, dtype=np.uint32)
            lib.gpugrep_db_copy_group(h, g, cls.ctypes.data_as(ctypes.c_void_p), trans.ctypes.data_as(ctypes.c_void_p),
                                      acc.ctypes.data_as(ctypes.c_void_p))
            reports = []
            for k in range(gi.accept_sets):
                ids_buf = (ctypes.c_uint * 4096)()
                sm_buf = (ctypes.c_uint * 4096)()
                cnt = lib.gpugrep_db_accept_reports(h, g, k, ids_buf, sm_buf, 4096)
                reports.append([(ids_buf[i], sm_buf[i]) for i in range(cnt)])
            self.groups.append((gi, cls, trans.reshape(gi.states, gi.stride), acc, reports))
            lib.gpugrep_db_copy_depth.restype = ctypes.c_size_t
            lib.gpugrep_db_copy_depth.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_void_p, ctypes.c_size_t]
            depth = np.zeros(gi.states, dtype=np.uint8)
            assert lib.gpugrep_db_copy_depth(h, g, depth.ctypes.data_as(ctypes.c_void_p), gi.states) == gi.states
            self.depths.append(depth)
        self.prefilter_note = lib.gpugrep_db_prefilter_note(h).decode()
        self._load_grams()

    def retune(self, sample: bytes) -> None:
        """Re-choose the prefilter windows against a text sample (what the scan entry points do with their input)."""
        self.lib.gpugrep_db_tune.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
        self.lib.gpugrep_db_tune(ctypes.c_void_p(self.handle), sample, len(sample))
        self.lib.gpugrep_db_get_info(ctypes.c_void_p(self.handle), ctypes.byref(self.info))
        self.prefilter_note = self.lib.gpugrep_db_prefilter_note(ctypes.c_void_p(self.handle)).decode()
        self._load_grams()

    def _load_grams(self) -> None:
        lib = self.lib
        h = ctypes.c_void_p(self.handle)
        self.grams = None
        self.odd = []
        if self.info.prefilter:
            lib.gpugrep_db_copy_grams.restype = ctypes.c_size_t
            count = lib.gpugrep_db_copy_grams(h, None, 0)
            grams = np.zeros(count, dtype=np.uint32)
            lib.gpugrep_db_copy_grams(h, grams.ctypes.data_as(ctypes.c_void_p), count)
            self.grams = set(int(g) for g in grams)
            lib.gpugrep_db_copy_odd_compares.restype = ctypes.c_size_t
            lib.gpugrep_db_copy_odd_compares.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
            pairs = (ctypes.c_uint32 * 8)()
            count = lib.gpugrep_db_copy_odd_compares(h, pairs, 4)
            self.odd = [(int(pairs[2 * k]), int(pairs[2 * k + 1])) for k in range(count)]

    def __del__(self):
        if getattr(self, "handle", None):
            self.lib.gpugrep_db_free(ctypes.c_void_p(self.handle))
            self.handle = None

    # ---- line semantics shared with the kernels ----
    @staticmethod
    def block_of(pseudo_line: bytes) -> bytes:
        """Leading NULs stripped, cut at the next NUL (reference hyperscanner.c:205-217)."""
        i = 0
        while i < len(pseudo_line) and pseudo_line[i] == 0:
            i += 1
        rest = pseudo_line[i:]
        cut = rest.find(b"\0")
        return rest if cut < 0 else rest[:cut]

    def events(self, block: bytes):
        """All (end_offset, id, singlematch) reports of a block, unordered."""
        out = []
        for gi, cls, trans, acc, reports in self.groups:
            s = 0
            for pos, b in enumerate(block):
                s = int(trans[s, cls[b]])
                a = int(acc[s])
                if a:
                    for rid, sm in reports[a]:
                        out.append((pos, rid, sm))   # match ended just before byte `pos`
                    if gi.sink_match >= 0 and s == gi.sink_match:
                        break
                if s == gi.dead:
                    break
            else:
                s = int(trans[s, gi.classes])
                a = int(acc[s])
                if a:
                    for rid, sm in reports[a]:
                        out.append((len(block), rid, sm))
        return out

    def line_reports(self, pseudo_line: bytes):
        """Ordered ids delivered for one pseudo-line (dedupe per (id,end); SINGLEMATCH ids once)."""
        block = self.block_of(pseudo_line)
        evs = sorted(set(self.events(block)))
        if self.info.simple:
            return [self.info.simple_id] if evs else []
        seen = set()
        out = []
        for end, rid, sm in evs:
            if sm:
                if rid in seen:
                    continue
                seen.add(rid)
            out.append(rid)
        return out

    def gram_hit(self, gram: int, offset: int) -> bool:
        """What the streaming kernel tests at text offset `offset` (gram already case-folded if the table is)."""
        st = self.info.prefilter_stride
        if offset % st == 0 and gram in self.grams:
            return True
        if self.odd and offset % 4 == 2:   # mixed sampling: register compares between the table lookups
            return any((gram * mul + add) & 0xFFFFFFFF == 0 for mul, add in self.odd)
        return False

    def prefilter_hits(self, text: bytes) -> bool:
        """True if some sampled 4-gram of `text` hits at EVERY alignment of the sampling grid (superset test)."""
        if self.grams is None:
            return True
        fold = 0x20202020 if self.info.prefilter_fold else 0
        for phase in range(4):
            if not any(self.gram_hit(int.from_bytes(text[q:q + 4], "little") | fold, q + phase)
                       for q in range(0, max(0, len(text) - 3))):
                return False
        return True


def _is_word(b: int) -> bool:
    return (48 <= b <= 57) or (65 <= b <= 90) or (97 <= b <= 122) or b == 95


def prefilter_flagged_chunks(db: "CompiledDb", data: bytes) -> set:
    """16-byte chunks (index = offset >> 4) in which a sampled gram starting below len(data) is one of the exact grams
    (bytes past the end read as NUL)."""
    st = db.info.prefilter_stride
    fold = 0x20202020 if db.info.prefilter_fold else 0
    flagged = set()
    for q in range(0, len(data), 2 if db.odd else st):
        gram = int.from_bytes(data[q:q + 4].ljust(4, b"\0"), "little") | fold
        if db.gram_hit(gram, q):
            flagged.add(q >> 4)
    return flagged


def fast_path_matched_line_starts(db: "CompiledDb", data: bytes) -> set:
    """CPU model of the fast path (simple mode): gram hits flag 16-byte chunks; every flagged chunk is verified by a
    LOCAL DFA walk that starts `lookback` bytes before the chunk (or at the line start if that is nearer), treats NUL
    as end-of-data + restart, follows lines that start inside the chunk and stops once the automaton is idle past
    the chunk.  Lines containing NUL are re-checked exactly.  Returns the start offsets of the matched lines."""
    n = len(data)
    lookback = db.info.prefilter_lookback
    flagged = prefilter_flagged_chunks(db, data)
    marked = set()
    for c in sorted(flagged):
        o = c * 16
        lo = 0 if lookback == 0xFFFFFFFF else max(0, o - lookback) & ~3   # the kernel starts on a word boundary
        nl = data.rfind(b"\n", lo, o)
        if lookback == 0xFFFFFFFF:
            nl = data.rfind(b"\n", 0, o)
        t = nl + 1 if nl >= 0 else lo
        # a '\n' right before the start of the walk: the line begins exactly at t (walk_local checks data[t - 1])
        at_line_start = nl >= 0 or lo == 0 or data[t - 1] == 10
        line_start = data.rfind(b"\n", 0, o) + 1   # bookkeeping for the model only
        states = []
        for gi, cls, trans, acc, reports in db.groups:
            if at_line_start:
                states.append(0)
            else:
                states.append(gi.entry_mid_word if _is_word(data[t - 1]) else gi.entry_mid_other)
        pos = t
        cur_line = line_start
        done_line = False
        while pos < n:
            b = data[pos]
            if not done_line:
                if b == 0:
                    hit = False
                    for k, (gi, cls, trans, acc, reports) in enumerate(db.groups):
                        s = int(trans[states[k], gi.classes])
                        hit |= s >= gi.first_accept
                        states[k] = 0
                    if hit:
                        marked.add(cur_line)
                        done_line = True
                else:
                    hit = False
                    for k, (gi, cls, trans, acc, reports) in enumerate(db.groups):
                        s = int(trans[states[k], cls[b]])
                        if s >= gi.first_accept:
                            hit = True
                        states[k] = s
                    if not hit and b == 10:
                        for k, (gi, cls, trans, acc, reports) in enumerate(db.groups):
                            if int(trans[states[k], gi.classes]) >= gi.first_accept:
                                hit = True
                    if hit:
                        marked.add(cur_line)
                        done_line = True
            pos += 1
            if b == 10:
                if pos >= o + 16 or pos >= n:
                    break
                cur_line = pos
                done_line = False
                states = [0] * len(db.groups)
                continue
            # past the last sampled gram of the chunk the walk stops as soon as nothing that is still in progress can have begun at
            # or before that gram (automata.hpp Dfa::depth; the kernels test this once per word, the model per byte)
            ifrom = o + (18 if db.odd else 20 - db.info.prefilter_stride)
            if pos >= ifrom and (done_line or all(int(db.depths[k][states[k]]) < min(pos - ifrom + 4, 255) for k in range(len(db.groups)))):
                break
            if done_line and pos >= o + 16:
                break
        else:
            if not done_line:
                for k, (gi, cls, trans, acc, reports) in enumerate(db.groups):
                    if int(trans[states[k], gi.classes]) >= gi.first_accept:
                        marked.add(cur_line)
    # exact re-check of marked lines that contain NUL bytes
    out = set()
    for ls in marked:
        end = data.find(b"\n", ls)
        line = data[ls:end + 1] if end >= 0 else data[ls:]
        if b"\0" in line:
            if db.line_reports(line):
                out.add(ls)
        else:
            out.add(ls)
    return out


def split_pseudo_lines(data: bytes, buffer_size: int):
    """gzgets() splitting (reference hyperscanner.c:199): up to buffer_size-1 bytes, stop after '\\n'."""
    out = []
    pos = 0
    lim = buffer_size - 1
    n = len(data)
    while pos < n:
        nl = data.find(b"\n", pos, pos + lim)
        end = nl + 1 if nl >= 0 else min(n, pos + lim)
        out.append(data[pos:end])
        pos = end
    return out
