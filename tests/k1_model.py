"""Test-only CPU model of K1, the streaming kernel (hypergrep_b200/csrc/k_stream.cuh): which 16-byte chunks it flags as
candidates and how many newlines it counts, for the gram tables of a compiled database (tests/dfa_sim.CompiledDb).

The kernel reads every byte at offset >= n as 0 (ld_chunk), looks up the 4-byte gram at every sampled offset q of the
chunks that start below n, and flags the chunk of q on a hit:
  - bloom mode (the default): p = gram * bloom_mul; bit (p & 7) of byte p >> (32 - (log2_bits - 3)) of the bitmap;
  - exact mode (GPUGREP_FILTER=exact, only for tables without odd compares): the gram is one of the database's grams;
  - mixed sampling (odd compares, bloom mode only): also gram * mul + add == 0 at q = 2 (mod 4).
Grams are OR-ed with 0x20202020 when the table is folded, the odd compares included.  Table lookups sample q = 0
(mod stride).  Vectorised with numpy: 64 MiB take a few seconds.
"""

from __future__ import annotations

import ctypes

import numpy as np

_PIECE = 8 << 20   # bytes modelled per step (bounds the temporaries)


class K1Tables:
    """The streaming kernel's view of a compiled database's prefilter."""

    def __init__(self, db):
        info = db.info
        assert info.prefilter, "the database has no prefilter"
        lib = db.lib
        lib.gpugrep_db_copy_prefilter.restype = ctypes.c_size_t
        lib.gpugrep_db_copy_prefilter.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_uint32)]
        h = ctypes.c_void_p(db.handle)
        mul = ctypes.c_uint32(0)
        words = lib.gpugrep_db_copy_prefilter(h, None, 1 << 30, ctypes.byref(mul))
        bitmap = np.zeros(words, dtype=np.uint32)
        assert lib.gpugrep_db_copy_prefilter(h, bitmap.ctypes.data_as(ctypes.c_void_p), words, ctypes.byref(mul)) == words
        self.bitmap = bitmap.view(np.uint8)
        self.log2_bits = int(words * 32).bit_length() - 1
        assert 1 << self.log2_bits == words * 32
        self.bloom_mul = int(mul.value)
        self.grams = np.array(sorted(db.grams), dtype=np.uint32)
        self.odd = list(db.odd)
        self.stride = int(info.prefilter_stride)
        self.fold = bool(info.prefilter_fold)
        self.exact_table = bool(info.reserved)   # the exact two-choice table exists (GPUGREP_FILTER=exact can use it)
        self.log2_slots = int(info.prefilter_log2_bits) if self.exact_table else 0

    def exact_mode_possible(self) -> bool:
        """GPUGREP_FILTER=exact takes the exact table only when there is one and no odd compares (engine_upload_prefilter)."""
        return self.exact_table and not self.odd

    def bloom_hit(self, grams: np.ndarray) -> np.ndarray:
        p = grams * np.uint32(self.bloom_mul)
        byte = p >> np.uint32(32 - (self.log2_bits - 3))
        return ((self.bitmap[byte] >> (p & np.uint32(7)).astype(np.uint8)) & 1).astype(bool)

    def exact_hit(self, grams: np.ndarray) -> np.ndarray:
        if self.grams.size == 0:
            return np.zeros(grams.shape, dtype=bool)
        at = np.minimum(np.searchsorted(self.grams, grams), self.grams.size - 1)
        return self.grams[at] == grams

    def odd_hit(self, grams: np.ndarray) -> np.ndarray:
        hit = np.zeros(grams.shape, dtype=bool)
        for mul, add in self.odd:
            hit |= grams * np.uint32(mul) + np.uint32(add) == 0
        return hit


def _grams_at(buf: np.ndarray, q: np.ndarray, fold: bool) -> np.ndarray:
    g = buf[q].astype(np.uint32)
    g |= buf[q + 1].astype(np.uint32) << np.uint32(8)
    g |= buf[q + 2].astype(np.uint32) << np.uint32(16)
    g |= buf[q + 3].astype(np.uint32) << np.uint32(24)
    if fold:
        g |= np.uint32(0x20202020)
    return g


def k1_candidates(data, tables: K1Tables, exact: bool = False):
    """(newlines in data, sorted array of the chunk indices K1 flags) for the first len(data) bytes.  `exact`: exact mode."""
    text = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    n = int(text.size)
    newlines = int(np.count_nonzero(text == 10))
    nchunks = (n + 15) // 16
    out = []
    for c0 in range(0, nchunks, _PIECE // 16):
        c1 = min(nchunks, c0 + _PIECE // 16)
        lo, hi = c0 * 16, c1 * 16
        buf = np.zeros(hi - lo + 4, dtype=np.uint8)   # bytes at or past n read as 0
        take = min(n, hi + 4) - lo
        buf[:take] = text[lo:lo + take]
        hit = np.zeros(c1 - c0, dtype=bool)
        q = np.arange(0, hi - lo, tables.stride, dtype=np.int64)
        grams = _grams_at(buf, q, tables.fold)
        found = tables.exact_hit(grams) if exact else tables.bloom_hit(grams)
        hit[q[found] >> 4] = True
        if tables.odd:
            q = np.arange(2, hi - lo, 4, dtype=np.int64)
            found = tables.odd_hit(_grams_at(buf, q, tables.fold))
            hit[q[found] >> 4] = True
        out.append(np.flatnonzero(hit) + c0)
    chunks = np.concatenate(out) if out else np.zeros(0, dtype=np.int64)
    return newlines, chunks


def stream_sweep_bytes(tables: K1Tables, sms: int, exact: bool = False) -> int:
    """Bytes that the persistent grid of K1 covers in one sweep (slot_submit: shared memory of the table -> CTAs per SM
    and threads per CTA; each warp takes four 512-byte blocks per step)."""
    if exact:
        slots = 1 << tables.log2_slots
        rshift = 5
        while rshift > 0 and (3 * slots * 4) << rshift > 200 * 1024:
            rshift -= 1
        copies = 1 << rshift
        smem = 2 * slots * copies * 4 + slots * copies * 4
    else:
        smem = (1 << tables.log2_bits) // 8
    block = 1024 if smem > 32 * 1024 else 256
    ctas = 1 if smem > 100 * 1024 else (2 if smem > 32 * 1024 else 6)
    return sms * ctas * (block // 32) * 4 * 512


def super_block_bytes(buffer_size: int) -> int:
    """Super-block size of the fast path's long-line check (slot_submit); 0: the fast path is off for this buffer_size."""
    if buffer_size < 4096:
        return 0
    s = 2048
    while s * 4 <= buffer_size and s < 65536:
        s *= 2
    return s


def has_newline_free_super_block(data: bytes, super_bytes: int) -> bool:
    """k_list_candidates flag 1: an aligned super-block that ends inside the last (zero-padded) 512-byte block and holds
    no newline."""
    n = len(data)
    end = (n + 511) // 512 * 512
    text = np.frombuffer(data, dtype=np.uint8)
    nl = np.flatnonzero(text == 10)
    for start in range(0, end - super_bytes + 1, super_bytes):
        k = np.searchsorted(nl, start)
        if k == nl.size or nl[k] >= start + super_bytes:
            return True
    return False
