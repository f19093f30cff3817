// Fixed-string kernels (grep -F, gpugrep_literal_scan_*): a line is selected when its scanned block holds one of the
// literals.  No automaton: a text position is compared byte for byte against the literals that can start there.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
//
// The kept literals are prefix-free per class (database.hpp LiteralSet), so at a text position at most one literal of a
// class can match - the largest one that is not above the text - and a sorted run of literals is binary-searched.
//  - fast path: k_verify_literals replaces the DFA verification.  Each gram hit that k_confirm found again is looked up
//    in the literal index (Prefilter::lit_begin): one binary search per (class, offset) run of the gram's entries.
//  - general path and the NUL re-check of the emit kernel: every position of the scanned block is looked up by its first
//    two bytes (LiteralView::bucket) and binary-searched there; one-byte literals are a bitmap.
#pragma once

namespace gpugrep {

struct LiteralView {
    const uint8_t* __restrict__ bytes;    // the literals, caseless ones folded (A-Z -> a-z)
    const uint32_t* __restrict__ off;     // per literal: offset into bytes
    const uint32_t* __restrict__ len;     // per literal: length
    const uint32_t* __restrict__ order;   // literals of >= 2 bytes, by class, then in byte order
    const uint32_t* __restrict__ bucket;  // [class * 65537 + (b0 << 8 | b1)]: range of `order` with that two-byte prefix
    const uint32_t* __restrict__ one;     // [class * 8 + b / 32]: one-byte literals
    uint32_t classes;                     // bit c: class c (0 exact, 1 caseless) has literals
};

// Literal index of a sample-tuned prefilter (Prefilter::lit_begin / lit_entries) next to its confirm table.
struct LiteralIndex {
    const uint32_t* __restrict__ begin;             // per confirm slot, + 1
    const unsigned long long* __restrict__ entries; // (class << 31 | offset) << 32 | literal
};

__device__ __forceinline__ uint32_t lit_norm(uint32_t b, uint32_t cls) { return cls && b - 'A' < 26u ? b | 0x20u : b; }

// Literal `id` of class `cls` against the text at x (the text ends at lim): -1 literal below the text, 0 literal is a
// prefix of the text (a match), 1 literal above it (a text that ends inside the literal is below it).
// Eight bytes per step where the whole step lies in the text and the class is exact.
__device__ __forceinline__ int lit_compare(const LiteralView& L, uint32_t id, uint32_t cls, const uint8_t* __restrict__ data, size_t x, size_t lim) {
    const uint32_t base = L.off[id], len = L.len[id];
    const uint8_t* __restrict__ p = L.bytes + base;
    uint32_t k = 0;
    if (!cls) {
        // (the literal bytes are padded by 16 on the device: the aligned form of the load stays inside the array)
        for (; k + 8 <= len && x + k + 16 <= lim; k += 8) {
            const unsigned long long t = load64_unaligned(data, x + k, lim), l = load64_unaligned(L.bytes, base + k, base + len + 8);
            if (t != l) {
                const uint32_t at = (uint32_t)(__ffsll((long long)(t ^ l)) - 1) >> 3;   // first differing byte (little endian)
                return ((l >> (8 * at)) & 0xffu) < ((t >> (8 * at)) & 0xffu) ? -1 : 1;
            }
        }
    }
    for (; k < len; k++) {
        if (x + k >= lim) return 1;
        const uint32_t t = lit_norm(data[x + k], cls), l = p[k];
        if (l != t) return l < t ? -1 : 1;
    }
    return 0;
}

// Does a literal of `ids[lo, hi)` (one class, byte order, prefix-free) match at x?
template <class Ids>
__device__ __forceinline__ bool lit_search(const LiteralView& L, const Ids& ids, uint32_t lo, uint32_t hi, uint32_t cls, const uint8_t* __restrict__ data,
                                           size_t x, size_t lim) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const int c = lit_compare(L, ids(mid), cls, data, x, lim);
        if (c == 0) return true;
        if (c < 0) lo = mid + 1;
        else hi = mid;
    }
    return false;
}

// Does some literal start at x (x < lim)?
__device__ __forceinline__ bool lit_match_at(const LiteralView& L, const uint8_t* __restrict__ data, size_t x, size_t lim) {
    const uint32_t b0 = data[x], b1 = x + 1 < lim ? data[x + 1] : 0u;
    for (uint32_t cls = 0; cls < 2; cls++) {
        if (!((L.classes >> cls) & 1u)) continue;
        const uint32_t n0 = lit_norm(b0, cls);
        if ((L.one[cls * 8 + (n0 >> 5)] >> (n0 & 31u)) & 1u) return true;
        if (x + 1 >= lim) continue;
        const uint32_t key = cls * 65537u + (n0 << 8 | lit_norm(b1, cls));
        const uint32_t lo = L.bucket[key], hi = L.bucket[key + 1];
        if (lo < hi && lit_search(L, [&](uint32_t k) { return L.order[k]; }, lo, hi, cls, data, x, lim)) return true;
    }
    return false;
}

// The scanned block of [start, lim) (leading NULs skipped, cut at the next NUL) holds a literal?  A literal holds no NUL,
// so no occurrence that starts in front of the cut reaches past it.
__device__ bool block_matches_literal(const LiteralView& L, const uint8_t* __restrict__ data, size_t start, size_t lim) {
    for (size_t x = skip_leading_nuls(data, start, lim); x < lim && data[x] != 0; x++)
        if (lit_match_at(L, data, x, lim)) return true;
    return false;
}

// General path: one thread per pseudo-line, like k_match_pl_simple.
__global__ void __launch_bounds__(128) k_match_pl_literals(LiteralView L, const uint8_t* __restrict__ data, const uint32_t* __restrict__ pl_start,
                                                           const uint32_t* __restrict__ pl_len, size_t npl, uint8_t* __restrict__ flags, bool invert) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl) return;
    const size_t st = pl_start[i];
    flags[i] = block_matches_literal(L, data, st, st + pl_len[i]) != invert ? 1 : 0;   // invert: select the lines without a match
}

// Fast path: the verification of the candidates k_confirm kept (survivor list, gram hits in hitinfo), in place of
// k_verify_local.  Per hit q: the gram's confirm slot, then per (class, offset) run of its index entries one binary search
// of the text at q - offset.  A match marks the line that holds its first byte, which is also the line of q (a literal has
// no '\n' before its last byte): bit j = the j-th line that intersects the chunk.  Lines with NUL bytes are re-checked by
// the emit kernel (block_matches_literal), as with the DFA verifiers.
__global__ void __launch_bounds__(128) k_verify_literals(LiteralView L, LiteralIndex X, ReprobeParams rp, const uint8_t* __restrict__ data, size_t n,
                                                         const uint32_t* __restrict__ cand, const unsigned long long* __restrict__ hitinfo,
                                                         const uint32_t* __restrict__ survivors, const Totals* totals, uint32_t* __restrict__ marks,
                                                         uint32_t* __restrict__ tile_records) {
    const size_t count = (size_t)totals->survivors;
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += (size_t)gridDim.x * blockDim.x) {
        const size_t i = survivors[j];
        const size_t o = (size_t)cand[i] * 16;
        uint32_t hits = (uint32_t)(hitinfo[i] >> 32);
        const uint32_t nlm = newline_mask16(ld_chunk(data, o, n));
        uint32_t mask = 0;
        while (hits) {
            const uint32_t at = __ffs(hits) - 1;
            hits &= hits - 1;
            const size_t q = o + at;
            uint32_t gram = 0;
            for (uint32_t k = 0; k < 4 && q + k < n; k++) gram |= (uint32_t)data[q + k] << (8 * k);
            if (rp.fold) gram |= 0x20202020u;
            const uint32_t h1 = (gram * rp.mul) >> rp.shift, h2 = rp.half + ((gram * rp.mul2) >> rp.shift);
            const uint32_t slot = rp.keys[h1] == gram ? h1 : (rp.keys[h2] == gram ? h2 : 0xffffffffu);
            if (slot == 0xffffffffu) continue;
            uint32_t b = X.begin[slot];
            const uint32_t e = X.begin[slot + 1];
            while (b < e) {
                const uint32_t key = (uint32_t)(X.entries[b] >> 32);
                uint32_t lo = b + 1, hi = e;   // end of the run: the first entry with a larger key
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if ((uint32_t)(X.entries[mid] >> 32) == key) lo = mid + 1;
                    else hi = mid;
                }
                const uint32_t off = key & 0x7fffffffu, cls = key >> 31;
                if (q >= off) {
                    const size_t x = q - off;
                    const uint32_t bit = x < o ? 1u : 1u << __popc(nlm & ((1u << (uint32_t)(x - o)) - 1u));
                    if (!(mask & bit) && lit_search(L, [&](uint32_t k) { return (uint32_t)X.entries[k]; }, b, lo, cls, data, x, n)) mask |= bit;
                }
                b = lo;
            }
        }
        marks[i] = mask;
        if (mask) atomicAdd(&tile_records[i / kEmitTile], (uint32_t)__popc(mask));
    }
}

}  // namespace gpugrep
