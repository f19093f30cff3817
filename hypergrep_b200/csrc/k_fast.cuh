// Fast-path kernels: long-line check, candidate list, local verification, record offsets, emit, segment cuts.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
#pragma once

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// FAST PATH kernels
// ------------------------------------------------------------------------------------------------------------
// meta/prefix -> ordered list of candidate chunk indices.  Along the way: flags segments that may contain a line too long
// for the fast path - an aligned super-block of `blocks_per_super` 512-byte blocks (a multiple of kGroupBlocks; 0: no
// check) without any newline.
__global__ void k_list_candidates(const unsigned long long* __restrict__ meta, const unsigned long long* __restrict__ prefix, size_t nblk,
                                  size_t blocks_per_super, const unsigned long long* meta_total, uint32_t* __restrict__ cand, size_t cap,
                                  Totals* totals) {
    const size_t ngroups = (nblk + kGroupBlocks - 1) / kGroupBlocks;
    for (size_t grp = (size_t)blockIdx.x * blockDim.x + threadIdx.x; grp < ngroups; grp += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long before = prefix[grp];
        const size_t first = grp * kGroupBlocks;
        if (blocks_per_super && first % blocks_per_super == 0 && first + blocks_per_super <= nblk) {
            // (a partial trailing super-block cannot hide a full one)
            const size_t hi = first + blocks_per_super;
            const uint32_t b = hi < nblk ? (uint32_t)prefix[hi / kGroupBlocks] : (uint32_t)*meta_total;
            if ((uint32_t)before == b) atomicOr(&totals->flags, 1u);
        }
        size_t at = (size_t)(before >> 32);
        for (size_t g = first; g < nblk && g < first + kGroupBlocks; g++) {
            uint32_t mask = (uint32_t)meta[g];
            while (mask) {
                int b = __ffs(mask) - 1;
                mask &= mask - 1;
                if (at < cap) cand[at] = (uint32_t)(g * 32 + b);
                else atomicOr(&totals->flags, 2u);
                at++;
            }
        }
    }
}

__device__ __forceinline__ bool is_word_dev(uint32_t b) {
    return (b - '0' < 10u) || ((b | 0x20u) - 'a' < 26u) || b == '_';
}

// Transition-table accessors for the local walk.  Both present the same byte-indexed view in which '\n' and NUL are
// ordinary columns and "matched" is one absorbing state (see engine_upload).
struct FlatTable {   // [state][256] u16 in global memory
    const uint16_t* __restrict__ flat;
    const uint8_t* __restrict__ depth;
    __device__ __forceinline__ uint32_t depth_of(uint32_t s) const { return depth[s]; }
    __device__ __forceinline__ uint32_t cls_of(uint32_t b) const { return b; }   // the table is byte-indexed
    __device__ __forceinline__ uint32_t next(uint32_t s, uint32_t c) const { return flat[(s << 8) | c]; }
    __device__ __forceinline__ uint32_t step(uint32_t s, uint32_t b) const { return flat[(s << 8) | b]; }
};
struct SharedTable {   // class-compressed [state][classes] u16 in shared memory + byte -> class map (GroupDev::ctab)
    const uint16_t* tab;
    const uint8_t* cls;
    uint32_t ncls;   // entries per table row
    const uint8_t* depth;
    __device__ __forceinline__ uint32_t depth_of(uint32_t s) const { return depth[s]; }
    // the class lookups do not depend on the state: the walk issues the four of a word first, the state chain is then one
    // multiply-add and one load per byte
    __device__ __forceinline__ uint32_t cls_of(uint32_t b) const { return cls[b]; }
    __device__ __forceinline__ uint32_t next(uint32_t s, uint32_t c) const { return tab[s * ncls + c]; }
    __device__ __forceinline__ uint32_t step(uint32_t s, uint32_t b) const { return tab[s * ncls + cls[b]]; }
};
// Text accessors: aligned words of the segment.
struct GlobalText {
    const uint8_t* __restrict__ data;
    __device__ __forceinline__ uint32_t word(uint32_t wpos) const { return *reinterpret_cast<const uint32_t*>(data + wpos); }
};
// LOCAL verification walk of one DFA group around candidate chunk [o, o+16).
//  - starts at t (at most `lookback` bytes before the chunk, never before the line start) in the start-of-line state
//    or in the mid-line entry state that matches the previous byte;
//  - a NUL acts as end-of-data followed by a restart (lines with NULs are re-checked exactly by the emit kernel);
//  - a '\n' ends the line: the walk continues with the next line only if that line starts inside the chunk;
//  - once past every gram hit of the chunk (idle_from: the end of its last sampled gram, or of the last gram that the
//    verification kernel found again) the walk stops as soon as the automaton is idle: a match that contains a gram hit
//    of this chunk would still be in progress.
// line_bit: bit of the line that contains t (bit j = j-th line intersecting the chunk).
// Returns bit j set if the j-th line intersecting the chunk matched.
// The walk advances one ALIGNED WORD per step:
//  - a full word without a newline is four chained lookups and nothing else (no per-byte tests: a match sticks until
//    the line ends);
//  - a word with a newline, the first word of an unaligned start and the last word of the segment take the byte-wise
//    form, straight-line code without inner loops (threads of a warp diverge here, so it is short).
// The line bit is set when the line ends in the matched state, or at the end of the walk.
template <class Table, class Text>
__device__ __forceinline__ uint32_t walk_words(const Table& T, const Text& X, const GroupDev& G, uint32_t s, uint32_t end, uint32_t cend, uint32_t pos,
                                               uint32_t ifrom, uint32_t line_bit) {
    const uint32_t first_accept = G.first_accept;
    uint32_t mask = 0;
    if (pos >= end) return G.eod_next[s] >= first_accept ? line_bit : 0u;
    // Whole words.  Every lane of the warp runs the SAME four table steps per word; what a newline adds sits in four
    // short guarded blocks (a warp enters one only if some lane has its '\n' at that very byte), and a walk that starts
    // inside its first word (it begins right behind a newline) skips the leading bytes of that word by predicate.  An
    // earlier form took a byte-wise copy of the step for words with a newline and a byte loop for the unaligned start: most
    // warps had to execute those as well, with one or two lanes busy (ncu: 13 of 32 lanes, issue slots 72 % used).
    uint32_t wpos = pos & ~3u;
    if (wpos + 4 <= end) {
        uint32_t skip = pos & 3u;   // bytes of the first word that lie in front of the start
        uint32_t word = X.word(wpos);
        bool over = false;   // the walk ended at a newline whose successor line starts outside the chunk
        while (true) {
            // the next word is requested before the (dependent) table lookups of this one
            const uint32_t next_word = wpos + 8 <= end ? X.word(wpos + 4) : 0u;
            const uint32_t z = eq_mask4(word, 0x0a0a0a0au);
            const uint32_t c0 = T.cls_of(word & 0xffu), c1 = T.cls_of((word >> 8) & 0xffu), c2 = T.cls_of((word >> 16) & 0xffu), c3 = T.cls_of(word >> 24);
#define GPUGREP_WALK_BYTE(K, C, ZBIT)                                   \
            if (skip <= (K)) {                                          \
                s = T.next(s, (C));                                     \
                if (z & (ZBIT)) {                                       \
                    if (s >= first_accept) mask |= line_bit;            \
                    if (wpos + (K) + 1 >= cend) { over = true; break; } \
                    line_bit <<= 1;                                     \
                    s = 0;                                              \
                }                                                       \
            }
            GPUGREP_WALK_BYTE(0u, c0, 0x80u)
            GPUGREP_WALK_BYTE(1u, c1, 0x8000u)
            GPUGREP_WALK_BYTE(2u, c2, 0x800000u)
            GPUGREP_WALK_BYTE(3u, c3, 0x80000000u)
#undef GPUGREP_WALK_BYTE
            skip = 0;
            wpos += 4;
            if (s >= first_accept) {
                if (wpos >= cend) return mask | line_bit;   // matched, and no further line starts inside the chunk
            } else if (wpos >= ifrom && T.depth_of(s) < min(wpos - ifrom + 4u, 255u)) {
                // whatever is still in progress began behind the last gram of the chunk (Dfa::depth): it belongs to a later
                // candidate.  (Before: only when NOTHING was in progress - the longest lane of a warp then walked some 60
                // bytes past its chunk.)
                return mask;
            }
            if (wpos + 4 > end) break;
            word = next_word;
        }
        if (over) return mask;
        pos = wpos;
    }
    // tail: the last (partial) word of the segment, byte by byte
    while (pos < end) {
        const uint32_t b = (X.word(pos & ~3u) >> (8 * (pos & 3u))) & 0xffu;
        s = T.step(s, b);
        if (b == '\n') {
            if (s >= first_accept) mask |= line_bit;
            if (pos + 1 >= cend) return mask;
            line_bit <<= 1;
            s = 0;
        }
        pos++;
        if (s >= first_accept) {
            if (pos >= cend) return mask | line_bit;
        } else if (pos >= ifrom && T.depth_of(s) < min(pos - ifrom + 4u, 255u)) {
            return mask;
        }
    }
    if (s >= first_accept || G.eod_next[s] >= first_accept) mask |= line_bit;
    return mask;
}

// entry state of a walk that starts at t: the byte before the walk decides; a '\n' there means the line starts exactly at t
// (the callers only look for newlines inside [t, o)), so the walk enters in the start-of-line state: ^ and \A see a line start
__device__ __forceinline__ uint32_t entry_state(const GroupDev& G, bool at_line_start, uint32_t before) {
    if (at_line_start || before == '\n') return 0u;
    return is_word_dev(before) ? G.mid_word : G.mid_other;
}

__device__ uint32_t walk_local(const GroupDev& G, const uint8_t* __restrict__ data, size_t n, size_t o, size_t t, bool at_line_start,
                               size_t idle_from, uint32_t line_bit) {
    uint32_t s = entry_state(G, at_line_start, at_line_start ? 0u : data[t - 1]);
    uint32_t mask = 0;
    const size_t chunk_end = o + 16;
    const uint32_t first_accept = G.first_accept, idle_end = G.idle_end;
    if (G.flat) return walk_words(FlatTable{G.flat, G.depth}, GlobalText{data}, G, s, (uint32_t)n, (uint32_t)chunk_end, (uint32_t)t, (uint32_t)idle_from, line_bit);
    bool done = false;
    ByteCursor c(data, t, n);
    while (c.pos < n) {
        const uint32_t b = c.get();
        if (!done) {
            bool hit;
            if (b == 0) {
                hit = G.trans[s * G.stride + G.eod] >= first_accept;
                s = 0;
            } else {
                s = G.trans[s * G.stride + G.cls[b]];
                hit = s >= first_accept;
                if (!hit && b == '\n') hit = G.trans[s * G.stride + G.eod] >= first_accept;
            }
            if (hit) { mask |= line_bit; done = true; }
        }
        c.next();
        if (b == '\n') {
            if (c.pos >= chunk_end || c.pos >= n) return mask;
            line_bit <<= 1;
            done = false;
            s = 0;
            continue;
        }
        if (c.pos >= idle_from && (done || s < idle_end)) return mask;
        if (done && c.pos >= chunk_end) return mask;
    }
    if (!done && G.trans[s * G.stride + G.eod] >= first_accept) mask |= line_bit;
    return mask;
}

// Confirmation of candidate chunks (databases with several DFA groups, large gram sets, NFA-fallback patterns): which
// sampled grams of the chunk are REALLY in the set, and which DFA groups do they lead to?  k_stream only said "some gram
// of this chunk may be".  One thread per candidate:
//  1. the bloom byte table again, from shared memory like in k_stream (8 cheap lookups);
//  2. for the few positions that pass: the exact two-choice gram table in global memory, and - where the factor around
//     the gram is exact - 6 or 8 bytes of text against a second exact table (digit grams like "1234" are everywhere in
//     numeric text, the factor "12345\"" they stand for is not);
//  3. result per candidate: hit offsets (bit = byte offset in the chunk) << 32 | DFA group mask; 0 = dropped.
// The verification kernel then walks only what is left (for the 10,000-pattern set: one candidate in a few hundred).
// Doing this inside the verification kernel (round 1) cost two scattered global loads per sampled gram and candidate.
// (Tried and dropped: a variant that streams the whole text again, one warp per 512-byte block with the candidate lanes
// doing this work - no gather from DRAM, but only a fifth of the lanes are busy in the expensive part: 1.66 -> 3.07 ms
// per GiB for the 10,000-pattern set.  Packing 32 candidates into a warp is what makes this kernel affordable.)
constexpr int kConfirmThreads = 1024;
__global__ void __launch_bounds__(kConfirmThreads, 1) k_confirm(const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ cand,
                                                                const unsigned long long* meta_total, size_t cap, const uint32_t* __restrict__ table,
                                                                int table_words, ProbeParams pp, ReprobeParams rp,
                                                                unsigned long long* __restrict__ hitinfo, uint32_t* __restrict__ marks,
                                                                uint32_t* __restrict__ survivors, Totals* totals) {
    extern __shared__ __align__(16) uint32_t s_bloom[];
    for (int k = threadIdx.x; k < table_words; k += blockDim.x) s_bloom[k] = table[k];
    __syncthreads();
    const uint8_t* s_bytes = reinterpret_cast<const uint8_t*>(s_bloom);
    size_t ncand = (size_t)(*meta_total >> 32);
    if (ncand > cap) ncand = cap;
    // The text of a candidate comes from DRAM (the segment was streamed long ago): the chunk of the NEXT candidate of this
    // thread is requested before the current one is looked at.
    const size_t step = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t o_next = i < ncand ? (size_t)cand[i] * 16 : 0;
    uint4 v_next = ld_chunk(data, o_next, n);
    uint32_t x_next = o_next + 16 < n ? *reinterpret_cast<const uint32_t*>(data + o_next + 16) : 0u;
    for (; (i & ~(size_t)31) < ncand; i += step) {
        const bool live = i < ncand;
        const size_t o = o_next;
        const uint4 v = v_next;
        uint32_t w[5] = {v.x, v.y, v.z, v.w, x_next};
        if (o + 20 > n) w[4] = o + 16 < n ? ld_chunk(data, o + 16, n).x : 0u;   // the last words of the segment: bytes beyond n read as zero
        if (i + step < ncand) {
            o_next = (size_t)cand[i + step] * 16;
            v_next = ld_chunk(data, o_next, n);
            x_next = o_next + 16 < n ? *reinterpret_cast<const uint32_t*>(data + o_next + 16) : 0u;
        } else {
            o_next = 0;
        }
        if (rp.fold) {
#pragma unroll
            for (int k = 0; k < 5; k++) w[k] |= 0x20202020u;
        }
        uint32_t hits = 0, group_mask = 0;
        if (live) confirm_chunk(w, o, s_bytes, pp, rp, data, n, hits, group_mask);
        // The candidates that are left go into a compact list (in no particular order: the verification kernel writes its
        // result by candidate index): few survive for large sets, and a warp of the verification kernel should be full.
        const bool keep = live && hits != 0u;
        if (live) {
            hitinfo[i] = keep ? ((unsigned long long)hits << 32) | group_mask : 0ull;
            if (!keep) marks[i] = 0u;
        }
        const uint32_t alive = __ballot_sync(0xffffffffu, keep);
        if (alive) {
            const uint32_t lane = threadIdx.x & 31;
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(&totals->survivors, (unsigned int)__popc(alive));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (keep) survivors[base + __popc(alive & ((1u << lane) - 1u))] = (uint32_t)i;
        }
    }
}

// One thread per candidate chunk: local verification (see walk_local); writes the bitmask of matched lines.
// With the result of k_confirm at hand (hitinfo), the walk covers [first gram hit - lookback, end of the last gram hit] and
// then runs on until the automaton is idle, only the DFA groups that own the grams are walked, and a chunk without a
// confirmed gram is dropped without a walk.
// WITH_NFA: the database also holds patterns that are simulated as bit-parallel NFAs (their own DFA exceeds the state
// budget).  Their grams carry bit 31 of the group mask; a candidate chunk with such a gram gets every line that
// intersects it checked by the NFA simulation over the whole line (rare, and far cheaper than sending the whole segment
// down the general path because of one such pattern).
template <bool WITH_NFA>
__global__ void __launch_bounds__(128, WITH_NFA ? 8 : 16) k_verify_local(DbView db, const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ cand,
                                                          const unsigned long long* meta_total, size_t cap, uint32_t lookback, uint32_t idle_span,
                                                          const unsigned long long* __restrict__ hitinfo,
                                                          const uint32_t* __restrict__ survivors, const Totals* totals,
                                                          uint32_t* __restrict__ marks, uint32_t* __restrict__ tile_records) {
    size_t ncand = (size_t)(*meta_total >> 32);
    if (ncand > cap) ncand = cap;
    // with a survivor list (k_confirm) the kernel walks that list, in whatever order it has: results go by candidate index
    const size_t count = survivors ? (size_t)totals->survivors : ncand;
    // whole warps stay in the loop (without a survivor list a warp's 32 candidates are consecutive and lie in one emit
    // tile: the records of the tile are counted with one warp reduction and one atomic)
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; (j & ~(size_t)31) < count; j += (size_t)gridDim.x * blockDim.x) {
    uint32_t mask = 0;
    size_t i = j;
    if (j < count) {
    if (survivors) i = survivors[j];
    const size_t o = (size_t)cand[i] * 16;
    size_t t;
    bool at_line_start;
    size_t idle_from = o + idle_span;   // end of the last sampled gram of the chunk
    uint32_t line_bit = 1u;
    uint32_t group_mask = 0xffffffffu;   // DFA groups to walk
    if (lookback == 0xffffffffu) {
        t = line_start_of(data, o);
        at_line_start = true;
    } else {
        size_t hi = o;   // the walk has to start at or before hi - lookback
        uint32_t nl_in_chunk = 0;
        if (hitinfo) {
            const unsigned long long info = hitinfo[i];
            const uint32_t hits = (uint32_t)(info >> 32);
            if (hits == 0) { marks[i] = 0; goto counted; }   // k_confirm found no gram of the set in this chunk
            group_mask = (uint32_t)info;
            const uint32_t first = __ffs(hits) - 1, last = 31 - __clz(hits);
            hi = o + first;
            idle_from = o + last + 4;
            nl_in_chunk = newline_mask16(ld_chunk(data, o, n)) & ((1u << first) - 1u);   // newlines in [o, hi)
        }
        // start: at most `lookback` bytes before the first hit, rounded down to a word, never before the line start
        size_t lo = hi > lookback ? (hi - lookback) & ~(size_t)3 : 0;
        t = lo;
        at_line_start = lo == 0;
        if (nl_in_chunk) {
            const uint32_t after = 32 - __clz(nl_in_chunk);   // offset just past the last newline before the hit
            t = o + after;
            at_line_start = true;
            line_bit = 1u << __popc(nl_in_chunk);
        } else {
            size_t p = o;   // 16-byte aligned; scan words [p-4, p) downwards for the last '\n' in [lo, o) (nothing to scan if lo >= o)
            while (p > lo) {
                uint32_t z = eq_mask4(*reinterpret_cast<const uint32_t*>(data + p - 4), 0x0a0a0a0au);
                if (p - 4 < lo) z &= ~((1u << (8 * (uint32_t)(lo - (p - 4)))) - 1u);
                if (z) {
                    t = (p - 4) + ((31 - __clz(z)) >> 3) + 1;
                    at_line_start = true;
                    break;
                }
                p -= 4;
            }
        }
    }
    for (int g = 0; g < db.ngroups; g++)
        if ((group_mask >> (g & 31)) & 1u) mask |= walk_local(db.groups[g], data, n, o, t, at_line_start, idle_from, line_bit);
    if (WITH_NFA && (group_mask & 0x80000000u)) {
        // lines that intersect the chunk: line 0 contains byte o, line j starts after the j-th newline of the chunk
        uint32_t nlm = newline_mask16(ld_chunk(data, o, n));
        size_t ls = line_start_of(data, o);
        for (uint32_t bit = 1u;; bit <<= 1) {
            bool nul = false;
            const size_t le = line_end_of(data, ls, n, &nul);
            if (!(mask & bit) && block_matches_nfa(db, data, ls, le)) mask |= bit;
            if (!nlm) break;
            ls = o + __ffs(nlm);
            nlm &= nlm - 1;
            if (ls >= o + 16 || ls >= n) break;   // that line starts outside the chunk
        }
    }
    marks[i] = mask;
    }
counted:
    if (survivors) {
        if (mask) atomicAdd(&tile_records[i / kEmitTile], (uint32_t)__popc(mask));
    } else {
        const uint32_t records = __reduce_add_sync(0xffffffffu, __popc(mask));
        if ((threadIdx.x & 31) == 0 && records) atomicAdd(&tile_records[i / kEmitTile], records);
    }
    }
}

// The same verification with the transition table in shared memory (single-group databases whose class-compressed table
// fits twice into one SM, GroupDev::ctab): [state][class] u16 plus the byte -> class map.  A step is one multiply-add and
// one shared load (the class lookups do not depend on the state and run ahead) instead of a dependent 2-byte gather
// from global memory through L1, which is what bounds k_verify_local.  Two blocks of 1,024 threads per SM: the same
// 64 warps as the global-table kernel, so the text loads (still global) are hidden as well as there.
constexpr int kVerifySmemThreads = 1024;
__global__ void __launch_bounds__(kVerifySmemThreads, 2) k_verify_smem(DbView db, const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ cand,
                                                                       const unsigned long long* meta_total, size_t cap, uint32_t lookback,
                                                                       uint32_t idle_span, uint32_t* __restrict__ marks,
                                                                       uint32_t* __restrict__ tile_records) {
    extern __shared__ __align__(16) uint32_t s_verify[];
    const GroupDev G = db.groups[0];
    // class map (256 bytes), table (rounded up to 16 bytes), depths of the states
    const uint32_t table_words = G.cdepth_off + (G.cstates + 15u) / 16u * 4u;
    {
        const uint32_t* src_cls = reinterpret_cast<const uint32_t*>(G.cmap);
        const uint32_t* src_tab = reinterpret_cast<const uint32_t*>(G.ctab);
        for (uint32_t k = threadIdx.x; k < 64u + table_words; k += blockDim.x) s_verify[k] = k < 64u ? src_cls[k] : src_tab[k - 64u];
        __syncthreads();
    }
    const SharedTable T{reinterpret_cast<const uint16_t*>(s_verify + 64), reinterpret_cast<const uint8_t*>(s_verify), G.crow / 2u,
                        reinterpret_cast<const uint8_t*>(s_verify + 64 + G.cdepth_off)};
    const GlobalText X{data};
    const uint32_t end = (uint32_t)n;
    size_t ncand = (size_t)(*meta_total >> 32);
    if (ncand > cap) ncand = cap;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; (i & ~(size_t)31) < ncand; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t mask = 0;
        if (i < ncand) {
            const uint32_t o = cand[i] * 16u;
            // start: at most `lookback` bytes before the chunk, rounded down to a word, never before the line start
            const uint32_t lo = o > lookback ? (o - lookback) & ~3u : 0u;
            uint32_t t = lo;
            bool at_line_start = lo == 0;
            for (uint32_t p = o; p > lo; p -= 4) {   // words [p-4, p) downwards: the last '\n' in [lo, o)
                const uint32_t z = eq_mask4(X.word(p - 4), 0x0a0a0a0au);   // lo is word-aligned: the word lies inside [lo, o)
                if (z) {
                    t = (p - 4) + ((31 - __clz(z)) >> 3) + 1;
                    at_line_start = true;
                    break;
                }
            }
            const uint32_t before = at_line_start ? 0u : data[t - 1];
            mask = walk_words(T, X, G, entry_state(G, at_line_start, before), end, o + 16u, t, o + idle_span, 1u);
            marks[i] = mask;
        }
        const uint32_t records = __reduce_add_sync(0xffffffffu, __popc(mask));
        if ((threadIdx.x & 31) == 0 && records) atomicAdd(&tile_records[i / kEmitTile], records);
    }
}

// Exclusive scan of the per-tile record counts (some thousand entries: one block, every thread takes a run of consecutive
// tiles so that one block-wide scan does it), in place; total -> *rec_total.
__global__ void __launch_bounds__(1024) k_tile_offsets(uint32_t* __restrict__ tile_records, const unsigned long long* meta_total, size_t cap,
                                                       unsigned long long* rec_total) {
    __shared__ unsigned long long s_warp[32], s_total;
    size_t ncand = (size_t)(*meta_total >> 32);
    if (ncand > cap) ncand = cap;
    const size_t ntiles = (ncand + kEmitTile - 1) / kEmitTile;
    const size_t per = (ntiles + blockDim.x - 1) / blockDim.x;
    const size_t lo = min(ntiles, (size_t)threadIdx.x * per), hi = min(ntiles, lo + per);
    unsigned long long sum = 0;
    for (size_t k = lo; k < hi; k++) sum += tile_records[k];
    unsigned long long run = block_exclusive_scan(sum, s_warp, &s_total);
    for (size_t k = lo; k < hi; k++) {
        const uint32_t v = tile_records[k];
        tile_records[k] = (uint32_t)run;
        run += v;
    }
    if (threadIdx.x == 0) *rec_total = s_total;
}

// Emit.  Candidates with marked lines are compacted per block (few candidates carry a match), then one thread per marked
// candidate computes line extents, line numbers and the exact re-check of lines with NULs.  The same line can be marked
// by several candidate chunks: every marking yields a record here, k_dedupe_records invalidates the repeats.
// Persistent blocks walk tiles of kEmitTile candidates.  The marked candidates of a tile go into a shared-memory queue
// together with their record offset (tile offset from k_tile_offsets + a block scan inside the tile); the block takes them
// out in FULL batches of one per thread and carries the remainder over to the next tile, so that the per-record work runs
// with every thread busy instead of a last, mostly empty round per tile.
constexpr uint32_t kEmitQueue = 1024;   // >= kEmitTile + kEmitThreads, power of two

// ------------------------------------------------------------------------------------------------------------
// Emit from the newline-chunk masks of k_stream (nlmask[block]: bit l set iff chunk l of the block holds a '\n').
// Line start, line end and line number of a record come from a few mask words and the two text chunks that hold the
// bounding newlines; the text of the line itself is read once, for the NUL test (hyperscanner.c:205-217 makes a line
// with NUL bytes a different scanned block, so such lines are re-checked exactly).  (Round 1 searched the text chunk by
// chunk for all of this, about 2,000 instructions per record: 211 -> 143 us per 2 GiB of the C2 workload.)
// ------------------------------------------------------------------------------------------------------------
// Index just past the last '\n' strictly before `pos` (the start of the line that contains byte pos), or 0.
__device__ uint32_t nlm_line_start(const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ nlmask, uint32_t pos) {
    const uint32_t c = pos >> 4;
    uint32_t b = c >> 5;
    uint32_t w = nlmask[b];
    if ((pos & 15u) && ((w >> (c & 31u)) & 1u)) {
        const uint32_t m = newline_mask16(ld_chunk(data, (size_t)c * 16, n)) & ((1u << (pos & 15u)) - 1u);
        if (m) return c * 16u + (32u - __clz(m));
    }
    w &= (1u << (c & 31u)) - 1u;   // chunks of this block below c
    while (true) {
        if (w) {
            const uint32_t cc = b * 32u + (31u - __clz(w));
            const uint32_t m = newline_mask16(ld_chunk(data, (size_t)cc * 16, n));
            return cc * 16u + (32u - __clz(m | 1u));
        }
        if (b == 0) return 0u;
        if (b >= 4) {   // four mask words per step (long lines: 2 KiB of text per step)
            const uint32_t w3 = nlmask[b - 1], w2 = nlmask[b - 2], w1 = nlmask[b - 3], w0 = nlmask[b - 4];
            if (w3) { b -= 1; w = w3; } else if (w2) { b -= 2; w = w2; } else if (w1) { b -= 3; w = w1; } else { b -= 4; w = w0; }
        } else {
            b--;
            w = nlmask[b];
        }
    }
}
// Index just past the first '\n' at or after `pos` (the end of the line that contains byte pos), or n.
__device__ uint32_t nlm_line_end(const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ nlmask, uint32_t nblk, uint32_t pos) {
    const uint32_t c = pos >> 4;
    uint32_t b = c >> 5;
    uint32_t w = nlmask[b];
    if ((w >> (c & 31u)) & 1u) {
        const uint32_t m = newline_mask16(ld_chunk(data, (size_t)c * 16, n)) & ~((1u << (pos & 15u)) - 1u);
        if (m) return c * 16u + __ffs(m);
    }
    w &= ~((2u << (c & 31u)) - 1u);   // chunks of this block above c (c == 31: 2u << 31 == 0, the mask clears everything)
    while (true) {
        if (w) {
            const uint32_t cc = b * 32u + (__ffs(w) - 1u);
            const uint32_t m = newline_mask16(ld_chunk(data, (size_t)cc * 16, n));
            return m ? cc * 16u + __ffs(m) : (uint32_t)n;
        }
        if (b + 4 < nblk) {
            const uint32_t w0 = nlmask[b + 1], w1 = nlmask[b + 2], w2 = nlmask[b + 3], w3 = nlmask[b + 4];
            if (w0) { b += 1; w = w0; } else if (w1) { b += 2; w = w1; } else if (w2) { b += 3; w = w2; } else { b += 4; w = w3; }
        } else {
            b++;
            if (b >= nblk) return (uint32_t)n;
            w = nlmask[b];
        }
    }
}
// Number of '\n' in [0, st), for st == 0 or st just past a newline.
__device__ uint32_t nlm_line_number(const uint8_t* __restrict__ data, const unsigned long long* __restrict__ meta,
                                    const unsigned long long* __restrict__ prefix, const uint32_t* __restrict__ nlmask, uint32_t st) {
    if (st == 0) return 0u;
    const uint32_t cq = (st - 1u) >> 4, bq = cq >> 5;
    const uint32_t base = newlines_before_block(prefix, meta, bq);
    const uint32_t w = nlmask[bq];
    // every newline chunk of the block holds exactly one newline (lines of 16 bytes and more): chunks below + the one at st - 1
    if ((uint32_t)(meta[bq] >> 32) == (uint32_t)__popc(w)) return base + __popc(w & ((1u << (cq & 31u)) - 1u)) + 1u;
    return base + count_newlines(data, (size_t)bq << 9, st);
}
// NUL bytes in [from, to)?  Per-thread loop over at most `bound` bytes; returns false and sets *resume (16-byte aligned,
// no NUL in [from, *resume)) when the range is longer.
__device__ bool nul_scan_bounded(const uint8_t* __restrict__ data, size_t n, uint32_t from, uint32_t to, uint32_t bound, bool* has_nul, uint32_t* resume) {
    uint32_t base = from & ~15u;
    bool nul = false;
    const uint32_t stop = from + bound < to ? ((from + bound) & ~15u) : to;
    while (base < stop && !nul) {
        // up to four chunks per step, all loads issued before the first test
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = base + 16u * k < stop ? ld_chunk(data, (size_t)base + 16u * k, n) : make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t cb = base + 16u * k;
            if (cb < stop && (haszero4(v[k].x) | haszero4(v[k].y) | haszero4(v[k].z) | haszero4(v[k].w))) {
                uint32_t zm = byte_mask16(v[k], 0u);
                if (cb < from) zm &= ~((1u << (from - cb)) - 1u);
                if (cb + 16u > to) zm &= (1u << (to - cb)) - 1u;
                nul |= zm != 0u;
            }
        }
        base += 64u;
    }
    *has_nul = nul;
    if (nul || stop >= to) return true;
    *resume = stop;
    return false;
}
// Whole warp: NUL bytes in [from, to)?  from is 16-byte aligned.  2 KiB per step (four loads per lane in flight: the
// lines are read from DRAM, so the steps of a 16 KiB line cost a round trip each).
__device__ bool warp_nul_scan(const uint8_t* __restrict__ data, size_t n, uint32_t from, uint32_t to) {
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t pos = from; pos < to; pos += 2048u) {
        uint4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t cb = pos + 512u * j + 16u * lane;
            v[j] = cb < to ? ld_chunk(data, cb, n) : make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
        }
        bool nul = false;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t cb = pos + 512u * j + 16u * lane;
            if (cb < to) {
                uint32_t zm = byte_mask16(v[j], 0u);
                if (cb + 16u > to) zm &= (1u << (to - cb)) - 1u;
                nul |= zm != 0u;
            }
        }
        if (__any_sync(0xffffffffu, nul)) return true;
    }
    return false;
}

// Count-only identity of a line that is cheaper than its start: the chunk c that holds the newline in front of the line and
// the rank r of that newline among the newlines of c counted from the last one (r = 0: the last), as c * 16 + 15 - r;
// kNoNewlineKey for the first line of the segment.  Two records of one line get the same key, records of different lines
// different keys, and the key of the line that contains an aligned chunk start o comes from nlmask words alone.
constexpr uint32_t kNoNewlineKey = 0xfffffffeu;   // (chunk * 16 + 15 stays below it: segments are < 4 GiB - 1 KiB)
__device__ uint32_t nlm_line_key(const uint32_t* __restrict__ nlmask, uint32_t o) {
    const uint32_t c = o >> 4;
    uint32_t b = c >> 5;
    uint32_t w = nlmask[b] & ((1u << (c & 31u)) - 1u);   // chunks of this block below c
    while (true) {
        if (w) return (b * 32u + (31u - __clz(w))) * 16u + 15u;
        if (b == 0) return kNoNewlineKey;
        if (b >= 4) {   // four mask words per step, as nlm_line_start
            const uint32_t w3 = nlmask[b - 1], w2 = nlmask[b - 2], w1 = nlmask[b - 3], w0 = nlmask[b - 4];
            if (w3) { b -= 1; w = w3; } else if (w2) { b -= 2; w = w2; } else if (w1) { b -= 3; w = w1; } else { b -= 4; w = w0; }
        } else {
            b--;
            w = nlmask[b];
        }
    }
}

constexpr uint32_t kNulBound = 512;
// Records of one marked candidate chunk per lane; whole warps call it (`live`: this lane has a candidate).
// `nul_free` (count-only scans): k_stream found no NUL byte in the segment, so no line needs the NUL scan and the exact re-check.
// COUNT_ONLY: instead of a LineRec, one 32-bit key per record goes to keys[at] (kInvalidLen: failed NUL re-check), from
// which k_count_keys counts the distinct valid lines; no line numbers.  In a NUL-free segment the key is nlm_line_key
// (no line extents at all), else the line start (the extents are needed for the re-check anyway).
template <bool WITH_NFA, bool COUNT_ONLY, bool LITERAL>
__device__ uint32_t emit_lane_nlm(const DbView& db, const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ cand,
                                  const uint32_t* __restrict__ marks, const unsigned long long* __restrict__ meta,
                                  const unsigned long long* __restrict__ prefix, const uint32_t* __restrict__ nlmask, uint32_t nblk, bool live, size_t i,
                                  size_t at, LineRec* __restrict__ recs, uint32_t* __restrict__ keys, size_t rec_cap, bool nul_free, Totals* totals,
                                  const LiteralView& lits) {
    const uint32_t lane = threadIdx.x & 31;
    uint32_t valid = 0;
    uint32_t mask = live ? marks[i] : 0u;
    const uint32_t o = live ? cand[i] * 16u : 0u;
    uint32_t nlm = 0;
    if (live && ((nlmask[o >> 9] >> ((o >> 4) & 31u)) & 1u)) nlm = newline_mask16(ld_chunk(data, o, n));
    uint32_t st = 0;
    bool first = true;   // still on line 0 of the chunk (the line that contains byte o)
    if (COUNT_ONLY && nul_free) {
        // key of line j > 0 of the chunk: c * 16 + 15 - (newlines of the chunk behind the one in front of the line)
        const uint32_t key_base = (o >> 4) * 16u + 15u;
        while (mask != 0) {
            while (!(mask & 1u)) {   // lines of the chunk that are not marked
                if (!nlm) { mask = 0; break; }
                nlm &= nlm - 1;
                first = false;
                mask >>= 1;
            }
            if (mask == 0) break;
            const uint32_t key = first ? nlm_line_key(nlmask, o) : key_base - __popc(nlm);
            valid++;
            if (at < rec_cap) keys[at] = key;
            else atomicOr(&totals->flags, 4u);
            at++;
            if (!nlm) mask = 0;
            else {
                nlm &= nlm - 1;
                first = false;
                mask >>= 1;
            }
        }
        return valid;
    }
    while (__any_sync(0xffffffffu, mask != 0)) {
        while (mask != 0 && !(mask & 1u)) {   // lines of the chunk that are not marked
            if (!nlm) { mask = 0; break; }
            st = o + __ffs(nlm);
            nlm &= nlm - 1;
            first = false;
            mask >>= 1;
        }
        const bool work = mask != 0;
        uint32_t en = 0, resume = 0;
        bool has_nul = false, settled = true, ok = true;
        if (work) {
            if (first) st = nlm_line_start(data, n, nlmask, o);
            en = nlm ? o + __ffs(nlm) : nlm_line_end(data, n, nlmask, nblk, o + 16u < (uint32_t)n ? o + 16u : (uint32_t)n - 1u);
            // (nlm == 0 here means: no newline at or after st inside the chunk, so the line ends beyond it; if the chunk is
            //  the last one, the search starts at the last byte and returns n)
            if (!nul_free) settled = nul_scan_bounded(data, n, st, en, kNulBound, &has_nul, &resume);
        }
        for (uint32_t pend = __ballot_sync(0xffffffffu, work && !settled); pend; pend &= pend - 1) {
            const int src = __ffs(pend) - 1;
            const bool more = warp_nul_scan(data, n, __shfl_sync(0xffffffffu, resume, src), __shfl_sync(0xffffffffu, en, src));
            if ((int)lane == src) has_nul = more;
        }
        if (work) {
            if (ok && has_nul)
                ok = LITERAL ? block_matches_literal(lits, data, st, en) : block_matches<false>(db, data, st, en) || (WITH_NFA && block_matches_nfa(db, data, st, en));
            valid += ok ? 1u : 0u;
            if (COUNT_ONLY) {
                if (at < rec_cap) keys[at] = ok ? st : kInvalidLen;
                else atomicOr(&totals->flags, 4u);
            } else {
                const uint32_t line_no = nlm_line_number(data, meta, prefix, nlmask, st);
                if (at < rec_cap) recs[at] = LineRec{line_no, st, ok ? ((en - st) | (has_nul ? kHasNulBit : 0u)) : kInvalidLen};
                else atomicOr(&totals->flags, 4u);
            }
            at++;
            if (!nlm) mask = 0;
            else {
                st = o + __ffs(nlm);
                nlm &= nlm - 1;
                first = false;
                mask >>= 1;
            }
        }
    }
    return valid;
}

// COUNT_ONLY (the caller wants no records: grep -c, count-only scans): keys for k_count_keys instead of records (see
// emit_lane_nlm); `recs` is unused and `rec_cap` is the capacity of `keys`.
// LITERAL: a fixed-string set (k_literal.cuh): lines with NUL bytes are re-checked against `lits`, which only it reads.
template <bool WITH_NFA, bool COUNT_ONLY, bool LITERAL = false>   // WITH_NFA: the database holds NFA-fallback patterns: lines with NUL bytes are re-checked with them too (1 KiB of local memory)
__global__ void __launch_bounds__(kEmitThreads, 6) k_emit_nlm(DbView db, const uint8_t* __restrict__ data, size_t n, const uint32_t* __restrict__ cand,
                                                           const uint32_t* __restrict__ marks, const uint32_t* __restrict__ tile_offsets,
                                                           const unsigned long long* __restrict__ meta, const unsigned long long* __restrict__ prefix,
                                                           const uint32_t* __restrict__ nlmask, const unsigned long long* meta_total, size_t cap,
                                                           LineRec* __restrict__ recs, uint32_t* __restrict__ keys, size_t rec_cap, Totals* totals,
                                                           LiteralView lits = {}) {
    __shared__ uint32_t q_cand[kEmitQueue], q_at[kEmitQueue];
    __shared__ unsigned long long s_warp[kEmitThreads / 32], s_total;
    const uint32_t nblk = (uint32_t)((n + 511) >> 9);
    const bool nul_free = COUNT_ONLY && !(totals->flags & kSegmentNulFlag);   // (k_stream tests for NUL bytes in count-only scans only)
    uint32_t valid = 0;
    uint32_t head = 0, queued = 0;   // the same in every thread of the block
    size_t ncand = (size_t)(*meta_total >> 32);
    if (ncand > cap) ncand = cap;
    constexpr int kPer = kEmitTile / kEmitThreads;
    const size_t ntiles = (ncand + kEmitTile - 1) / kEmitTile;
    for (size_t block_base = (size_t)blockIdx.x * kEmitTile; block_base < ncand; block_base += (size_t)gridDim.x * kEmitTile) {
        {
            // a tile without any record (sparse matches among many candidates): nothing to queue, not even its marks are read
            const size_t tile = block_base / kEmitTile;
            const uint32_t next = tile + 1 < ntiles ? tile_offsets[tile + 1] : (uint32_t)totals->rec_total;
            if (next == tile_offsets[tile]) continue;
        }
        uint32_t mk[kPer];
        uint32_t records = 0, marked = 0;
#pragma unroll
        for (int j = 0; j < kPer; j++) {
            const size_t i = block_base + (size_t)threadIdx.x * kPer + j;
            mk[j] = i < ncand ? marks[i] : 0u;
            records += __popc(mk[j]);
            marked += mk[j] != 0u;
        }
        const unsigned long long before = block_exclusive_scan(((unsigned long long)marked << 32) | records, s_warp, &s_total);
        uint32_t slot = head + queued + (uint32_t)(before >> 32);
        uint32_t at = tile_offsets[block_base / kEmitTile] + (uint32_t)before;
#pragma unroll
        for (int j = 0; j < kPer; j++) {
            if (mk[j]) {
                q_cand[slot & (kEmitQueue - 1)] = (uint32_t)(block_base + (size_t)threadIdx.x * kPer + j);
                q_at[slot & (kEmitQueue - 1)] = at;
                slot++;
                at += __popc(mk[j]);
            }
        }
        queued += (uint32_t)(s_total >> 32);
        __syncthreads();
        while (queued >= (uint32_t)kEmitThreads) {
            const uint32_t k = (head + threadIdx.x) & (kEmitQueue - 1);
            valid += emit_lane_nlm<WITH_NFA, COUNT_ONLY, LITERAL>(db, data, n, cand, marks, meta, prefix, nlmask, nblk, true, q_cand[k], q_at[k], recs, keys,
                                                                  rec_cap, nul_free, totals, lits);
            head += kEmitThreads;
            queued -= kEmitThreads;
        }
        __syncthreads();
    }
    if (queued) {
        // the remainder is dealt out across the warps (entry j -> lane j / 8 of warp j % 8), not to the first warps only: the
        // long-line searches of one warp run one after the other
        constexpr uint32_t kWarps = kEmitThreads / 32;
        const uint32_t j = (threadIdx.x >> 5) + kWarps * (threadIdx.x & 31);
        const uint32_t k = (head + j) & (kEmitQueue - 1);
        const bool live = j < queued;
        valid += emit_lane_nlm<WITH_NFA, COUNT_ONLY, LITERAL>(db, data, n, cand, marks, meta, prefix, nlmask, nblk, live, live ? q_cand[k] : 0,
                                                              live ? q_at[k] : 0, recs, keys, rec_cap, nul_free, totals, lits);
    }
    (void)valid;   // the unique valid records are counted by k_dedupe_records / k_count_keys
}

// The same line can be marked by several candidate chunks that intersect it.  Their records are ADJACENT in the record
// array (records follow candidate order, and every candidate between two chunks of one line lies on that line too), so a
// repeat is a record with the start offset of its predecessor: it is marked kInvalidLen here (the host skips those), and
// the valid records - what a count-only caller needs - are counted.  (Round 1 looked back over the earlier candidates of
// the line inside the emit kernel: with a fifth of all chunks being candidates and 8 KiB lines that was a walk over
// ~100 candidates per record.)
__global__ void __launch_bounds__(256) k_dedupe_records(LineRec* __restrict__ recs, size_t rec_cap, Totals* totals) {
    size_t nrec = (size_t)totals->rec_total;
    if (nrec > rec_cap) nrec = rec_cap;
    uint32_t valid = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nrec; i += (size_t)gridDim.x * blockDim.x) {
        if (i > 0 && recs[i].start == recs[i - 1].start) recs[i].len = kInvalidLen;
        else if (recs[i].len != kInvalidLen) valid++;
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0 && valid) atomicAdd(&totals->aux_total, (unsigned long long)valid);
}

// Count-only counterpart of k_dedupe_records over the keys of k_emit_nlm<*, true>: the valid keys that differ from their
// predecessor (the records of one line are adjacent, see above) are the distinct matched lines -> aux_total.
__global__ void __launch_bounds__(256) k_count_keys(const uint32_t* __restrict__ keys, size_t cap, Totals* totals) {
    size_t nkeys = (size_t)totals->rec_total;
    if (nkeys > cap) nkeys = cap;
    uint32_t valid = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nkeys; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t key = keys[i];
        if (key != kInvalidLen && (i == 0 || key != keys[i - 1])) valid++;
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0 && valid) atomicAdd(&totals->aux_total, (unsigned long long)valid);
}

// Device-resident inputs: the end of segment j is the byte after a '\n' before boundary (j+1)*chunk, chosen so that the
// NEXT segment starts 16-byte aligned (the kernels use 16-byte loads): one line end in 16 qualifies on average.
// One thread per boundary scans backwards (gives up after `window` bytes -> 0 = not found).
__global__ void k_find_cuts(const uint8_t* __restrict__ data, size_t size, size_t chunk, size_t window, size_t ncuts, unsigned long long* __restrict__ cuts) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ncuts) return;
    size_t b = (j + 1) * chunk;
    if (b >= size) { cuts[j] = size; return; }
    size_t lo = b > window ? b - window : 0;
    unsigned long long found = 0;
    for (size_t p = b; p > lo; p--) {
        if ((p & 15) == 0 && data[p - 1] == '\n') { found = p; break; }
    }
    cuts[j] = found;
}

}  // namespace gpugrep
