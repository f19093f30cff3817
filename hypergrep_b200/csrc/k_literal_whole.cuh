// Whole-word and whole-line fixed strings (gpugrep_literal_whole_scan_*, grep -F -w / -F -x).  Part of the CUDA engine
// (engine.cu includes these files in this order; they form one translation unit).
//
// An occurrence of a literal as a word, or a line that is a literal, is always a plain occurrence, so the lines that the
// fixed-string selection picks (k_verify_literals / k_match_pl_literals) are a superset of the answer.  The prefix-free
// selection set cannot decide which of them stay (`foo` hides `foobar`), the report table can: lit_reports_at lists every
// literal that starts at a position, with its end.
//  - word (kWholeWord): some occurrence [s, end) has no word byte at s - 1 (or s is the block start) and none at end (or
//    end is the block end).  Word bytes are [0-9A-Za-z_]; the test reads the raw bytes, CASELESS or not.  The lanes of a
//    warp take 32 positions per round, positions behind a word byte are not looked up, and the first passing occurrence
//    ends the line.
//  - line (kWholeLine): the block without its final '\n' is a literal: one lookup at the block start, for a node that ends
//    there.  A literal holding a '\n' never matches.
//  - fast path: k_literal_whole_filter runs after k_emit_nlm<*, LITERAL> and before k_dedupe_records, one warp per record,
//    and turns the records of failing lines into kInvalidLen.  Repeats of a line (the records of several candidate chunks
//    that intersect it, adjacent in the array) are skipped: k_dedupe_records invalidates them by their start, whatever
//    the first record of the line became.  So the valid count, inversion, context lines and delivery stay as they are.
//  - general path: k_match_pl_literal_whole takes the place of k_match_pl_literals (the per-pseudo-line flag, with invert).
// (__launch_bounds__(128, 8): with (128) alone ptxas holds these kernels to 40 registers and spills; 8 blocks allow 64)
#pragma once

namespace gpugrep {

constexpr unsigned kWholeWord = 1, kWholeLine = 2;

__device__ __forceinline__ bool lit_word_byte(uint32_t b) { return b - '0' < 10u || (b | 0x20u) - 'a' < 26u || b == '_'; }

// Whole warp: does the scanned block [a, e) pass `whole`?  The same answer in every lane.
__device__ __forceinline__ bool warp_block_whole(const LiteralReportView& R, const uint8_t* __restrict__ data, size_t a, size_t e, unsigned whole) {
    const uint32_t lane = threadIdx.x & 31u;
    if (whole == kWholeLine) {
        const size_t end = e > a && data[e - 1] == '\n' ? e - 1 : e;
        bool ok = false;
        if (lane == 0 && end > a) lit_reports_at(R, data, a, end, [&](uint32_t, size_t at) { ok |= at == end; });
        return __shfl_sync(0xffffffffu, ok, 0);
    }
    for (size_t base = a; base < e; base += 32) {
        const size_t x = base + lane;
        bool ok = false;
        if (x < e && (x == a || !lit_word_byte(data[x - 1])))
            lit_reports_at(R, data, x, e, [&](uint32_t, size_t at) { ok |= at == e || !lit_word_byte(data[at]); });
        if (__any_sync(0xffffffffu, ok)) return true;
    }
    return false;
}

// Fast path: the first min(rec_total, rec_cap) records of k_emit_nlm, a warp per record.  Only fast-path records of lines
// with NUL bytes (kHasNulBit) need the scanned block cut out of the line.
__global__ void __launch_bounds__(128, 8) k_literal_whole_filter(LiteralReportView R, const uint8_t* __restrict__ data, LineRec* __restrict__ recs,
                                                              size_t rec_cap, const Totals* totals, unsigned whole) {
    const uint32_t lane = threadIdx.x & 31u;
    size_t nrec = (size_t)totals->rec_total;
    if (nrec > rec_cap) nrec = rec_cap;
    const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nrec; r += warps) {
        const LineRec rec = recs[r];
        if (rec.len == kInvalidLen || (r > 0 && recs[r - 1].start == rec.start)) continue;
        const size_t st = rec.start, lim = st + (rec.len & kLineLenMask);
        size_t a = st, e = lim;
        if (rec.len & kHasNulBit) warp_scanned_block(data, st, lim, a, e);
        if (!warp_block_whole(R, data, a, e, whole) && lane == 0) recs[r].len = kInvalidLen;
    }
}

// General path: flags[i] = (pseudo-line i passes `whole`) != invert, a warp per pseudo-line.
__global__ void __launch_bounds__(128, 8) k_match_pl_literal_whole(LiteralReportView R, const uint8_t* __restrict__ data, const uint32_t* __restrict__ pl_start,
                                                                const uint32_t* __restrict__ pl_len, size_t npl, uint8_t* __restrict__ flags, bool invert,
                                                                unsigned whole) {
    const uint32_t lane = threadIdx.x & 31u;
    const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < npl; i += warps) {
        const size_t st = pl_start[i];
        size_t a, e;
        warp_scanned_block(data, st, st + pl_len[i], a, e);
        const bool hit = warp_block_whole(R, data, a, e, whole);
        if (lane == 0) flags[i] = hit != invert ? 1 : 0;
    }
}

}  // namespace gpugrep
