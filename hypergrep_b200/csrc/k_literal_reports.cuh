// Report stage of fixed-string scans (gpugrep_literal_report_scan_*): every (literal, end) in the lines that the
// selection (k_verify_literals on the fast path, k_match_pl_literals on the general path) picked.  Part of the CUDA engine
// (engine.cu includes these files in this order; they form one translation unit).
//
// Search rule (database.hpp LiteralReports): at a text position, let x be the greatest node of the position's two-byte
// bucket that is not above the text, and k the length of the common prefix of x and the text.  A node m that matches there
// satisfies m <= x <= text, so m is a prefix of x: the matches are x's parent chain from the first node of length <= k on.
// One binary search per position and class, then a walk that reports every node it visits after the cut.
//
// One warp per selected line, its positions spread over the lanes, so that a long pseudo-line (up to buffer_size bytes)
// is not left to one thread.  Run twice like k_match_pl_events: a count pass (events per record), a scan of the counts,
// and a write pass that stores each record's events at its offset.
#pragma once

namespace gpugrep {

struct LiteralReportView {
    LiteralView lits;                     // nodes: bytes / off / len / order / bucket as LiteralSet; `one` unused
    const uint32_t* __restrict__ parent;  // per node: longest proper prefix node of its class, or kNoLiteral
    const uint32_t* __restrict__ one;     // [class * 256 + b]: node of the one-byte literal b, or kNoLiteral
};

// Length of the common prefix of node `id` (class `cls`) and the text at x (the text ends at lim).
__device__ __forceinline__ uint32_t lit_common_prefix(const LiteralView& L, uint32_t id, uint32_t cls, const uint8_t* __restrict__ data,
                                                      size_t x, size_t lim) {
    const uint8_t* __restrict__ p = L.bytes + L.off[id];
    const uint32_t len = L.len[id];
    uint32_t k = 0;
    while (k < len && x + k < lim && lit_norm(data[x + k], cls) == p[k]) k++;
    return k;
}

// Every node that starts at x (x < lim): emit(node, x + length of the node).  Returns the number of nodes.
template <class Emit>
__device__ __forceinline__ uint32_t lit_reports_at(const LiteralReportView& R, const uint8_t* __restrict__ data, size_t x, size_t lim, Emit emit) {
    const LiteralView& L = R.lits;
    uint32_t found = 0;
    const uint32_t b0 = data[x], b1 = x + 1 < lim ? data[x + 1] : 0u;
    for (uint32_t cls = 0; cls < 2; cls++) {
        if (!((L.classes >> cls) & 1u)) continue;
        const uint32_t n0 = lit_norm(b0, cls);
        uint32_t node = kNoLiteral, k = 1;
        if (x + 1 < lim) {
            const uint32_t key = cls * 65537u + (n0 << 8 | lit_norm(b1, cls));
            const uint32_t first = L.bucket[key];
            uint32_t lo = first, hi = L.bucket[key + 1];
            while (lo < hi) {   // first node above the text
                const uint32_t mid = (lo + hi) >> 1;
                if (lit_compare(L, L.order[mid], cls, data, x, lim) <= 0) lo = mid + 1;
                else hi = mid;
            }
            if (lo > first) {
                node = L.order[lo - 1];
                k = lit_common_prefix(L, node, cls, data, x, lim);
            }
        }
        if (node == kNoLiteral) node = R.one[cls * 256 + n0];   // no node of >= 2 bytes below the text: the one-byte node, if any
        for (; node != kNoLiteral; node = R.parent[node]) {
            const uint32_t len = L.len[node];
            if (len > k) continue;
            emit(node, x + len);
            found++;
        }
    }
    return found;
}

// Whole warp: the scanned block [a, e) of the pseudo-line [st, lim): leading NULs skipped, cut at the next NUL.
__device__ __forceinline__ void warp_scanned_block(const uint8_t* __restrict__ data, size_t st, size_t lim, size_t& a, size_t& e) {
    const uint32_t lane = threadIdx.x & 31u;
    a = st;
    for (;; a += 32) {
        const uint32_t nonzero = __ballot_sync(0xffffffffu, a + lane < lim && data[a + lane] != 0);
        if (nonzero) { a += __ffs(nonzero) - 1; break; }
        if (a + 32 >= lim) { a = lim; break; }
    }
    e = a;
    for (; e < lim; e += 32) {
        const uint32_t nul = __ballot_sync(0xffffffffu, e + lane < lim && data[e + lane] == 0);
        if (nul) { e += __ffs(nul) - 1; break; }
    }
    if (e > lim) e = lim;
}

// Count pass (out == nullptr): counts[r] = events of record r.  Write pass: the events of record r at out + off[r].
// Records marked kLineInvalid (fast-path repeats, failed NUL re-checks) have none.
__global__ void __launch_bounds__(128) k_literal_reports(LiteralReportView R, const uint8_t* __restrict__ data, const LineRec* __restrict__ recs,
                                                         size_t nrec, uint32_t* __restrict__ counts, const unsigned long long* __restrict__ off,
                                                         EventRec* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nrec; r += warps) {
        const LineRec rec = recs[r];
        if (rec.len == kLineInvalid || (out && counts[r] == 0)) {
            if (!out && lane == 0) counts[r] = 0;
            continue;
        }
        const size_t st = rec.start, lim = st + (rec.len & kLineLenMask);
        // the scanned block [a, e) (a literal holds no NUL: none spans the cut)
        size_t a, e;
        warp_scanned_block(data, st, lim, a, e);
        uint32_t total = 0;   // events of the lanes' earlier rounds (write pass: events already written)
        EventRec* dst = out ? out + off[r] : nullptr;
        const uint32_t line_len = rec.len & kLineLenMask;
        for (size_t base = a; base < e; base += 32) {
            const size_t x = base + lane;
            uint32_t c = 0;
            if (x < e) c = lit_reports_at(R, data, x, e, [](uint32_t, size_t) {});
            if (out) {
                uint32_t incl = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= (uint32_t)d) incl += t;
                }
                uint32_t at = total + incl - c;
                if (c) lit_reports_at(R, data, x, e, [&](uint32_t node, size_t end) {
                    dst[at++] = EventRec{rec.line, rec.start, line_len, (uint32_t)(end - a), node};
                });
                total += __shfl_sync(0xffffffffu, incl, 31);
            } else {
                total += __reduce_add_sync(0xffffffffu, c);
            }
        }
        if (!out && lane == 0) counts[r] = total;
    }
}

}  // namespace gpugrep
