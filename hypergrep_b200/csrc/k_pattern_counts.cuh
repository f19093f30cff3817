// Per-pattern line counts (gpugrep_pattern_counts_*): how many lines each pattern reports in.  Part of the CUDA engine
// (engine.cu includes these files in this order; they form one translation unit).
//
// Every route ends in events that are grouped by line in line order: k_line_events (regex sets, fast path: the lines the
// selection picked), k_match_pl_events (regex sets, general path: every pseudo-line) and k_literal_reports (fixed
// strings).  A line's events are [off[r], off[r] + counts[r]) of the count pass and its scan.  k_count_patterns expands
// each event's report to its ids (ReportIdView) and adds 1 per distinct (line, id) into one unsigned long long per id;
// only that array goes to the host.
//  - a warp per line, the distinct ids of the line in a shared-memory hash set of kCountSlots slots.  Nothing is added
//    while the line is being read: a line with more than kCountCap distinct ids leaves the set unused and is passed on
//    whole, so no line is ever counted twice or in part.  Repeats of an id (10^5 events of one pattern) cost one probe each.
//  - k_count_patterns_big: a block per line that overflowed, with a bitmap of every id in global memory (one per block,
//    zero before and after each line); the first thread that sets a bit counts it.  Exact for any fan-out.
#pragma once

namespace gpugrep {

// ids[begin[r] .. begin[r + 1]): the ids of flat report r (EventRec::report: an accept set of a DFA group, an NFA-fallback
// pattern, or a node of a fixed-string report table)
struct ReportIdView {
    const uint32_t* __restrict__ begin;
    const uint32_t* __restrict__ ids;
};

constexpr uint32_t kCountSlots = 2048, kCountCap = 1024, kCountEmpty = 0xffffffffu;
constexpr int kCountWarps = 4;   // warps per block of k_count_patterns (128 threads, 32 KiB of hash sets)

// Regex sets, fast path: the events of the first `nrec` records (the selected lines; kLineInvalid ones have none) under the
// attribution database, one thread per record.  Count pass (out == nullptr): counts[r]; write pass: the events at off[r].
// block_events cuts the scanned block at its NULs itself, so a kHasNulBit line needs nothing more than its length.
__global__ void __launch_bounds__(128) k_line_events(DbView db, const uint8_t* __restrict__ data, const LineRec* __restrict__ recs, size_t nrec,
                                                     uint32_t* __restrict__ counts, const unsigned long long* __restrict__ off, EventRec* __restrict__ out) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrec) return;
    const LineRec rec = recs[r];
    if (rec.len == kLineInvalid) {
        if (!out) counts[r] = 0;
        return;
    }
    const uint32_t len = rec.len & kLineLenMask;
    if (out) {
        if (counts[r]) block_events(db, data, rec.start, (size_t)rec.start + len, rec.line, rec.start, len, out + off[r]);
    } else {
        counts[r] = block_events(db, data, rec.start, (size_t)rec.start + len, rec.line, rec.start, len, nullptr);
    }
}

// meta[0]: lines with at least one event; meta[1]: lines passed on to k_count_patterns_big, whose numbers go to `big`.
__global__ void __launch_bounds__(128) k_count_patterns(ReportIdView R, const EventRec* __restrict__ ev, const uint32_t* __restrict__ counts,
                                                        const unsigned long long* __restrict__ off, size_t nrec, unsigned long long* __restrict__ pcounts,
                                                        unsigned long long* __restrict__ meta, uint32_t* __restrict__ big) {
    __shared__ uint32_t table[kCountWarps][kCountSlots];
    __shared__ uint32_t fill[kCountWarps];
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    uint32_t* t = table[w];
    volatile uint32_t* vfill = &fill[w];
    const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nrec; r += warps) {
        const uint32_t n = counts[r];
        if (n == 0) continue;
        for (uint32_t k = lane; k < kCountSlots; k += 32) t[k] = kCountEmpty;
        if (lane == 0) *vfill = 0;
        __syncwarp();
        const size_t b = (size_t)off[r];
        bool over = false;
        for (uint32_t base = 0; base < n; base += 32) {
            if (base + lane < n && !over) {
                const uint32_t rep = ev[b + base + lane].report;
                for (uint32_t k = R.begin[rep], e = R.begin[rep + 1]; k < e; k++) {
                    if (*vfill > kCountCap) { over = true; break; }
                    const uint32_t id = R.ids[k];
                    uint32_t h = (id * 2654435761u) >> 21;   // kCountSlots = 2^11
                    while (true) {
                        const uint32_t old = atomicCAS(&t[h], kCountEmpty, id);
                        if (old == kCountEmpty) { atomicAdd(&fill[w], 1u); break; }
                        if (old == id) break;
                        h = (h + 1) & (kCountSlots - 1);
                    }
                }
            }
            if (__any_sync(0xffffffffu, over)) { over = true; break; }
        }
        __syncwarp();
        if (over) {
            if (lane == 0) big[atomicAdd(&meta[1], 1ull)] = (uint32_t)r;
        } else {
            for (uint32_t k = lane; k < kCountSlots; k += 32)
                if (t[k] != kCountEmpty) atomicAdd(&pcounts[t[k]], 1ull);
        }
        if (lane == 0) atomicAdd(&meta[0], 1ull);
        __syncwarp();
    }
}

// The lines k_count_patterns passed on, a block each; `bitmaps`: one zeroed bitmap of `words` words per block.
__global__ void __launch_bounds__(256) k_count_patterns_big(ReportIdView R, const EventRec* __restrict__ ev, const uint32_t* __restrict__ counts,
                                                            const unsigned long long* __restrict__ off, const unsigned long long* __restrict__ meta,
                                                            const uint32_t* __restrict__ big, unsigned long long* __restrict__ pcounts,
                                                            uint32_t* __restrict__ bitmaps, size_t words) {
    uint32_t* bm = bitmaps + (size_t)blockIdx.x * words;
    const size_t nbig = (size_t)meta[1];
    for (size_t i = blockIdx.x; i < nbig; i += gridDim.x) {
        const uint32_t r = big[i];
        const size_t b = (size_t)off[r], n = counts[r];
        for (size_t j = threadIdx.x; j < n; j += blockDim.x) {
            const uint32_t rep = ev[b + j].report;
            for (uint32_t k = R.begin[rep], e = R.begin[rep + 1]; k < e; k++) {
                const uint32_t id = R.ids[k], bit = 1u << (id & 31u);
                if (!(atomicOr(&bm[id >> 5], bit) & bit)) atomicAdd(&pcounts[id], 1ull);
            }
        }
        __syncthreads();
        for (size_t j = threadIdx.x; j < n; j += blockDim.x) {
            const uint32_t rep = ev[b + j].report;
            for (uint32_t k = R.begin[rep], e = R.begin[rep + 1]; k < e; k++) bm[R.ids[k] >> 5] = 0;
        }
        __syncthreads();
    }
}

}  // namespace gpugrep
