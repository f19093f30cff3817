// Span stage (grep -o, gpugrep_match_spans): the leftmost-first match spans of one pattern in every pseudo-line, from the
// pike_vm.hpp simulation, one thread per pseudo-line.  Run twice like k_match_pl_events: a count pass (spans per line, 1 for
// a line over its step budget), a scan of the counts, and a write pass that stores each line's spans at its offset.
#pragma once
#include "pike_vm.hpp"

namespace gpugrep {

// The program and its byte sets are copied to shared memory (dynamic: ninst + 8 * nsets words).
__global__ void __launch_bounds__(128) k_spans(const uint32_t* __restrict__ prog, int ninst, int nsets, int start_pc,
                                               const uint8_t* __restrict__ data, const uint32_t* __restrict__ pl_start,
                                               const uint32_t* __restrict__ pl_len, size_t npl, uint32_t* __restrict__ counts,
                                               const unsigned long long* __restrict__ off, SpanRec* __restrict__ out) {
    extern __shared__ uint32_t s_prog[];
    const int words = ninst + 8 * nsets;
    for (int k = threadIdx.x; k < words; k += blockDim.x) s_prog[k] = prog[k];
    __syncthreads();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl) return;
    if (out && counts[i] == 0) return;
    // the scanned block: leading NULs skipped, cut at the next NUL
    const uint8_t* line = data + pl_start[i];
    const uint32_t len = pl_len[i];
    uint32_t a = 0;
    while (a < len && line[a] == 0) a++;
    uint32_t e = a;
    while (e < len && line[e] != 0) e++;
    PikeView view;
    view.insts = s_prog;
    view.sets = s_prog + ninst;
    view.ninst = ninst;
    view.start = start_pc;
    uint32_t found = 0;
    const uint32_t room = out ? counts[i] : 0u;
    SpanRec* dst = out ? out + off[i] : nullptr;
    const bool ok = pike_spans(view, line + a, e - a, [&](uint32_t s, uint32_t t) {
        if (found < room) dst[found] = SpanRec{(uint32_t)i, s, t};
        found++;
    });
    if (!ok) {
        found = 1;
        if (out) dst[0] = SpanRec{(uint32_t)i, kSpanOverBudget, kSpanOverBudget};
    }
    if (!out) counts[i] = found;
}

}  // namespace gpugrep
