// Context stage of a scan with context lines (grep -A/-B/-C): which lines of a segment are output.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
//
// With P(k) the number of selected lines before line k, line i is output iff a selected line lies within A lines before or
// B lines after it, P(i+B+1) - P(i-A) > 0, or it is one of the segment's first A or last B lines: those are candidates for
// the selected lines of the neighbouring segments, and the host decides (capi.cpp ContextFilter).  The edge rule also makes
// the window of every other line lie inside the segment, so the test needs no clamping, and the width costs nothing.
// Output lines that are not selected carry kLineContext (engine.hpp) in LineRec.len.
//   fast path:    k_mark_lines -> scan of selected-word popcounts -> k_context_bits -> scan of output-word popcounts
//                 -> k_newline_positions (newline chunks only) -> k_emit_context
//   general path: k_match_pl_simple -> scan of its flags -> k_context_flags -> scan -> k_emit_pl_context
#pragma once

namespace gpugrep {

__device__ __forceinline__ bool context_output(size_t i, size_t nlines, uint32_t before, uint32_t after, unsigned long long p_lo_excl,
                                               unsigned long long p_hi_excl) {
    return i < after || i + before >= nlines || p_hi_excl > p_lo_excl;
}

// Selected lines of bitmap word w of a fast-path segment: the marked (matched) lines, or with invert the unmarked ones
// that exist.
__device__ __forceinline__ uint32_t selected_word(const uint32_t* bits, size_t w, size_t nlines, bool invert) {
    const uint32_t b = bits[w];
    if (!invert) return b;
    const size_t tail = nlines & 31u;
    const uint32_t valid = (w == nlines / 32 && tail) ? (1u << tail) - 1u : 0xffffffffu;
    return ~b & valid;
}

struct LoadSelectedPopc {   // selected lines per bitmap word
    const uint32_t* p;
    size_t nlines;
    bool invert;
    __device__ unsigned long long operator()(size_t i) const { return (unsigned long long)__popc(selected_word(p, i, nlines, invert)); }
};

// One thread per line, one warp per bitmap word: bit i of `out` is set iff line i is output.  `word_prefix`: exclusive
// prefix of LoadSelectedPopc, `total`: its sum.
__global__ void __launch_bounds__(256) k_context_bits(const uint32_t* __restrict__ bits, size_t nlines, bool invert,
                                                      const unsigned long long* __restrict__ word_prefix, const unsigned long long* __restrict__ total,
                                                      uint32_t before, uint32_t after, uint32_t* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nwords = (nlines + 31) / 32;
    if ((i >> 5) >= nwords) return;   // whole warps: the ballot below needs every lane of the word
    auto prefix = [&](size_t k) -> unsigned long long {   // P(k), 0 <= k <= nlines
        const size_t w = k >> 5;
        if (w >= nwords) return *total;
        return word_prefix[w] + (unsigned long long)__popc(selected_word(bits, w, nlines, invert) & ((1u << (k & 31u)) - 1u));
    };
    bool o = false;
    if (i < nlines) o = context_output(i, nlines, before, after, i >= after ? prefix(i - after) : 0ull,
                                       i + before < nlines ? prefix(i + before + 1) : 0ull);
    const uint32_t word = __ballot_sync(0xffffffffu, o);
    if ((threadIdx.x & 31u) == 0) out[i >> 5] = word;
}

// One thread per line: output line i becomes record (output lines before i).  The NUL hint is set on every record, as in
// k_emit_unmarked.
__global__ void __launch_bounds__(256) k_emit_context(const uint32_t* __restrict__ nlpos, size_t nl_total, size_t n, size_t nlines,
                                                      const uint32_t* __restrict__ bits, bool invert, const uint32_t* __restrict__ out_bits,
                                                      const unsigned long long* __restrict__ out_prefix, LineRec* __restrict__ recs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nlines) return;
    const uint32_t w = out_bits[i >> 5], bit = 1u << (i & 31u);
    if (!(w & bit)) return;
    const size_t at = (size_t)out_prefix[i >> 5] + (size_t)__popc(w & (bit - 1u));
    const bool selected = (selected_word(bits, i >> 5, nlines, invert) & bit) != 0;
    uint32_t st, len;
    line_extent(nlpos, nl_total, n, i, st, len);
    recs[at] = LineRec{(uint32_t)i, st, len | kHasNulBit | (selected ? 0u : kLineContext)};
}

// General path, one thread per pseudo-line: out[i] = 1 iff pseudo-line i is output.  `prefix`: exclusive prefix of the
// selected flags (k_match_pl_simple), `total`: their sum.
__global__ void k_context_flags(const unsigned long long* __restrict__ prefix, const unsigned long long* __restrict__ total, size_t npl,
                                uint32_t before, uint32_t after, uint8_t* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl) return;
    const size_t hi = i + before + 1;
    out[i] = context_output(i, npl, before, after, i >= after ? prefix[i - after] : 0ull, hi < npl ? prefix[hi] : (hi == npl ? *total : 0ull)) ? 1 : 0;
}

__global__ void k_emit_pl_context(const uint32_t* __restrict__ pl_start, const uint32_t* __restrict__ pl_len, size_t npl,
                                  const uint8_t* __restrict__ selected, const uint8_t* __restrict__ out, const unsigned long long* __restrict__ off,
                                  LineRec* __restrict__ recs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl || !out[i]) return;
    recs[off[i]] = LineRec{(uint32_t)i, pl_start[i], pl_len[i] | (selected[i] ? 0u : kLineContext)};
}

}  // namespace gpugrep
