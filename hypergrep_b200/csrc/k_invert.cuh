// Complement stage of an inverted fast-path scan (grep -v): the pseudo-lines that no record of the fast path matched.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
//   k_mark_lines -> scan of per-word popcounts -> k_newline_positions (newline chunks only) -> k_emit_unmarked
// On the fast path pseudo-lines are '\n'-terminated lines (no line needs gzgets splitting), so line i spans
// (nlpos[i-1], nlpos[i]] and the last line without '\n' ends at n.
#pragma once

namespace gpugrep {

// bit `line` of `bits` for every valid record (repeats and failed NUL re-checks carry kInvalidLen and mark nothing)
__global__ void __launch_bounds__(256) k_mark_lines(const LineRec* __restrict__ recs, size_t nrec, uint32_t* __restrict__ bits) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nrec; i += (size_t)gridDim.x * blockDim.x) {
        const LineRec r = recs[i];
        if (r.len != kInvalidLen) atomicOr(&bits[r.line >> 5], 1u << (r.line & 31u));
    }
}

struct LoadPopc {   // matched lines per bitmap word
    const uint32_t* p;
    __device__ unsigned long long operator()(size_t i) const { return (unsigned long long)__popc(p[i]); }
};

// One thread per line: an unmarked line i becomes record i - (marked lines before i).  The NUL hint is set on every record
// (the text is not read here): the host applies the strip rule to each delivered line, as it does for general-path records.
__global__ void __launch_bounds__(256) k_emit_unmarked(const uint32_t* __restrict__ nlpos, size_t nl_total, size_t n, size_t nlines,
                                                       const uint32_t* __restrict__ bits, const unsigned long long* __restrict__ word_prefix,
                                                       LineRec* __restrict__ recs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nlines) return;
    const uint32_t w = bits[i >> 5], below = w & ((1u << (i & 31u)) - 1u);
    if ((w >> (i & 31u)) & 1u) return;
    const size_t at = i - ((size_t)word_prefix[i >> 5] + (size_t)__popc(below));
    uint32_t st, len;
    line_extent(nlpos, nl_total, n, i, st, len);
    recs[at] = LineRec{(uint32_t)i, st, len | kHasNulBit};
}

}  // namespace gpugrep
