// General-path kernels: newline positions, pseudo-line table (gzgets splitting), per-line matching, record / event emit.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
#pragma once

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// GENERAL PATH kernels
// ------------------------------------------------------------------------------------------------------------
// warp per 512-byte block: write the offset of every '\n' at its global rank.  `nlmask` (optional, the newline-chunk masks of
// k_stream): only the 16-byte chunks that hold a newline are read.
__global__ void __launch_bounds__(256) k_newline_positions(const uint8_t* __restrict__ data, size_t n, size_t nblk, const unsigned long long* __restrict__ meta,
                                                           const unsigned long long* __restrict__ prefix, uint32_t* __restrict__ nlpos,
                                                           const uint32_t* __restrict__ nlmask = nullptr) {
    const int lane = threadIdx.x & 31;
    size_t g = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= nblk) return;
    size_t off = g * 512 + (size_t)lane * 16;
    uint32_t m = 0;
    if (off < n && (!nlmask || ((nlmask[g] >> lane) & 1u))) {
        uint4 v = ld_chunk(data, off, n);
        m = newline_mask16(v);
        if (off + 16 > n) m &= (1u << (n - off)) - 1u;
    }
    uint32_t cnt = __popc(m), incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    size_t at = (size_t)newlines_before_block(prefix, meta, g) + (incl - cnt);
    while (m) {
        int b = __ffs(m) - 1;
        m &= m - 1;
        nlpos[at++] = (uint32_t)(off + b);
    }
}

__device__ __forceinline__ void line_extent(const uint32_t* nlpos, size_t nl_total, size_t n, size_t i, uint32_t& start, uint32_t& len) {
    start = i ? nlpos[i - 1] + 1 : 0;
    uint32_t end = i < nl_total ? nlpos[i] + 1 : (uint32_t)n;
    len = end - start;
}

// pseudo-lines per line for a gzgets buffer of buffer_size (limit = buffer_size - 1 bytes per read)
__global__ void k_count_pseudo_lines(const uint32_t* __restrict__ nlpos, size_t nl_total, size_t n, size_t nlines, uint32_t limit,
                                     uint32_t* __restrict__ npl, Totals* totals) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nlines) return;
    uint32_t st, len;
    line_extent(nlpos, nl_total, n, i, st, len);
    npl[i] = len / limit + (len % limit != 0u);   // no 32-bit overflow of len + limit for huge buffer_size
    if (len > limit) atomicMax(&totals->max_line, len);
}

__global__ void k_build_pseudo_lines(const uint32_t* __restrict__ nlpos, size_t nl_total, size_t n, size_t nlines, uint32_t limit,
                                     const unsigned long long* __restrict__ ploff, uint32_t* __restrict__ pl_start, uint32_t* __restrict__ pl_len) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nlines) return;
    uint32_t st, len;
    line_extent(nlpos, nl_total, n, i, st, len);
    size_t at = ploff ? (size_t)ploff[i] : i;
    while (len > 0) {
        uint32_t take = len < limit ? len : limit;
        pl_start[at] = st;
        pl_len[at] = take;
        at++;
        st += take;
        len -= take;
    }
}

__global__ void __launch_bounds__(128) k_match_pl_simple(DbView db, const uint8_t* __restrict__ data, const uint32_t* __restrict__ pl_start,
                                                         const uint32_t* __restrict__ pl_len, size_t npl, uint8_t* __restrict__ flags, bool invert) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl) return;
    size_t st = pl_start[i];
    flags[i] = block_matches<true>(db, data, st, st + pl_len[i]) != invert ? 1 : 0;   // invert: select the lines without a match
}

__global__ void k_emit_pl_simple(const uint32_t* __restrict__ pl_start, const uint32_t* __restrict__ pl_len, size_t npl, const uint8_t* __restrict__ flags,
                                 const unsigned long long* __restrict__ off, LineRec* __restrict__ recs) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl || !flags[i]) return;
    recs[off[i]] = LineRec{(uint32_t)i, pl_start[i], pl_len[i]};
}

__global__ void __launch_bounds__(128) k_match_pl_events(DbView db, const uint8_t* __restrict__ data, const uint32_t* __restrict__ pl_start,
                                                         const uint32_t* __restrict__ pl_len, size_t npl, uint32_t* __restrict__ counts,
                                                         const unsigned long long* __restrict__ off, EventRec* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npl) return;
    size_t st = pl_start[i];
    uint32_t len = pl_len[i];
    if (out) {
        if (counts[i]) block_events(db, data, st, st + len, (uint32_t)i, (uint32_t)st, len, out + off[i]);
    } else {
        counts[i] = block_events(db, data, st, st + len, (uint32_t)i, (uint32_t)st, len, nullptr);
    }
}

// warp per record: copy matched line bytes into a packed buffer (device-resident scans with a callback)
__global__ void k_gather_lines(const uint8_t* __restrict__ data, const uint32_t* __restrict__ starts, const uint32_t* __restrict__ lens,
                               const unsigned long long* __restrict__ outoff, size_t count, uint8_t* __restrict__ out) {
    size_t r = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= count) return;
    const uint8_t* src = data + starts[r];
    uint8_t* dst = out + outoff[r];
    uint32_t len = lens[r];
    for (uint32_t k = lane; k < len; k += 32) dst[k] = src[k];
    if (lane == 0) dst[len] = 0;
}

}  // namespace gpugrep
