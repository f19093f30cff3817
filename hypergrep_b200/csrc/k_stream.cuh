// K1, the streaming kernel: newline counts and gram-table lookups per 512-byte block (the roofline kernel).
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
#pragma once

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// K1: streaming kernel.  One warp owns four consecutive 512-byte blocks per step: 4 x (32 x 16-byte) coalesced
// loads in flight, newline count (SWAR + popc + warp reduce) and, when the prefilter is on, one gram-table lookup
// per sampled 4-byte gram (shared-memory table of exact keys, or a bloom bitmap for huge gram sets).
// Output: meta[block] = newline_count << 32 | ballot(lanes whose 16-byte chunk has a gram hit).
// STRIDE: sample every STRIDE-th byte position (4, 2, 1).  MODE: 0 no prefilter, 1 exact keys, 2 bloom byte table.
// Second output: nlmask[block] = ballot(lanes whose 16-byte chunk holds at least one '\n'); the emit kernel finds line
// extents and line numbers from these words instead of searching the text again.
// NUL: third output, Totals::flags bit 3 when some byte in [0, n) is NUL.  The count-only emit kernel then needs no line
// extents and no per-line NUL scans in a segment without one (log text has none).  One sticky register per thread, one
// vote per warp at the end.  Only count-only scans test: at stride 4 the test costs the kernel 7 % (0.457 -> 0.491 ms per
// 2 GiB for configs[0], B200), more than the NUL scans it saves a scan with records.
// Algorithmic traffic: 1 byte read per input byte + 12 bytes written per 512.
// ------------------------------------------------------------------------------------------------------------
// Gram lookups of one 16-byte chunk.  MODE 1: two-choice table of exact 32-bit keys; the table is replicated
// 2^rshift times with the copies interleaved word by word, and a lane only ever reads copy (lane mod 2^rshift):
// with 32 copies every lane stays in its own shared-memory bank and the loads are conflict-free.
// Byte offset of slot h for this lane = ((gram * mul) >> shift) & amask | replica4, where replica4 = 4 * copy.
__device__ __forceinline__ uint32_t lds32(uint32_t shared_addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(shared_addr));
    return v;
}

__device__ __forceinline__ uint32_t lds8(uint32_t shared_addr) {
    uint32_t v;
    asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(shared_addr));
    return v;
}

// c1 / c2: shared-window address of table half 1 / 2 (aligned to the size of a half) OR-ed with 4 * copy of this lane,
// so that an address is formed by ONE logic op: ((product >> shift) & amask) | c.
// (Measured and dropped, profiles/README.md: the table index as mulhi(product, 2^k) on the FMA pipe instead of a shift -
// IMAD.HI is the slower instruction, 0.545 -> 0.585 ms per 2 GiB.)
template <int STRIDE, bool FOLD, int MODE, int NODD>
__device__ __forceinline__ bool probe_chunk(const uint4& v, uint32_t next, const uint32_t* __restrict__ tab, const ProbeParams& pp, uint32_t c1,
                                            uint32_t c2) {
    if (MODE == 0) return false;
    uint32_t w[5] = {v.x, v.y, v.z, v.w, next};
    if (FOLD) {
#pragma unroll
        for (int i = 0; i < 5; i++) w[i] |= 0x20202020u;
    }
    uint32_t miss = 0xffffffffu;   // min over all lookups of (key ^ gram): 0 iff some key matched
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
        for (int s = 0; s < 4; s += STRIDE) {
            uint32_t gram = s == 0 ? w[i] : __funnelshift_r(w[i], w[i + 1], 8 * s);
            if (MODE == 1) {
                uint32_t e1 = lds32((((gram * pp.mul) >> pp.shift) & pp.amask) | c1);
                uint32_t e2 = lds32((((gram * pp.mul2) >> pp.shift) & pp.amask) | c2);
                miss = __vimin3_u32(miss, e1 - gram, e2 - gram);   // differences, not XORs: ptxas can place subtractions on the FMA pipe
            } else {
                // bloom: one byte load, bit (p & 7) of it.  The byte is replicated into all four bytes of a word (one
                // multiply on the FMA pipe) so that the wrap-around shift by p itself lands on the right bit.
                uint32_t p = gram * pp.mul;
                uint32_t b = lds8((p >> pp.shift) + c1);
                bits |= (b * 0x01010101u) >> (p & 31u);
            }
        }
    }
    if (NODD > 0) {
        // the grams at offsets 2, 6, 10, 14 of the chunk against two constants: two multiply-adds and one three-way minimum,
        // no shared-memory traffic
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t gram = __funnelshift_r(w[i], w[i + 1], 16);
            uint32_t x[2];
#pragma unroll
            for (int k = 0; k < 2; k++) asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(x[k]) : "r"(gram), "r"(pp.odd_mul[k]), "r"(pp.odd_add[k]));
            miss = __vimin3_u32(miss, x[0], x[1]);
        }
        return (MODE == 1 ? false : (bits & 1u) != 0u) || miss == 0u;
    }
    return MODE == 1 ? miss == 0u : (bits & 1u) != 0u;
}

// newlines in a 16-byte chunk: four flag words (bit 7 of matching bytes) are merged into one 64-bit word with three
// multiply-adds (FMA pipe) instead of shifts and ORs (ALU pipe, the pipe this kernel saturates first)
__device__ __forceinline__ uint32_t newline_count16_fma(const uint4& v, uint32_t cnl, uint32_t c80) {
    uint32_t a = eq_mask4_r(v.x, cnl, c80), b = eq_mask4_r(v.y, cnl, c80), c = eq_mask4_r(v.z, cnl, c80), d = eq_mask4_r(v.w, cnl, c80);
    unsigned long long acc = a;
    asm("mad.wide.u32 %0, %1, 2, %0;" : "+l"(acc) : "r"(b));
    asm("mad.wide.u32 %0, %1, 4, %0;" : "+l"(acc) : "r"(c));
    asm("mad.wide.u32 %0, %1, 8, %0;" : "+l"(acc) : "r"(d));
    return __popcll(acc);
}

// NUL test of one 16-byte chunk, OR-ed into a sticky word: bit 7 of some byte of acc ends up set iff some word held a zero
// byte (haszero4 without its final mask).  Per word one subtraction, which ptxas can place on the FMA pipe, and one
// three-input logic op: the ALU pipe is the one this kernel saturates first.
__device__ __forceinline__ void nul_accumulate(const uint4& v, uint32_t& acc) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t t;
        asm("mad.lo.u32 %0, %1, 1, 0xfefefeff;" : "=r"(t) : "r"(w[i]));   // w - 0x01010101
        asm("lop3.b32 %0, %1, %2, %0, 0xBA;" : "+r"(acc) : "r"(t), "r"(w[i]));   // acc | (t & ~w)
    }
}

constexpr int kStreamU = 4;   // 512-byte blocks per warp step

// Per-warp constants of the streaming kernel.
struct StreamRegs {
    uint32_t c1, c2, cnl, c80, lane;
};

// One warp step: four full 512-byte blocks (g0 .. g0+3) whose chunks are already in registers.
// (Tried and dropped, profiles/README.md: a CONFIRM variant in which a lane whose chunk passes the bloom table confirms it
// right here with the exact tables of confirm.cuh - for the 10,000-pattern set this kernel went from 0.31 to 2.5 ms per GiB:
// the warp runs the confirmation code, global lookups and all, in nearly every chunk step with a handful of lanes busy.)
template <int STRIDE, bool FOLD, int MODE, int NODD, bool NUL>
__device__ __forceinline__ void stream_group(const uint4 (&v)[kStreamU], uint32_t g0, const uint8_t* __restrict__ data, size_t n,
                                             unsigned long long* __restrict__ meta, uint32_t* __restrict__ nlmask, unsigned long long* __restrict__ gsum,
                                             const uint32_t* __restrict__ s_tab, const ProbeParams& pp, const StreamRegs& r, uint32_t& nul) {
    constexpr int U = kStreamU;
    const uint32_t lane = r.lane;
    uint32_t after = 0;   // first word after the group (only lane 31 needs it, for grams that straddle the end)
    if (MODE != 0 && (STRIDE < 4 || NODD > 0) && lane == 31) {
        size_t off = (size_t)(g0 + U) << 9;
        if (off + 4 <= n) after = *reinterpret_cast<const uint32_t*>(data + off);
        else if (off < n) after = ld_chunk(data, off, n).x;
    }
    uint32_t cnt01, cnt23, masks[U], nlm[U];
    {
        uint32_t c[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            c[u] = newline_count16_fma(v[u], r.cnl, r.c80);
            if (NUL) nul_accumulate(v[u], nul);
            nlm[u] = __ballot_sync(0xffffffffu, c[u] != 0u);
            uint32_t nx = 0;
            if (MODE != 0 && (STRIDE < 4 || NODD > 0)) {
                // first word of the next chunk: lane+1's word of this block, or (lane 31) lane 0's word of the next block
                uint32_t give = (u + 1 < U && lane == 0) ? v[u + 1 < U ? u + 1 : u].x : v[u].x;
                nx = __shfl_sync(0xffffffffu, give, (lane + 1) & 31);
                if (u + 1 == U && lane == 31) nx = after;
            }
            bool hit = probe_chunk<STRIDE, FOLD, MODE, NODD>(v[u], nx, s_tab, pp, r.c1, r.c2);
            masks[u] = __ballot_sync(0xffffffffu, hit);
        }
        cnt01 = __reduce_add_sync(0xffffffffu, c[0] | (c[1] << 16));
        cnt23 = __reduce_add_sync(0xffffffffu, c[2] | (c[3] << 16));
    }
    if (lane == 0) {
        uint4* out = reinterpret_cast<uint4*>(meta + g0);   // g0 is a multiple of 4: 32-byte aligned
        out[0] = make_uint4(masks[0], cnt01 & 0xffffu, masks[1], cnt01 >> 16);
        out[1] = make_uint4(masks[2], cnt23 & 0xffffu, masks[3], cnt23 >> 16);
        *reinterpret_cast<uint4*>(nlmask + g0) = make_uint4(nlm[0], nlm[1], nlm[2], nlm[3]);
        // totals of the group (candidates << 32 | newlines): what the scan over groups reads
        const uint32_t cands = __popc(masks[0]) + __popc(masks[1]) + __popc(masks[2]) + __popc(masks[3]);
        const uint32_t sum = cnt01 + cnt23;
        gsum[g0 / U] = ((unsigned long long)cands << 32) | ((sum & 0xffffu) + (sum >> 16));
    }
}

template <int STRIDE, bool FOLD, int MODE, int NODD, bool NUL>
__global__ void __launch_bounds__(1024) k_stream(const uint8_t* __restrict__ data, size_t n, unsigned long long* __restrict__ meta,
                                                 uint32_t* __restrict__ nlmask, unsigned long long* __restrict__ gsum,
                                                 const uint32_t* __restrict__ table, int table_words, ProbeParams pp,
                                                 unsigned int* __restrict__ flags) {
    extern __shared__ __align__(16) uint32_t s_raw[];
    // exact tables are placed at an address aligned to the size of one half (see probe_chunk); the launch reserves the slack
    uint32_t* s_tab = s_raw;
    uint32_t saddr = (uint32_t)__cvta_generic_to_shared(s_raw);
    if (MODE == 1) {
        uint32_t aligned = (saddr + pp.half_bytes - 1u) & ~(pp.half_bytes - 1u);
        s_tab = s_raw + ((aligned - saddr) >> 2);
        saddr = aligned;
    }
    if (MODE != 0) {
        for (int i = threadIdx.x; i < table_words; i += blockDim.x) s_tab[i] = table[i];
        __syncthreads();
    }
    constexpr int U = kStreamU;
    StreamRegs r;
    r.lane = threadIdx.x & 31;
    const uint32_t lane = r.lane;
    const uint32_t replica4 = (lane & ((1u << pp.rshift) - 1u)) << 2;
    r.c1 = MODE == 1 ? (saddr | replica4) : saddr;
    r.c2 = (saddr + pp.half_bytes) | replica4;
    asm volatile("mov.u32 %0, %0;" : "+r"(r.c1));   // materialise: each table address is then a single (x & amask) | c
    asm volatile("mov.u32 %0, %0;" : "+r"(r.c2));
    // opaque to the optimiser so that they stay in registers (see eq_mask4_r, newline_flags4)
    asm volatile("mov.u32 %0, 0x0a0a0a0a;" : "=r"(r.cnl));
    asm volatile("mov.u32 %0, 0x80808080;" : "=r"(r.c80));
    // block indices fit 32 bits (segments are < 4 GiB): fewer registers than size_t arithmetic
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t nblk = (uint32_t)((n + 511) >> 9);
    const uint32_t nfull = (uint32_t)(n >> 9);   // blocks that lie entirely inside [0, n)
    const uint32_t step = nwarps * U;
    uint32_t nul = 0;   // sticky NUL test (nul_accumulate) of the full blocks

    // ---- main loop: groups of U full blocks, no bounds checks on the data loads
    // The loads of the NEXT group are issued before the current group is processed (twice the bytes in flight per warp:
    // with stride-4 sampling the kernel waits for HBM, not for its lookups).
    uint4 ahead[U];
    const uint8_t* lane_data = data + lane * 16;
    if (warp * U + U <= nfull) {
#pragma unroll
        for (int u = 0; u < U; u++) ahead[u] = ld_stream16(lane_data + ((size_t)(warp * U) << 9) + u * 512);
    }
    for (uint32_t g0 = warp * U; g0 + U <= nfull; g0 += step) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) v[u] = ahead[u];
        const uint32_t g1 = g0 + step;
        if (g1 + U <= nfull) {
#pragma unroll
            for (int u = 0; u < U; u++) ahead[u] = ld_stream16(lane_data + ((size_t)g1 << 9) + u * 512);
        }
        stream_group<STRIDE, FOLD, MODE, NODD, NUL>(v, g0, data, n, meta, nlmask, gsum, s_tab, pp, r, nul);
    }

    // ---- tail: the last (< U) full blocks and the partial block, one block per warp step, bounds-checked; the totals of
    // that last, partial group are added up by its first warp
    const uint32_t tail0 = (nfull / U) * U;
    bool tail_nul = false;
    for (uint32_t g = tail0 + warp; g < nblk; g += nwarps) {
        size_t off = ((size_t)g << 9) + (size_t)lane * 16;
        uint4 v = off < n ? ld_chunk(data, off, n) : make_uint4(0, 0, 0, 0);
        uint32_t nx = 0;
        if (MODE != 0 && (STRIDE < 4 || NODD > 0)) {
            nx = __shfl_down_sync(0xffffffffu, v.x, 1);
            if (lane == 31) {
                size_t o2 = (size_t)(g + 1) << 9;
                nx = o2 < n ? ld_chunk(data, o2, n).x : 0u;
            }
        }
        uint32_t cnt = newline_count16_fma(v, r.cnl, r.c80);
        bool hit = probe_chunk<STRIDE, FOLD, MODE, NODD>(v, nx, s_tab, pp, r.c1, r.c2);
        if (off >= n) hit = false;   // chunks that start at or beyond n can never be candidates
        // the zero padding at and beyond n is not text: only the bytes below n count in the NUL test
        if (NUL) {
            const uint32_t inside = off >= n ? 0u : (off + 16 > n ? (1u << (uint32_t)(n - off)) - 1u : 0xffffu);
            tail_nul |= (byte_mask16(v, 0u) & inside) != 0u;
        }
        uint32_t mask = __ballot_sync(0xffffffffu, hit);
        uint32_t nl = __ballot_sync(0xffffffffu, cnt != 0u);
        uint32_t total = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0) {
            meta[g] = ((unsigned long long)total << 32) | mask;
            nlmask[g] = nl;
            // the tail group has at most U blocks: their totals are accumulated with atomics into a zeroed slot
            atomicAdd(&gsum[tail0 / U], ((unsigned long long)__popc(mask) << 32) | total);
        }
    }
    if (NUL && __any_sync(0xffffffffu, (nul & 0x80808080u) != 0u || tail_nul) && lane == 0) atomicOr(flags, kSegmentNulFlag);
}

}  // namespace gpugrep
