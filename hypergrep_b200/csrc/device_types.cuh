// Device-side views of the compiled database, segment totals and constants shared by all kernels.
// Part of the CUDA engine (engine.cu includes these files in this order; they form one translation unit).
#pragma once

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// device-side views
// ------------------------------------------------------------------------------------------------------------
struct GroupDev {
    const uint16_t* trans;      // [states][stride]
    const uint8_t* cls;         // [256] byte -> class
    const uint32_t* accept_of;  // [states] (general mode)
    const uint16_t* flat;       // [states][256] byte-indexed transitions (local verification: one load per byte), or null
    const uint16_t* eod_next;   // [states] transition on end-of-data (with `flat`)
    // The same byte-indexed view, class-compressed for shared memory (k_verify_smem): ctab[state * (crow / 2) + class],
    // cmap[byte] = class ('\n' and NUL have classes of their own); null when it does not fit.
    const uint16_t* ctab;
    const uint8_t* cmap;
    uint32_t crow, cstates;     // bytes per row of ctab, rows
    // depth[state] (Dfa::depth): how long ago the oldest partial match of the state can have begun, 255 = unbounded; the
    // copy for shared memory sits behind ctab (cdepth_off: its offset from ctab in 32-bit words)
    const uint8_t* depth;
    uint32_t cdepth_off;
    uint32_t stride, eod, first_accept, dead, accept_base, idle_end, mid_other, mid_word;
};

struct DbView {
    const GroupDev* groups;
    int ngroups;
    const NfaView* nfas;   // patterns simulated as bit-parallel NFAs (general path only)
    int nnfa;
};

constexpr uint32_t kInvalidLen = 0xffffffffu;   // LineRec.len of a record the host must drop (NUL re-check failed)
constexpr uint32_t kHasNulBit = 0x80000000u;    // LineRec.len flag: the line contains NUL bytes (host applies the strip/cut rule)
constexpr unsigned int kFallbackFlags = 7u;      // Totals::flags bits that send a fast-path segment to the general path
constexpr unsigned int kSegmentNulFlag = 8u;     // Totals::flags bit: some byte of the segment is NUL

struct Totals {
    unsigned long long meta_total;   // candidates << 32 | newlines
    unsigned long long rec_total;    // records to emit (fast path) / generic scan totals
    unsigned long long aux_total;
    // bit0: a 64 KiB super-block without newline; bit1: candidate overflow; bit2: record overflow (bits 0-2 send the segment
    // to the general path); bit3: the segment holds a NUL byte (k_stream)
    unsigned int flags;
    unsigned int last_byte;
    unsigned int max_line;           // general path: longest line
    unsigned int survivors;          // fast path: candidates that k_confirm kept (length of the survivor list)
};

#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            error = std::string(#expr) + ": " + cudaGetErrorString(e_);                     \
            return 7;                                                                       \
        }                                                                                   \
    } while (0)

}  // namespace gpugrep
