// Leftmost-first match spans (`grep -o`, gpugrep_match_spans): a priority-ordered Thompson simulation (Pike VM) of one
// pattern over one scanned block, reproducing re.finditer(): the leftmost start, then the end that a backtracking matcher
// picks (greedy and lazy quantifiers, alternation order), non-overlapping, each search resuming at the previous match end.
//
// The program is the Thompson NFA of automata.cpp built with lazy repeats honoured (nfa_add_pattern(..., lazy = true)):
// every Split lists its preferred branch first.  Threads are kept in priority order; a fresh thread is seeded at each
// position below all live threads (a later start has lower priority).  The first Match of a search stops the seeding
// and cuts the threads behind it; higher-priority threads run on and may replace the match with a later one.  The search
// ends when no thread is left.  Thompson deduplication by instruction is exact here because the exactness screen
// (gpugrep_span_exact) admits no repeat whose body can match empty.
// The same inline function runs in the span kernel (k_spans.cuh) and in the CPU stand-in of the engine.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "nfa_sim.hpp"   // GPUGREP_HD

namespace gpugrep {

// Program bound of the span route: larger programs keep the re.finditer() path.  The per-thread lists below are sized by it.
constexpr int kPikeMaxInsts = 128;
// Work bound per scanned block: kPikeStepsPerByte * (block length + 1) thread steps (closure visits and list entries) over all
// its searches, and never more than kPikeMaxStepsPerBlock, so that one kernel thread stays bounded whatever buffer_size a
// caller passes (2^25 is the per-byte bound of a block of the default 256 KiB buffer).  A block over its bound yields one
// sentinel span instead of its spans.  What trips it: searches that rescan the block (`a.*b|a` on a long run of `a`), or
// programs near the instruction cap that keep most of their threads alive on long lines.
constexpr uint64_t kPikeStepsPerByte = 128;
constexpr uint64_t kPikeMaxStepsPerBlock = (uint64_t)1 << 25;
constexpr uint32_t kSpanOverBudget = 0xffffffffu;

// Instruction word: op in bits 0-3, arg in bits 4-11 (Byte: set index, Assert: AssertKind), x in bits 12-19, y in bits 20-27.
enum : uint32_t { kPikeByte = 0, kPikeSplit = 1, kPikeAssert = 2, kPikeMatch = 3 };
// AssertKind values of regex.hpp that the screen admits
enum : uint32_t { kPikeBeginBuffer = 0, kPikeWordBoundary = 4, kPikeNotWordBoundary = 5 };

GPUGREP_HD inline uint32_t pike_inst(uint32_t op, uint32_t arg, uint32_t x, uint32_t y) { return op | arg << 4 | x << 12 | y << 20; }

struct PikeView {
    const uint32_t* insts = nullptr;   // [ninst]
    const uint32_t* sets = nullptr;    // [nsets][8]: 256-bit byte sets
    int ninst = 0;
    int start = 0;
};

// Host copy of a program (built by build_pike_program, capi_db.cpp).
struct PikeProgram {
    std::vector<uint32_t> insts;
    std::vector<uint32_t> sets;
    int start = 0;
    PikeView view() const {
        PikeView v;
        v.insts = insts.data();
        v.sets = sets.data();
        v.ninst = (int)insts.size();
        v.start = start;
        return v;
    }
};

// Parses `pattern` without flags and builds its span program; false if it does not pass gpugrep_span_exact.
bool build_pike_program(const char* pattern, PikeProgram& out);

GPUGREP_HD inline bool pike_word(uint32_t b) { return (b - '0' < 10u) || ((b | 0x20u) - 'a' < 26u) || b == '_'; }

namespace pike_detail {

struct List {
    uint8_t pc[kPikeMaxInsts];
    uint32_t start[kPikeMaxInsts];
    uint32_t mark[kPikeMaxInsts / 32];
    int n;
    GPUGREP_HD void clear() {
        n = 0;
        for (int w = 0; w < kPikeMaxInsts / 32; w++) mark[w] = 0;
    }
};

// Adds the epsilon closure of `pc` at position `pos` to `list`, in priority order (depth first, preferred branch first; an
// instruction is taken the first time it is reached).  Only Byte and Match instructions become threads.
GPUGREP_HD inline void add_thread(const PikeView& p, List& list, int pc, uint32_t start, const uint8_t* text, uint32_t len, uint32_t pos,
                                  uint64_t& steps) {
    uint8_t stack[2 * kPikeMaxInsts + 2];
    int top = 0;
    stack[top++] = (uint8_t)pc;
    while (top > 0) {
        const int at = stack[--top];
        steps++;
        if ((list.mark[at >> 5] >> (at & 31)) & 1u) continue;
        list.mark[at >> 5] |= 1u << (at & 31);
        const uint32_t in = p.insts[at];
        const uint32_t op = in & 15u, arg = (in >> 4) & 255u, x = (in >> 12) & 255u, y = (in >> 20) & 255u;
        if (op == kPikeSplit) {
            stack[top++] = (uint8_t)y;
            stack[top++] = (uint8_t)x;
        } else if (op == kPikeAssert) {
            bool ok;
            if (arg == kPikeBeginBuffer) {
                ok = pos == 0;
            } else {
                const bool before = pos > 0 && pike_word(text[pos - 1]);
                const bool after = pos < len && pike_word(text[pos]);
                ok = (arg == kPikeWordBoundary) ? before != after : before == after;
            }
            if (ok) stack[top++] = (uint8_t)x;
        } else {
            list.pc[list.n] = (uint8_t)at;
            list.start[list.n] = start;
            list.n++;
        }
    }
}

}  // namespace pike_detail

// Calls on_span(start, end) for every match of re.finditer() over text[0, len), in order.  Returns false (after possibly
// having reported some spans) when the block needs more than its step budget; the caller then reports the sentinel.
template <class OnSpan>
GPUGREP_HD inline bool pike_spans(const PikeView& p, const uint8_t* text, uint32_t len, OnSpan on_span) {
    using pike_detail::List;
    List lists[2];
    const uint64_t per_byte = kPikeStepsPerByte * ((uint64_t)len + 1);
    const uint64_t budget = per_byte < kPikeMaxStepsPerBlock ? per_byte : kPikeMaxStepsPerBlock;
    uint64_t steps = 0;
    uint32_t from = 0;
    while (from <= len) {
        List* cur = &lists[0];
        List* nxt = &lists[1];
        cur->clear();
        bool matched = false;
        uint32_t best_start = 0, best_end = 0;
        for (uint32_t i = from;; i++) {
            if (!matched) pike_detail::add_thread(p, *cur, p.start, i, text, len, i, steps);
            if (steps > budget) return false;
            if (cur->n == 0) {
                if (matched || i >= len) break;
                cur->clear();   // (the closure may have marked instructions that did not become threads)
                continue;
            }
            nxt->clear();
            const uint32_t b = i < len ? text[i] : 256u;
            for (int k = 0; k < cur->n; k++) {
                steps++;
                const uint32_t in = p.insts[cur->pc[k]];
                if ((in & 15u) == kPikeMatch) {
                    matched = true;
                    best_start = cur->start[k];
                    best_end = i;
                    break;   // lower-priority threads are cut
                }
                // Byte
                if (b < 256u && ((p.sets[((in >> 4) & 255u) * 8 + (b >> 5)] >> (b & 31)) & 1u))
                    pike_detail::add_thread(p, *nxt, (int)((in >> 12) & 255u), cur->start[k], text, len, i + 1, steps);
            }
            if (steps > budget) return false;
            List* t = cur; cur = nxt; nxt = t;
            if (i >= len || (cur->n == 0 && matched)) break;   // (at the end nothing is consumed: the list is empty)
        }
        if (!matched) break;
        on_span(best_start, best_end);
        from = best_end;   // best_end > best_start: the screen admits no pattern that matches empty
    }
    return true;
}

}  // namespace gpugrep
