// Pattern compiler back end: AST -> Thompson NFA -> byte-class-compressed, minimised DFA tables.
//
// Semantics reproduced (what the reference gets from hs_compile_multi(..., HS_MODE_BLOCK, ...) + hs_scan,
// reference hyperscanner.c:136,217): for a block, report (match id, END offset) for every offset at which
// some expression with that id has a non-empty match ending there.  The DFA is the determinised union of
// ".*(pattern_i)" over a group of patterns; each state carries the set of patterns whose match ended just
// BEFORE the byte that led into the state (reports are delayed by one symbol so that one byte of look-ahead
// resolves $, \b, \B, \z); a synthetic end-of-data symbol flushes matches ending at the block end.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "regex.hpp"

namespace gpugrep {

struct NfaInst {
    enum Op : uint8_t { Byte, Split, Assert, Match } op;
    int x = -1, y = -1;   // Byte/Assert: x = next.  Split: x, y.
    int arg = 0;          // Byte: index into Nfa::sets.  Assert: AssertKind.  Match: pattern index (in the group)
};

struct Nfa {
    std::vector<NfaInst> prog;
    std::vector<ByteSet> sets;       // deduplicated byte sets referenced by Byte instructions
    std::vector<int> starts;         // entry instruction per pattern
    bool uses_line_ctx = false;      // any BeginBuffer/BeginLine assert
    bool uses_word_ctx = false;      // any \b / \B
    bool uses_lookahead = false;     // any EndLine/EndBuffer/\b/\B
};

// Append pattern `ast` as pattern number `index` of the group.  Returns false if the program would exceed
// `max_insts` (bounded repeats are expanded by copying).  Every Split lists the branch a backtracking matcher tries first
// as x: the earlier alternative, and for a repeat the greedy choice, or with `lazy` the lazy choice of a repeat marked so
// (the span program, pike_vm.hpp).  The automata do not depend on the order, and are built without `lazy`.
bool nfa_add_pattern(Nfa& nfa, const Node& ast, int index, size_t max_insts, bool lazy = false);

struct Dfa {
    // alphabet
    uint8_t byte_class[256];         // byte -> class
    int num_classes = 0;             // byte classes; column `num_classes` is the end-of-data symbol
    int stride = 0;                  // num_classes + 1
    // states: 0 = start of block.  trans[s * stride + c]
    std::vector<uint32_t> trans;
    int num_states = 0;
    // accept info: accept_of[s] = index into accept sets (0 = none)
    std::vector<uint32_t> accept_of;
    std::vector<std::vector<int>> accept_sets;  // [0] is empty; pattern indices within the group, sorted
    int first_accept = 0;            // states >= first_accept have accept_of != 0 (states are renumbered so)
    int sink_match = -1;             // simple mode: absorbing "line matched" state, else -1
    int dead = -1;                   // absorbing non-accepting state that can never reach an accept, else -1
    bool simple = false;
    // Entry states for a walk that starts in the middle of a line (local verification): the byte before the first
    // consumed byte was a non-word / a word character.  Equal to 0 when the patterns cannot observe the difference.
    int entry_mid_other = 0, entry_mid_word = 0;
    // States < idle_end have no partial match in progress (only the implicit ".*" restart): once a walk is idle
    // past a prefilter hit, no match containing that hit can still complete.  State 0 is always idle.
    int idle_end = 1;
    // depth[s]: no partial match in progress in state s began more than depth[s] bytes ago (255: unbounded - a loop).
    // Finer than "idle": a local walk that is `k` bytes past the last gram of its chunk can stop as soon as depth < k,
    // because whatever is still in progress began behind that gram and belongs to a later candidate.  From the longest
    // path of the NFA to every item of the state's kernel; the maximum over the states that minimisation merges.
    std::vector<uint8_t> depth;
};

struct DfaBuildOptions {
    bool simple = false;         // stop at the first report (all patterns SINGLEMATCH with one shared id)
    size_t max_states = 60000;
};

// Tables of the bit-parallel NFA fallback (see nfa_sim.hpp) for ONE pattern.
struct NfaTables {
    int positions = 0, words = 0;
    std::vector<uint32_t> reach;          // [256][words]
    std::vector<uint32_t> follow;         // [positions][12][words]
    std::vector<uint32_t> follow_match;   // [positions][12]
    std::vector<uint32_t> restart;        // [4][4][words]
};
// `nfa` must hold exactly one pattern.  Returns false if it has more positions than the simulation supports.
bool build_nfa_tables(const Nfa& nfa, NfaTables& out);

// Returns false when the state budget is exceeded (caller splits the group).
bool build_dfa(const Nfa& nfa, const DfaBuildOptions& opt, Dfa& out);

}  // namespace gpugrep
