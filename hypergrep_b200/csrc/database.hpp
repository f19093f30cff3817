// Compiled pattern database: what hs_compile_multi() produces in the reference (hyperscanner.c:126-142),
// rebuilt as DFA groups + literal prefilter tables laid out for the CUDA engine.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "automata.hpp"
#include "prefilter.hpp"

namespace gpugrep {

struct PatternInfo {
    std::string source;
    unsigned flags = 0;
    unsigned id = 0;
};

struct DfaGroup {
    Dfa dfa;
    std::vector<int> members;   // group-local pattern index -> database pattern index
};

// One (id, singlematch) report descriptor; accept sets of every group are flattened into lists of these.
struct ReportDesc {
    unsigned id;
    unsigned singlematch;
};

// A pattern whose own DFA exceeds the state budget: simulated as a bit-parallel NFA (general path only).
struct NfaPattern {
    int pattern = 0;          // index into Database::patterns
    NfaTables tables;
    uint32_t report_begin = 0;   // its single report: Database::reports[report_begin]
};

// Fixed-string set (grep -F): the literals that can select a line, without automata.  A literal with an inner '\n' never
// matches and is dropped; so is one that has another literal of its class as a prefix (the shorter one matches wherever the
// longer one does).  What is kept is prefix-free per class, so at any text position at most one literal of a class can
// match: the largest one not above the text, found by binary search.
struct LiteralSet {
    std::vector<uint8_t> bytes;          // the kept literals, caseless ones folded to lower case (A-Z only)
    std::vector<uint32_t> off, len;      // per kept literal: offset into bytes, length
    std::vector<uint8_t> caseless;       // per kept literal: class 1 (compared folded) or 0 (exact)
    std::vector<uint32_t> rank;          // per kept literal: position in `order` (sorted by folded bytes within the class)
    std::vector<uint32_t> order;         // class 0 literals of >= 2 bytes in byte order, then those of class 1
    std::vector<uint32_t> bucket;        // [class][65537]: the literals of `order` whose first two bytes are (b0 << 8 | b1) are
                                         // order[bucket[k] .. bucket[k + 1])
    std::vector<uint32_t> one;           // [class][8]: bitmap of the one-byte literals
    unsigned given = 0;                  // literals passed in
};

struct Database {
    std::vector<PatternInfo> patterns;
    std::vector<NfaPattern> nfas;
    // simple: every pattern has SINGLEMATCH and all share one id -> "does any pattern match this line?"
    bool simple = false;
    unsigned simple_id = 0;
    std::vector<DfaGroup> groups;
    // event mode: accept set k of group g -> reports[report_begin[g][k] .. report_begin[g][k+1])
    std::vector<std::vector<uint32_t>> report_begin;
    std::vector<ReportDesc> reports;
    FactorSet factors;       // required factors per pattern (input of the prefilter builder)
    Prefilter prefilter;     // statically chosen windows (used when no input sample is available)
    std::string key;   // cache key: patterns + flags + ids
    bool literal = false;   // fixed-string set: no groups, `literals` holds what a line is matched against
    LiteralSet literals;
};

// Return codes follow the reference's enum (hyperscanner.c:25-33): 0 ok, 4 = HYPERSCANNER_DB for any rejection.
// `error` receives a human-readable reason (printed to stderr by the boundary, never returned).
int compile_database(const char* const* patterns, const unsigned* flags, const unsigned* ids, unsigned n,
                     std::shared_ptr<Database>& out, std::string& error);

// Process-wide cache (the reference recompiles per call, hyperscanner.c:296; SURVEY.md §8f-3).
std::shared_ptr<Database> cached_database(const char* const* patterns, const unsigned* flags, const unsigned* ids,
                                          unsigned n, int& rc, std::string& error);

// Fixed strings (gpugrep_literal_scan_*): `n` >= 1 non-empty literals, flags CASELESS (honoured) and DOTALL / MULTILINE /
// SINGLEMATCH (accepted, they change nothing).  Returns 0 or 4 like compile_database.
int check_literals(const char* const* literals, const unsigned* flags, unsigned n, std::string& error);
int compile_literal_database(const char* const* literals, const unsigned* flags, unsigned n, std::shared_ptr<Database>& out,
                             std::string& error);
// Cached like cached_database, apart from it: the literal "a.b" is not the regex "a.b".
std::shared_ptr<Database> cached_literal_database(const char* const* literals, const unsigned* flags, unsigned n, int& rc,
                                                  std::string& error);

inline uint8_t fold_ascii(uint8_t b) { return (uint8_t)((unsigned)b - 'A' < 26u ? b | 0x20u : b); }

}  // namespace gpugrep
