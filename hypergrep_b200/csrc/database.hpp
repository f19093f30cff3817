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

// Report table of a fixed-string set compiled for reports (gpugrep_literal_report_scan_*): every distinct (class, folded
// bytes) literal that can lie inside a line is one node, numbered in (class, byte) order.  Unlike LiteralSet nothing is
// pruned: every literal that matches at a position reports.  At a text position the matching nodes of a class are the
// parent chain of the greatest node of the two-byte bucket that is not above the text, cut where a node is longer than
// the common prefix of that node and the text (DESIGN.md section 9).
constexpr uint32_t kNoLiteral = 0xffffffffu;
struct LiteralReports {
    std::vector<uint8_t> bytes;          // the nodes, caseless ones folded to lower case (A-Z only)
    std::vector<uint32_t> off, len;      // per node: offset into bytes, length
    std::vector<uint8_t> caseless;       // per node: class
    std::vector<uint32_t> parent;        // per node: its longest proper prefix that is a node of its class, or kNoLiteral
    std::vector<uint32_t> order;         // nodes of >= 2 bytes, in node order
    std::vector<uint32_t> bucket;        // [class][65537]: the nodes of `order` whose first two bytes are (b0 << 8 | b1) are
                                         // order[bucket[k] .. bucket[k + 1])
    std::vector<uint32_t> one;           // [class][256]: the node of the one-byte literal b, or kNoLiteral
    std::vector<uint32_t> report_begin;  // per node, + 1: its (id, singlematch) descriptors are
                                         // Database::reports[report_begin[k] .. report_begin[k + 1])
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
    // fixed-string set compiled for reports: `literals` selects the lines (simple stays true), then `literal_reports` finds
    // every (node, end) in them and `reports` expands a node to its ids
    bool literal_reports = false;
    LiteralReports lit_reports;
    // fixed-string set compiled for whole-word / whole-line scans (gpugrep_literal_whole_scan_*): `literals` selects the
    // lines, then `lit_reports` (ids 0) decides which of them hold a literal as a word or as the whole line
    bool literal_whole = false;
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
// Fixed strings with reports (gpugrep_literal_report_scan_*): the set of compile_literal_database plus the report table.
// SINGLEMATCH is honoured, and literals that share an id must agree on it (4 otherwise, as compile_database).  `ids` null:
// all 0.  Cached apart from both kinds above.
int compile_literal_report_database(const char* const* literals, const unsigned* flags, const unsigned* ids, unsigned n,
                                    std::shared_ptr<Database>& out, std::string& error);
std::shared_ptr<Database> cached_literal_report_database(const char* const* literals, const unsigned* flags, const unsigned* ids,
                                                         unsigned n, int& rc, std::string& error);
// Fixed strings for whole-word and whole-line scans (gpugrep_literal_whole_scan_*): the set of compile_literal_database
// plus the report table of every literal, not only the prefix-free kept ones (`foo` must not hide `foobar`).  One database
// serves both modes.  Cached apart from the three kinds above.
int compile_literal_whole_database(const char* const* literals, const unsigned* flags, unsigned n, std::shared_ptr<Database>& out,
                                   std::string& error);
std::shared_ptr<Database> cached_literal_whole_database(const char* const* literals, const unsigned* flags, unsigned n, int& rc,
                                                        std::string& error);

inline uint8_t fold_ascii(uint8_t b) { return (uint8_t)((unsigned)b - 'A' < 26u ? b | 0x20u : b); }

}  // namespace gpugrep
