// Pattern compiler front end: PCRE-subset parser -> AST.
//
// Replaces the reference's call into Intel Hyperscan's compiler, hs_compile_multi()
// (reference hypergrep/lib/c/hyperscanner.c:136), for the regex subset Hyperscan documents as supported
// (SURVEY.md Appendix A).  Written from scratch; Hyperscan's source is not available to this build.
#pragma once
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

namespace gpugrep {

// hs_compile.h flag bits (reference hypergrep/utils.py:9-13)
enum : unsigned { FLAG_CASELESS = 1, FLAG_DOTALL = 2, FLAG_MULTILINE = 4, FLAG_SINGLEMATCH = 8 };

struct ByteSet {
    uint64_t w[4] = {0, 0, 0, 0};
    void set(unsigned b) { w[b >> 6] |= 1ull << (b & 63); }
    void set_range(unsigned lo, unsigned hi) { for (unsigned b = lo; b <= hi; b++) set(b); }
    bool test(unsigned b) const { return (w[b >> 6] >> (b & 63)) & 1; }
    bool any() const { return (w[0] | w[1] | w[2] | w[3]) != 0; }
    int count() const { return __builtin_popcountll(w[0]) + __builtin_popcountll(w[1]) + __builtin_popcountll(w[2]) + __builtin_popcountll(w[3]); }
    ByteSet operator|(const ByteSet& o) const { ByteSet r; for (int i = 0; i < 4; i++) r.w[i] = w[i] | o.w[i]; return r; }
    ByteSet operator&(const ByteSet& o) const { ByteSet r; for (int i = 0; i < 4; i++) r.w[i] = w[i] & o.w[i]; return r; }
    ByteSet operator~() const { ByteSet r; for (int i = 0; i < 4; i++) r.w[i] = ~w[i]; return r; }
    ByteSet& operator|=(const ByteSet& o) { for (int i = 0; i < 4; i++) w[i] |= o.w[i]; return *this; }
    bool operator==(const ByteSet& o) const { return std::memcmp(w, o.w, sizeof(w)) == 0; }
    bool operator!=(const ByteSet& o) const { return !(*this == o); }
    bool operator<(const ByteSet& o) const { return std::memcmp(w, o.w, sizeof(w)) < 0; }
    static ByteSet all() { ByteSet r; for (int i = 0; i < 4; i++) r.w[i] = ~0ull; return r; }
    static ByteSet of(unsigned b) { ByteSet r; r.set(b); return r; }
};

enum class AssertKind : uint8_t {
    BeginBuffer,   // \A, ^ without MULTILINE
    BeginLine,     // ^ with MULTILINE: offset 0 or after '\n' (also the '\n' that ends the block: Hyperscan semantics)
    EndBuffer,     // \z
    EndLine,       // $ with MULTILINE: before '\n' or at end of block
    WordBoundary,  // \b
    NotWordBoundary  // \B
};

enum class NodeKind : uint8_t { Empty, Set, Concat, Alt, Repeat, Assert };

struct Node;
using NodePtr = std::unique_ptr<Node>;
struct Node {
    NodeKind kind = NodeKind::Empty;
    ByteSet set;                 // Set
    std::vector<NodePtr> kids;   // Concat / Alt / Repeat(1 kid)
    int min = 0, max = 0;        // Repeat; max < 0 = unbounded
    bool lazy = false;           // Repeat written with a lazy `?` (same language; only the span program's Split order differs)
    AssertKind assert_kind = AssertKind::BeginBuffer;
};

struct ParseResult {
    NodePtr root;        // null on failure
    std::string error;   // human-readable reason (the C boundary only reports code 4, like the reference)
};

// Parse one pattern (raw bytes, NUL-free) under HS_FLAG_{CASELESS,DOTALL,MULTILINE}.
ParseResult parse_regex(const std::string& pattern, unsigned flags);

// True if the pattern can match without consuming a byte, assertions aside (Hyperscan: "Pattern matches empty
// buffer; use HS_FLAG_ALLOWEMPTY").
bool matches_empty_buffer(const Node& n);

bool is_word_byte(unsigned b);

}  // namespace gpugrep
