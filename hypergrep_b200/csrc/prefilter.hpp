// Literal-factor prefilter: the role Hyperscan's FDR/Teddy literal matchers play in front of its automata,
// re-designed for a SIMT machine with no byte shuffle.  Every pattern contributes a REQUIRED FACTOR (a set of short
// class-strings one of which occurs in every match).  For a sampling stride k (4, 2 or 1) a window of 3+k bytes is
// chosen inside every factor alternative; the k four-byte grams of that window - one for each alignment the
// window can have against the sampled text positions - go into a gram table that lives in shared memory.  The
// streaming kernel looks up one gram per sampled position and flags 16-byte chunks with a hit; only lines
// touching flagged chunks are walked by the DFA.  The filter is a superset filter: it may flag lines that do not
// match, never the reverse - so WHICH window is chosen only affects speed, and it is chosen against a histogram of
// the grams in a sample of the input (a window made of "host" or "dur=" would flag every syslog line).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "regex.hpp"

namespace gpugrep {

using ClassString = std::vector<ByteSet>;

// Required factors of a pattern set (static, part of the compiled database).
struct FactorSet {
    bool usable = false;                               // every pattern has a factor of >= 4 bytes
    std::vector<std::vector<ClassString>> factors;     // per pattern: alternatives
    std::vector<size_t> before;                        // per pattern: max bytes between match start and factor start (SIZE_MAX: unbounded)
    std::vector<uint32_t> group_mask;                  // per pattern: bit (g mod 32) of the DFA group(s) the pattern is compiled into (empty: unknown)
    size_t min_len = 0;
    std::string note;
    // Fixed-string sets only (empty for regex sets): per pattern, i.e. per literal, its rank in the byte order of its class
    // and that class (1: caseless).  Their gram tables are not capped by size (they live in global memory) and carry a
    // literal index (Prefilter::lit_begin).
    std::vector<uint32_t> literal_rank;
    std::vector<uint8_t> literal_class;
    bool literal() const { return !literal_rank.empty(); }
};

// 4-gram histogram of a text sample (raw and case-folded), used to pick selective windows.
class GramHistogram {
public:
    void add_sample(const uint8_t* text, size_t n);
    uint32_t count(uint32_t gram, bool folded) const;
    // distinct grams of the sample with their counts
    const std::vector<uint32_t>& keys(bool folded) const { return folded ? folded_.keys : raw_.keys; }
    const std::vector<uint32_t>& counts(bool folded) const { return folded ? folded_.counts : raw_.counts; }
    size_t positions() const { return positions_; }
    uint64_t fingerprint() const { return fingerprint_; }
    struct Table {
        std::vector<uint32_t> keys, counts;
        uint32_t mask = 0;
        void init(size_t capacity_pow2);
        void add(uint32_t key);
        uint32_t get(uint32_t key) const;
    };
private:
    Table raw_, folded_;
    size_t positions_ = 0;
    uint64_t fingerprint_ = 0;
};

struct Prefilter {
    bool enabled = false;
    int stride = 4;             // text positions sampled: multiples of `stride` (4, 2 or 1)
    bool fold_case = false;     // text bytes are OR-ed with 0x20 before lookup (grams stored folded)
    // exact mode: two-choice (cuckoo) table of 32-bit keys.  A gram lives in keys[h1] or keys[slots + h2] with
    // h1 = (gram * hash_mul) >> (32 - log2_slots), h2 = (gram * hash_mul2) >> (32 - log2_slots); 0 = empty slot.
    bool exact = false;
    int log2_slots = 0;
    uint32_t hash_mul2 = 0x85EBCA6Bu;
    std::vector<uint32_t> keys;       // 2 << log2_slots entries
    // The same kind of table without the shared-memory size limit, kept in global memory: the verification kernel uses it
    // to find the gram hits of a flagged chunk again, EXACTLY (a chunk flagged only by a bloom collision is dropped there).
    std::vector<uint32_t> confirm_keys;   // 2 << confirm_log2 entries; empty if it could not be built
    std::vector<uint32_t> confirm_groups; // per slot: DFA groups (bit g mod 32) whose patterns own the gram; only those are walked
    int confirm_log2 = 0;
    uint32_t confirm_mul = 0, confirm_mul2 = 0;
    // Extended confirmation.  A 4-byte gram of digits ("1234") occurs all over numeric text although the factor it stands for
    // ("12345\"") does not: where the factor is exact (single-valued bytes) around the gram, the verification kernel also
    // compares 6 or 8 bytes of text around the hit with a second exact table before it walks any automaton.
    // confirm_ext[slot of confirm_keys]: 0 = the gram is accepted as it is; else up to three variants of 5 bits each:
    // bits 0-2 = bytes in front of the gram (0..4), bit 3 = 8-byte key (else 6), bit 4 = variant present.
    std::vector<uint32_t> confirm_ext;
    std::vector<uint64_t> ext_keys;       // two-choice table, 2 << ext_log2 entries, 0 = empty; 6-byte keys carry 0xA5A5 on top
    int ext_log2 = 0;
    uint64_t ext_mul = 0, ext_mul2 = 0;
    // bloom bitmap (default in the streaming kernel: one lookup per gram): with p = gram * bloom_mul,
    // byte = p >> (32 - (log2_bits - 3)), bit = p & 7
    int log2_bits = 16;
    uint32_t bloom_mul = 0x9E3779B1u;
    std::vector<uint32_t> bitmap;
    uint32_t hash_mul = 0x9E3779B1u;
    std::vector<uint32_t> grams;      // the exact gram set (sorted)
    // Mixed sampling (stride == 4 only).  Factors of >= 7 bytes are found by table lookups at text offsets = 0 (mod 4).  The
    // few factors that are too short for that are ALSO compared, in registers, at offsets = 2 (mod 4): gram * mul + add == 0
    // tests the leading 4, 3 or 2 bytes of the gram (mul = 1, 2^8, 2^16) against a constant.  At most two compares.
    struct OddCompare { uint32_t mul, add; };
    std::vector<OddCompare> odd;
    size_t num_grams = 0;
    int min_factor_len = 0;
    // A match whose window hit sits at text position q starts at or after q - lookback (0xffffffff: unbounded, verify
    // from the line start).
    uint32_t lookback = 0xffffffffu;
    double expected_hits_per_mib = -1;   // from the sample histogram, -1 without a sample
    std::string note;           // why it is disabled, or a one-line summary
    // Literal index (fixed-string sets): the grams of the window chosen in each literal, each with the literal and the
    // offset of the gram in it.  Entries of confirm slot h are lit_entries[lit_begin[h] .. lit_begin[h + 1]), each
    // (class << 31 | offset) << 32 | literal, sorted by that key and then by the literal's rank: one (class, offset) run
    // is in byte order and is searched, not walked.
    std::vector<uint32_t> lit_begin;
    std::vector<uint64_t> lit_entries;
};

// Required-factor analysis of one pattern.  Returns false if no usable factor exists.
bool extract_factor(const Node& ast, std::vector<ClassString>& alternatives);

FactorSet analyse_factors(const std::vector<const Node*>& asts);

// Build the gram tables.  `sample` may be null (static choice: fewest grams per window).
void build_prefilter(const FactorSet& fs, const GramHistogram* sample, Prefilter& out);

inline uint32_t prefilter_hash(uint32_t gram, uint32_t mul, int log2_size) { return (gram * mul) >> (32 - log2_size); }

}  // namespace gpugrep
