// Required-factor analysis and gram-bitmap construction.  See prefilter.hpp.
#include "prefilter.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <set>

namespace gpugrep {
namespace {

constexpr size_t kMaxSet = 64;     // alternatives tracked per node
constexpr size_t kMaxLen = 24;     // positions tracked per class-string
constexpr double kMaxGramsPerWindow = 4096.0;
constexpr size_t kMaxGramsTotal = 131072;

using Alts = std::vector<ClassString>;

constexpr size_t kInf = SIZE_MAX / 4;
size_t sat_add(size_t a, size_t b) { return (a >= kInf || b >= kInf) ? kInf : a + b; }

// A required factor together with the largest distance (bytes) from the start of the enclosing match to the start
// of the factor occurrence that the match is guaranteed to contain (kInf: unbounded).
struct Cand {
    std::vector<ClassString> alts;
    size_t before = 0;
};

struct Lits {
    bool exact_ok = false;
    std::vector<ClassString> exact;    // the node matches exactly one of these (valid iff exact_ok)
    std::vector<ClassString> prefix;   // every match starts with one of these ({""} = nothing known)
    std::vector<ClassString> suffix;   // every match ends with one of these
    Cand best;                         // required factor (empty = none found)
};

using Alts = std::vector<ClassString>;
const Alts kEpsilon = {ClassString{}};

size_t max_len(const Alts& a) { size_t m = 0; for (auto& s : a) m = std::max(m, s.size()); return m; }
size_t min_len(const Alts& a) { size_t m = a.empty() ? 0 : SIZE_MAX; for (auto& s : a) m = std::min(m, s.size()); return m; }

void dedupe(Alts& a) {
    std::sort(a.begin(), a.end());
    a.erase(std::unique(a.begin(), a.end()), a.end());
}

bool fits(const Alts& a, const Alts& b) { return a.size() * b.size() <= kMaxSet && max_len(a) + max_len(b) <= kMaxLen; }

Alts cross(const Alts& a, const Alts& b) {
    Alts r;
    for (auto& x : a) for (auto& y : b) { ClassString s = x; s.insert(s.end(), y.begin(), y.end()); r.push_back(std::move(s)); }
    dedupe(r);
    return r;
}
// product that may be truncated: a prefix keeps its head
Alts cross_head(const Alts& a, const Alts& b) {
    if (a.size() * b.size() > kMaxSet) return a;
    Alts r = cross(a, b);
    for (auto& s : r) if (s.size() > kMaxLen) s.resize(kMaxLen);
    dedupe(r);
    return r;
}

// Probability that a random 4-gram falls in the most selective window of `s` (uniform byte model).
double window_prob(const ClassString& s, size_t w) {
    if (s.empty()) return 1.0;
    w = std::min(w, s.size());
    double best = 1.0;
    for (size_t t = 0; t + w <= s.size(); t++) {
        double p = 1.0;
        for (size_t i = 0; i < w; i++) p *= s[t + i].count() / 256.0;
        best = std::min(best, p);
    }
    return best;
}

// Lower is better; infinity = unusable.
double cost(const Alts& a) {
    if (a.empty()) return INFINITY;
    size_t ml = min_len(a);
    if (ml < 4) return INFINITY;   // the filter looks up 4-byte grams
    double tier = ml >= 7 ? 1.0 : (ml >= 5 ? 2.0 : 4.0);   // stride 4 / 2 / 1 in the streaming kernel
    double p = 0;
    for (auto& s : a) p += window_prob(s, 4);
    return p * tier;
}
double cost(const Cand& c) { return cost(c.alts) * (c.before >= kInf ? 1.5 : 1.0); }   // bounded look-back verifies cheaper

void consider(Cand& best, const Cand& cand) {
    if (cost(cand) < cost(best)) best = cand;
}

size_t node_maxlen(const Node& n) {
    switch (n.kind) {
        case NodeKind::Empty: case NodeKind::Assert: return 0;
        case NodeKind::Set: return 1;
        case NodeKind::Concat: { size_t t = 0; for (auto& k : n.kids) t = sat_add(t, node_maxlen(*k)); return t; }
        case NodeKind::Alt: { size_t t = 0; for (auto& k : n.kids) t = std::max(t, node_maxlen(*k)); return std::min(t, kInf); }
        case NodeKind::Repeat: {
            size_t c = node_maxlen(*n.kids[0]);
            if (c == 0) return 0;
            if (n.max < 0 || c >= kInf) return kInf;
            return std::min(kInf, c * (size_t)n.max);
        }
    }
    return kInf;
}

Lits analyse(const Node& n) {
    Lits r;
    switch (n.kind) {
        case NodeKind::Empty:
        case NodeKind::Assert:
            r.exact_ok = true; r.exact = kEpsilon; r.prefix = kEpsilon; r.suffix = kEpsilon;
            return r;
        case NodeKind::Set: {
            r.exact_ok = true;
            r.exact = {ClassString{n.set}};
            r.prefix = r.suffix = r.exact;
            return r;
        }
        case NodeKind::Concat: {
            Alts run = kEpsilon;
            size_t run_before = 0;   // bytes of this concatenation that can precede the start of `run`
            size_t acc = 0;          // bytes that can precede the current kid
            bool whole = true;       // everything so far is inside `run`
            r.prefix = kEpsilon;
            for (auto& kid : n.kids) {
                Lits k = analyse(*kid);
                size_t km = node_maxlen(*kid);
                if (k.exact_ok && fits(run, k.exact)) { run = cross(run, k.exact); acc = sat_add(acc, km); continue; }
                Alts closed = cross_head(run, k.exact_ok ? k.exact : k.prefix);
                consider(r.best, Cand{closed, run_before});
                if (!k.best.alts.empty()) consider(r.best, Cand{k.best.alts, sat_add(acc, k.best.before)});
                if (k.exact_ok) consider(r.best, Cand{k.exact, acc});
                if (whole) r.prefix = closed;
                whole = false;
                run = k.exact_ok ? k.exact : k.suffix;
                for (auto& s : run) if (s.size() > kMaxLen) s.erase(s.begin(), s.end() - kMaxLen);
                dedupe(run);
                run_before = km >= kInf ? kInf : sat_add(acc, km - std::min(km, min_len(run)));
                acc = sat_add(acc, km);
            }
            if (whole) {
                r.exact_ok = true; r.exact = run; r.prefix = run; r.suffix = run;
            } else {
                consider(r.best, Cand{run, run_before});
                r.suffix = run;
            }
            return r;
        }
        case NodeKind::Alt: {
            r.exact_ok = true;
            bool all_factor = true;
            Alts pre, suf, fac;
            size_t before = 0;
            for (auto& kid : n.kids) {
                Lits k = analyse(*kid);
                if (k.exact_ok && r.exact_ok && r.exact.size() + k.exact.size() <= kMaxSet) r.exact.insert(r.exact.end(), k.exact.begin(), k.exact.end());
                else r.exact_ok = false;
                Cand as_exact{k.exact, 0};
                const Cand& f = (k.exact_ok && cost(as_exact) <= cost(k.best)) ? as_exact : k.best;
                if (std::isinf(cost(f))) all_factor = false;
                else { fac.insert(fac.end(), f.alts.begin(), f.alts.end()); before = std::max(before, f.before); }
                pre.insert(pre.end(), k.prefix.begin(), k.prefix.end());
                suf.insert(suf.end(), k.suffix.begin(), k.suffix.end());
            }
            dedupe(pre); dedupe(suf); dedupe(fac);
            r.prefix = pre.size() <= kMaxSet ? pre : kEpsilon;
            r.suffix = suf.size() <= kMaxSet ? suf : kEpsilon;
            if (r.exact_ok) dedupe(r.exact); else r.exact.clear();
            if (all_factor && fac.size() <= 4 * kMaxSet) r.best = Cand{fac, before};
            return r;
        }
        case NodeKind::Repeat: {
            Lits k = analyse(*n.kids[0]);
            if (n.min == 0) {
                r.prefix = r.suffix = kEpsilon;
                if (n.max == 1 && k.exact_ok && k.exact.size() + 1 <= kMaxSet) {
                    r.exact_ok = true; r.exact = k.exact; r.exact.push_back(ClassString{}); dedupe(r.exact);
                }
                return r;
            }
            // min >= 1: the child occurs at least `min` times in a row; the first iteration starts the match
            if (k.exact_ok) {
                Alts pow = k.exact;
                int reps = 1;
                while (reps < n.min && fits(pow, k.exact)) { pow = cross(pow, k.exact); reps++; }
                if (reps == n.min && n.max == n.min) { r.exact_ok = true; r.exact = pow; r.prefix = r.suffix = pow; return r; }
                r.prefix = r.suffix = pow;
                r.best = Cand{pow, 0};
                if (std::isinf(cost(r.best))) r.best = Cand{};
                return r;
            }
            r.prefix = k.prefix; r.suffix = k.suffix; r.best = k.best;
            return r;
        }
    }
    return r;
}

struct Window { const ClassString* s; size_t start; size_t pattern; };

double grams_in_window(const ClassString& s, size_t t, int stride, bool fold) {
    double total = 0;
    for (int j = 0; j < stride; j++) {
        double p = 1;
        for (int i = 0; i < 4; i++) {
            const ByteSet& b = s[t + j + i];
            int c = b.count();
            if (fold && c > 1) { ByteSet f; for (unsigned v = 0; v < 256; v++) if (b.test(v)) f.set(v | 0x20); c = f.count(); }
            p *= c;
        }
        total += p;
    }
    return total;
}

}  // namespace

static bool extract_cand(const Node& ast, Cand& out) {
    Lits l = analyse(ast);
    Cand best = l.best;
    if (l.exact_ok) consider(best, Cand{l.exact, 0});
    consider(best, Cand{l.prefix, 0});
    size_t total = node_maxlen(ast);
    consider(best, Cand{l.suffix, total >= kInf ? kInf : total - std::min(total, min_len(l.suffix))});
    if (std::isinf(cost(best))) return false;
    out = best;
    return true;
}

bool extract_factor(const Node& ast, std::vector<ClassString>& alternatives) {
    Cand c;
    if (!extract_cand(ast, c)) return false;
    alternatives = c.alts;
    return true;
}

FactorSet analyse_factors(const std::vector<const Node*>& asts) {
    FactorSet fs;
    fs.factors.resize(asts.size());
    size_t ml = SIZE_MAX;
    fs.before.resize(asts.size());
    for (size_t i = 0; i < asts.size(); i++) {
        Cand c;
        bool ok = extract_cand(*asts[i], c);
        fs.factors[i] = c.alts;
        fs.before[i] = c.before >= kInf ? SIZE_MAX : c.before;
        if (!ok) {
            fs.note = "pattern " + std::to_string(i) + " has no required factor of >= 4 bytes";
            fs.factors.clear();
            return fs;
        }
        ml = std::min(ml, min_len(fs.factors[i]));
    }
    fs.usable = true;
    fs.min_len = ml;
    return fs;
}

// ---- sample histogram ----------------------------------------------------------------------------------------
void GramHistogram::Table::init(size_t capacity_pow2) {
    keys.assign(capacity_pow2, 0);
    counts.assign(capacity_pow2, 0);
    mask = (uint32_t)capacity_pow2 - 1;
}
void GramHistogram::Table::add(uint32_t key) {
    uint32_t h = (key * 0x9E3779B1u) >> 7;
    for (;;) {
        h &= mask;
        if (counts[h] == 0) { keys[h] = key; counts[h] = 1; return; }
        if (keys[h] == key) { counts[h]++; return; }
        h++;
    }
}
uint32_t GramHistogram::Table::get(uint32_t key) const {
    if (keys.empty()) return 0;
    uint32_t h = (key * 0x9E3779B1u) >> 7;
    for (;;) {
        h &= mask;
        if (counts[h] == 0) return 0;
        if (keys[h] == key) return counts[h];
        h++;
    }
}
void GramHistogram::add_sample(const uint8_t* text, size_t n) {
    if (n < 4) return;
    size_t cap = 1;
    while (cap < 2 * n) cap <<= 1;   // load factor <= 0.5
    raw_.init(cap);
    folded_.init(cap);
    uint64_t fp = 1469598103934665603ull ^ n;
    for (size_t i = 0; i + 4 <= n; i++) {
        uint32_t g;
        std::memcpy(&g, text + i, 4);
        raw_.add(g);
        folded_.add(g | 0x20202020u);
        if ((i & 63) == 0) fp = (fp ^ g) * 1099511628211ull;
    }
    positions_ = n - 3;
    fingerprint_ = fp;
}
uint32_t GramHistogram::count(uint32_t gram, bool folded) const { return folded ? folded_.get(gram) : raw_.get(gram); }

namespace {

ByteSet effective(const ByteSet& b, bool fold) {
    if (!fold) return b;
    ByteSet f;
    for (unsigned v = 0; v < 256; v++) if (b.test(v)) f.set(v | 0x20);
    return f;
}

// The one gram of s[at, at+4) when every position holds one byte (literals, most regex factors); false otherwise.
bool single_gram(const ClassString& s, size_t at, bool fold, uint32_t& gram) {
    gram = 0;
    for (int i = 0; i < 4; i++) {
        const ByteSet& b = s[at + i];
        if (b.count() != 1) return false;
        unsigned v = 0;
        while (!b.w[v >> 6]) v += 64;
        v += (unsigned)__builtin_ctzll(b.w[v >> 6]);
        if (fold) v |= 0x20;
        gram |= v << (8 * i);
    }
    return true;
}

void expand_gram(const ClassString& s, size_t at, bool fold, std::vector<uint32_t>& out) {
    uint32_t one = 0;
    if (single_gram(s, at, fold, one)) { out.push_back(one); return; }
    std::vector<uint32_t> cur = {0};
    for (int i = 0; i < 4; i++) {
        ByteSet eff = effective(s[at + i], fold);
        std::vector<uint32_t> next;
        next.reserve(cur.size() * eff.count());
        for (uint32_t g : cur) for (unsigned v = 0; v < 256; v++) if (eff.test(v)) next.push_back(g | (v << (8 * i)));
        cur.swap(next);
    }
    out.insert(out.end(), cur.begin(), cur.end());
}

// Expected filter hits in the sample if window [t, t+3+stride) of s is used: each gram of alignment j is looked up
// at 1/stride of the text positions.
double window_hits(const ClassString& s, size_t t, int stride, bool fold, const GramHistogram& h) {
    std::vector<uint32_t> grams;
    double hits = 0;
    for (int j = 0; j < stride; j++) {
        uint32_t one = 0;
        if (single_gram(s, t + j, fold, one)) { hits += h.count(one, fold); continue; }
        grams.clear();
        expand_gram(s, t + j, fold, grams);
        for (uint32_t g : grams) hits += h.count(g, fold);
    }
    return hits / stride;
}

// Two-choice hashing: every key has one candidate slot in each half; insertion evicts (cuckoo) until everything is
// placed.  Tries table sizes 2 x 2^lb for lb in [first_lb, max_lb] and a few multiplier pairs.
bool build_two_choice(const std::vector<uint32_t>& grams, int first_lb, int max_lb, std::vector<uint32_t>& out_keys, int& out_lb,
                      uint32_t& out_m1, uint32_t& out_m2) {
    static const uint32_t muls[] = {0x9E3779B1u, 0x85EBCA6Bu, 0xC2B2AE35u, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Cu, 0xFD7046C5u, 0xB55A4F09u,
                                    0x7FEB352Du, 0x846CA68Bu, 0x9E3779B9u, 0xCC9E2D51u, 0x1B873593u, 0xE6546B64u, 0x2545F491u, 0x5851F42Du};
    const int nmul = (int)(sizeof(muls) / sizeof(muls[0]));
    for (int lb = first_lb; lb <= max_lb; lb++) {
        const size_t slots = (size_t)1 << lb;
        for (int a = 0; a + 1 < nmul; a += 2) {
            const uint32_t m1 = muls[a], m2 = muls[a + 1];
            std::vector<uint32_t> keys(2 * slots, 0);
            bool ok = true;
            for (uint32_t g : grams) {
                uint32_t cur = g;
                int side = 0;
                int kicks = 0;
                while (true) {
                    size_t at = side == 0 ? prefilter_hash(cur, m1, lb) : slots + prefilter_hash(cur, m2, lb);
                    if (keys[at] == 0) { keys[at] = cur; break; }
                    if (kicks == 0 && side == 0) {   // try the other side before evicting
                        size_t alt = slots + prefilter_hash(cur, m2, lb);
                        if (keys[alt] == 0) { keys[alt] = cur; break; }
                    }
                    std::swap(cur, keys[at]);
                    side ^= 1;
                    if (++kicks > 200) { ok = false; break; }
                }
                if (!ok) break;
            }
            if (ok) {
                out_keys.swap(keys);
                out_lb = lb;
                out_m1 = m1;
                out_m2 = m2;
                return true;
            }
        }
    }
    return false;
}

void build_exact_tables(const std::vector<uint32_t>& grams, Prefilter& out) {
    int lb = 4;
    while (lb < 24 && ((size_t)2 << lb) * 2 < grams.size() * 5) lb++;   // total slots >= 2.5 x keys
    // Shared-memory variant (GPUGREP_FILTER=exact): small tables matter, the engine replicates the table across the banks so
    // that lookups are conflict-free, and the replication factor is what fits.  At most 2 x 16384 slots = 128 KiB unreplicated.
    out.exact = lb <= 14 && build_two_choice(grams, lb, 14, out.keys, out.log2_slots, out.hash_mul, out.hash_mul2);
    // global-memory variant for the verification kernel
    if (out.exact) {
        out.confirm_keys = out.keys;
        out.confirm_log2 = out.log2_slots;
        out.confirm_mul = out.hash_mul;
        out.confirm_mul2 = out.hash_mul2;
    } else if (!build_two_choice(grams, lb, 24, out.confirm_keys, out.confirm_log2, out.confirm_mul, out.confirm_mul2)) {
        out.confirm_keys.clear();
    }
}

// Fills the gram tables of `out` (exact two-choice table and bloom byte table) from the final gram list.
// grams of the chosen windows, each with the DFA groups of the pattern it came from
// Exact bytes around a gram instance (see Prefilter::confirm_ext): `before` bytes in front of the gram, 6 or 8 in all.
struct GramExt {
    uint8_t before = 0, len = 0;   // len == 0: no extension (a class position is too close, or the factor is too short)
    uint64_t key = 0;
};
constexpr uint64_t kExt6Tag = 0xA5A5000000000000ull;

// The extended keys are compared case-folded on EVERY byte (text | 0x20, whatever the gram table does): a caseless letter
// {x, X} is then as good as an exact byte, and so is any other position whose bytes agree once bit 5 is set.  The filter
// stays a superset filter: folding can only make more text pass.
GramExt extension_of(const ClassString& s, size_t at) {
    auto single = [&](size_t i, unsigned& value) {
        int seen = -1;
        for (unsigned v = 0; v < 256; v++) {
            if (!s[i].test(v)) continue;
            const int f = (int)(v | 0x20u);
            if (seen >= 0 && seen != f) return false;
            seen = f;
        }
        if (seen < 0) return false;
        value = (unsigned)seen;
        return true;
    };
    for (size_t len : {(size_t)8, (size_t)6}) {
        for (size_t before = 0; before + 4 <= len; before++) {   // as much as possible behind the gram first
            if (before > at || at - before + len > s.size()) continue;
            uint64_t key = 0;
            bool ok = true;
            for (size_t i = 0; i < len && ok; i++) {
                unsigned v = 0;
                ok = single(at - before + i, v);
                key |= (uint64_t)v << (8 * i);
            }
            if (!ok) continue;
            GramExt e;
            e.before = (uint8_t)before;
            e.len = (uint8_t)len;
            e.key = len == 8 ? key : (key | kExt6Tag);
            return e;
        }
    }
    return GramExt();
}

struct GramList {
    struct Item { uint32_t gram, mask; GramExt ext; };
    std::vector<Item> items;   // (gram, group mask, exact bytes around this instance)
    void add(const ClassString& s, size_t at, bool fold, uint32_t mask) {
        scratch.clear();
        expand_gram(s, at, fold, scratch);
        const GramExt ext = extension_of(s, at);   // the same for every case variant of the gram
        for (uint32_t g : scratch) items.push_back(Item{g, mask, ext});
    }
    size_t size() const { return items.size(); }
private:
    std::vector<uint32_t> scratch;
};

// two-choice table of 64-bit keys (same scheme as build_two_choice)
bool build_two_choice64(const std::vector<uint64_t>& keys_in, std::vector<uint64_t>& out_keys, int& out_lb, uint64_t& out_m1, uint64_t& out_m2) {
    static const uint64_t muls[] = {0x9E3779B97F4A7C15ull, 0xC2B2AE3D27D4EB4Full, 0xD6E8FEB86659FD93ull, 0xFF51AFD7ED558CCDull,
                                    0xC4CEB9FE1A85EC53ull, 0x94D049BB133111EBull, 0xBF58476D1CE4E5B9ull, 0x2545F4914F6CDD1Dull};
    int lb = 4;
    while (lb < 26 && ((size_t)2 << lb) * 2 < keys_in.size() * 5) lb++;
    for (; lb <= 26; lb++) {
        const size_t slots = (size_t)1 << lb;
        for (int a = 0; a + 1 < 8; a += 2) {
            const uint64_t m1 = muls[a], m2 = muls[a + 1];
            std::vector<uint64_t> keys(2 * slots, 0);
            bool ok = true;
            for (uint64_t k : keys_in) {
                uint64_t cur = k;
                int side = 0, kicks = 0;
                while (true) {
                    size_t at = side == 0 ? (size_t)((cur * m1) >> (64 - lb)) : slots + (size_t)((cur * m2) >> (64 - lb));
                    if (keys[at] == 0) { keys[at] = cur; break; }
                    if (kicks == 0 && side == 0) {
                        size_t alt = slots + (size_t)((cur * m2) >> (64 - lb));
                        if (keys[alt] == 0) { keys[alt] = cur; break; }
                    }
                    std::swap(cur, keys[at]);
                    side ^= 1;
                    if (++kicks > 200) { ok = false; break; }
                }
                if (!ok) break;
            }
            if (ok) { out_keys.swap(keys); out_lb = lb; out_m1 = m1; out_m2 = m2; return true; }
        }
    }
    return false;
}

uint32_t mask_of(const FactorSet& fs, size_t pattern) { return pattern < fs.group_mask.size() ? fs.group_mask[pattern] : 0xffffffffu; }

void finish_tables(GramList& list, bool fold, const GramHistogram* sample, Prefilter& out) {
    // unique grams, group masks merged
    std::sort(list.items.begin(), list.items.end(), [](const GramList::Item& a, const GramList::Item& b) { return a.gram < b.gram; });
    std::vector<uint32_t> all, masks, exts;   // exts: confirm_ext encoding per unique gram (0 = accepted as it is)
    std::vector<uint64_t> ext_keys;
    for (size_t i = 0; i < list.items.size();) {
        size_t j = i;
        uint32_t mask = 0;
        bool confirmable = true;
        std::vector<std::pair<uint8_t, uint8_t>> variants;
        for (; j < list.items.size() && list.items[j].gram == list.items[i].gram; j++) {
            mask |= list.items[j].mask;
            const GramExt& e = list.items[j].ext;
            if (e.len == 0) { confirmable = false; continue; }
            auto v = std::make_pair(e.before, e.len);
            if (std::find(variants.begin(), variants.end(), v) == variants.end()) variants.push_back(v);
        }
        if (list.items[i].gram != 0u) {   // the empty-slot marker cannot be stored exactly; it can only be "\0\0\0\0", which never occurs in a block
            uint32_t enc = 0;
            if (confirmable && !variants.empty() && variants.size() <= 3) {
                for (size_t v = 0; v < variants.size(); v++)
                    enc |= (16u | (variants[v].second == 8 ? 8u : 0u) | variants[v].first) << (5 * v);
                for (size_t k = i; k < j; k++) ext_keys.push_back(list.items[k].ext.key);
            }
            all.push_back(list.items[i].gram);
            masks.push_back(mask);
            exts.push_back(enc);
        }
        i = j;
    }
    out.enabled = true;
    out.fold_case = fold;
    out.num_grams = all.size();
    out.grams = all;
    build_exact_tables(all, out);
    if (!out.confirm_keys.empty()) {
        const size_t half = (size_t)1 << out.confirm_log2;
        out.confirm_groups.assign(out.confirm_keys.size(), 0u);
        for (size_t k = 0; k < all.size(); k++) {
            const size_t h1 = prefilter_hash(all[k], out.confirm_mul, out.confirm_log2), h2 = half + prefilter_hash(all[k], out.confirm_mul2, out.confirm_log2);
            out.confirm_groups[out.confirm_keys[h1] == all[k] ? h1 : h2] |= masks[k];
        }
        // extended confirmation (Prefilter::confirm_ext): only when the second table can be built
        std::sort(ext_keys.begin(), ext_keys.end());
        ext_keys.erase(std::unique(ext_keys.begin(), ext_keys.end()), ext_keys.end());
        out.confirm_ext.clear();
        out.ext_keys.clear();
        if (!ext_keys.empty() && std::getenv("GPUGREP_NO_EXT_CONFIRM") == nullptr &&
            build_two_choice64(ext_keys, out.ext_keys, out.ext_log2, out.ext_mul, out.ext_mul2)) {
            out.confirm_ext.assign(out.confirm_keys.size(), 0u);
            for (size_t k = 0; k < all.size(); k++) {
                const size_t h1 = prefilter_hash(all[k], out.confirm_mul, out.confirm_log2), h2 = half + prefilter_hash(all[k], out.confirm_mul2, out.confirm_log2);
                out.confirm_ext[out.confirm_keys[h1] == all[k] ? h1 : h2] = exts[k];
            }
        }
    }
    // bloom bitmap, one probe per gram: byte = product >> (32 - log2_bytes), bit = product & 7.  Sized so that
    // a false hit is rare next to real gram occurrences (<= 2^20 bits = 128 KiB of shared memory).
    size_t need = all.size() * 2048;
    int lb = 17;
    while (lb < 20 && (1ull << lb) < need) lb++;
    if (sample) lb = 20;   // streaming scans: always the largest table (128 KiB), false hits cost DFA walks
    out.log2_bits = lb;
    // One unlucky collision with a FREQUENT text gram ("INFO", " hos") would flag a large share of all chunks:
    // pick, among a few multipliers, the one whose table is hit least by the non-member grams of the sample.
    static const uint32_t muls[] = {0x9E3779B1u, 0x85EBCA6Bu, 0xC2B2AE35u, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};
    double best_false = INFINITY;
    std::vector<uint32_t> best_map;
    for (uint32_t mul : muls) {
        std::vector<uint32_t> map((1u << lb) / 32, 0);
        uint8_t* bytes = reinterpret_cast<uint8_t*>(map.data());
        for (uint32_t g : all) {
            uint32_t p = g * mul;
            bytes[p >> (32 - (lb - 3))] |= (uint8_t)(1u << (p & 7));
        }
        double false_hits = 0;
        if (sample) {
            const auto& keys = sample->keys(fold);
            const auto& counts = sample->counts(fold);
            for (size_t k = 0; k < keys.size(); k++) {
                if (!counts[k]) continue;
                uint32_t p = keys[k] * mul;
                if ((bytes[p >> (32 - (lb - 3))] >> (p & 7)) & 1)
                    if (!std::binary_search(all.begin(), all.end(), keys[k])) false_hits += counts[k];
            }
        }
        if (false_hits < best_false) { best_false = false_hits; best_map.swap(map); out.bloom_mul = mul; }
        if (!sample || false_hits == 0) break;
    }
    out.bitmap.swap(best_map);
}

std::string describe(const Prefilter& out, bool tuned) {
    return "stride " + std::to_string(out.stride) + (out.odd.empty() ? "" : " + " + std::to_string(out.odd.size()) + " compares at 2 mod 4") + (out.fold_case ? ", folded" : "") + ", " + std::to_string(out.num_grams) + " grams, bloom bitmap of " + std::to_string(1u << out.log2_bits) +
           " bits, " + std::to_string((int)out.expected_hits_per_mib) + " expected hits/MiB" +
           (out.confirm_ext.empty() ? std::string() : ", " + std::to_string(std::count_if(out.confirm_ext.begin(), out.confirm_ext.end(), [](uint32_t e) { return e != 0; })) + " grams with extended confirmation") + (out.exact ? ", exact two-choice table of 2 x " + std::to_string(1u << out.log2_slots) + " slots" : "") + (tuned ? ", sample-tuned" : "");
}

// One register compare of the mixed scheme: the first `known` bytes of a 4-gram (little endian: the low bytes).
struct OddKey {
    uint32_t value = 0;
    int known = 0;
    bool operator==(const OddKey& o) const { return value == o.value && known == o.known; }
    uint32_t mask() const { return known >= 4 ? 0xffffffffu : (1u << (8 * known)) - 1u; }
};

// the bytes of s[at, at+4) that are the same in every expansion (leading ones only)
OddKey odd_key_of(const ClassString& s, size_t at, bool fold) {
    OddKey k;
    for (int i = 0; i < 4; i++) {
        ByteSet eff = effective(s[at + i], fold);
        if (eff.count() != 1) break;
        for (unsigned v = 0; v < 256; v++) if (eff.test(v)) k.value |= v << (8 * i);
        k.known++;
    }
    return k;
}

double odd_key_hits(const OddKey& k, bool fold, const GramHistogram& h) {
    const auto& keys = h.keys(fold);
    const auto& counts = h.counts(fold);
    double hits = 0;
    for (size_t i = 0; i < keys.size(); i++)
        if (counts[i] && (keys[i] & k.mask()) == k.value) hits += counts[i];
    return hits;
}

// Mixed sampling (see Prefilter::odd).  Every alternative with a usable 7-byte window is sampled at stride 4; the others
// get a 5-byte window whose two grams go into the table (for offsets = 0 mod 4) and into the compare list (for offsets
// = 2 mod 4).  Fails if that needs more than two compares or a compare of fewer than two known bytes.
bool build_mixed(const FactorSet& fs, const GramHistogram* sample, bool fold, Prefilter& out) {
    out = Prefilter();
    out.min_factor_len = (int)fs.min_len;
    GramList all;
    std::vector<OddKey> odd;
    size_t lookback = 0;
    double hits = 0;
    struct Short { const ClassString* s; size_t pattern; };
    std::vector<Short> shorts;
    for (size_t pi = 0; pi < fs.factors.size(); pi++) {
        for (auto& s : fs.factors[pi]) {
            double best = INFINITY; size_t bt = 0;
            for (size_t t = 0; t + 7 <= s.size(); t++) {
                double g = grams_in_window(s, t, 4, fold);
                if (g > kMaxGramsPerWindow * 4) continue;
                double score = sample ? window_hits(s, t, 4, fold, *sample) * 1000.0 + g : g;
                if (score < best) { best = score; bt = t; }
            }
            if (std::isinf(best)) { shorts.push_back(Short{&s, pi}); continue; }
            if (sample) hits += window_hits(s, bt, 4, fold, *sample);
            for (int j = 0; j < 4; j++) all.add(s, bt + j, fold, mask_of(fs, pi));
            size_t lb = fs.before[pi] == SIZE_MAX ? SIZE_MAX : fs.before[pi] + bt + 3;
            lookback = std::max(lookback, lb);
        }
    }
    if (shorts.empty()) return false;   // plain stride 4 does it
    for (auto& sh : shorts) {
        const ClassString& s = *sh.s;
        double best = INFINITY; size_t bt = 0;
        for (size_t t = 0; t + 5 <= s.size(); t++) {
            double g = grams_in_window(s, t, 2, fold);
            if (g > kMaxGramsPerWindow * 2) continue;
            OddKey k0 = odd_key_of(s, t, fold), k1 = odd_key_of(s, t + 1, fold);
            if (k0.known < 2 || k1.known < 2) continue;
            if (!sample && (k0.known < 3 || k1.known < 3)) continue;   // without a sample only selective compares
            // fewest NEW compares first, then expected hits (table part + compare part), then table growth
            int fresh = (std::find(odd.begin(), odd.end(), k0) == odd.end()) + (std::find(odd.begin(), odd.end(), k1) == odd.end() && !(k1 == k0));
            double h = sample ? window_hits(s, t, 2, fold, *sample) / 2 + (odd_key_hits(k0, fold, *sample) + odd_key_hits(k1, fold, *sample)) / 4 : 0;
            double score = fresh * 1e12 + h * 1000.0 + g;
            if (score < best) { best = score; bt = t; }
        }
        if (std::isinf(best)) return false;
        for (int j = 0; j < 2; j++) {
            all.add(s, bt + j, fold, mask_of(fs, sh.pattern));
            OddKey k = odd_key_of(s, bt + j, fold);
            if (std::find(odd.begin(), odd.end(), k) == odd.end()) odd.push_back(k);
        }
        if (odd.size() > 2) return false;
        if (sample) hits += window_hits(s, bt, 2, fold, *sample) / 2;   // the table part: sampled at every fourth offset
        size_t lb = fs.before[sh.pattern] == SIZE_MAX ? SIZE_MAX : fs.before[sh.pattern] + bt + 1;
        lookback = std::max(lookback, lb);
    }
    if (all.size() > kMaxGramsTotal) return false;
    if (sample) for (auto& k : odd) hits += odd_key_hits(k, fold, *sample) / 4;
    for (auto& k : odd) {
        const int shift = 8 * (4 - k.known);
        out.odd.push_back(Prefilter::OddCompare{1u << shift, 0u - (k.value << shift)});
    }
    out.stride = 4;
    out.lookback = lookback > 4096 ? 0xffffffffu : (uint32_t)lookback;
    if (sample && sample->positions()) out.expected_hits_per_mib = hits * 1048576.0 / (double)sample->positions();
    finish_tables(all, fold, sample, out);
    out.note = describe(out, sample != nullptr);
    return true;
}

// Literal index of a fixed-string set (Prefilter::lit_begin): every gram of each literal's window, under the confirm slot
// of the gram.  Without an exact confirm table there is no index, and the set goes without a prefilter.
void build_literal_index(const FactorSet& fs, const std::vector<Window>& wins, int stride, bool fold, Prefilter& out) {
    if (out.confirm_keys.empty()) {
        out = Prefilter();
        out.note = "no exact gram table for the literal index";
        return;
    }
    const size_t half = (size_t)1 << out.confirm_log2;
    struct E { uint32_t slot, key, rank, lit; };
    std::vector<E> es;
    es.reserve(wins.size() * (size_t)stride);
    std::vector<uint32_t> grams;
    for (const Window& wn : wins) {
        const uint32_t cls = fs.literal_class[wn.pattern];
        for (int j = 0; j < stride; j++) {
            grams.clear();
            expand_gram(*wn.s, wn.start + j, fold, grams);
            for (uint32_t g : grams) {
                const size_t h1 = prefilter_hash(g, out.confirm_mul, out.confirm_log2), h2 = half + prefilter_hash(g, out.confirm_mul2, out.confirm_log2);
                const uint32_t slot = (uint32_t)(out.confirm_keys[h1] == g ? h1 : h2);
                es.push_back(E{slot, cls << 31 | (uint32_t)(wn.start + (size_t)j), fs.literal_rank[wn.pattern], (uint32_t)wn.pattern});
            }
        }
    }
    std::sort(es.begin(), es.end(), [](const E& a, const E& b) {
        return a.slot != b.slot ? a.slot < b.slot : (a.key != b.key ? a.key < b.key : a.rank < b.rank);
    });
    es.erase(std::unique(es.begin(), es.end(), [](const E& a, const E& b) { return a.slot == b.slot && a.key == b.key && a.lit == b.lit; }), es.end());
    out.lit_begin.assign(out.confirm_keys.size() + 1, 0);
    out.lit_entries.resize(es.size());
    for (size_t k = 0; k < es.size(); k++) {
        out.lit_begin[es[k].slot + 1]++;
        out.lit_entries[k] = (uint64_t)es[k].key << 32 | es[k].lit;
    }
    for (size_t h = 0; h < out.confirm_keys.size(); h++) out.lit_begin[h + 1] += out.lit_begin[h];
}

}  // namespace

static void build_uniform(const FactorSet& fs, const GramHistogram* sample, Prefilter& out) {
    out = Prefilter();
    if (!fs.usable) { out.note = fs.note; return; }
    out.min_factor_len = (int)fs.min_len;
    int first_stride = fs.min_len >= 7 ? 4 : (fs.min_len >= 5 ? 2 : 1);
    for (int stride = first_stride; stride >= 1; stride /= 2) {
        size_t w = 3 + (size_t)stride;
        for (int pass = 0; pass < 2; pass++) {
            bool fold = pass == 1;
            std::vector<Window> wins;
            double total = 0, hits = 0;
            bool ok = true;
            size_t lookback = 0;
            for (size_t pi = 0; pi < fs.factors.size(); pi++) {
                auto& alts = fs.factors[pi];
                for (auto& s : alts) {
                    double best = INFINITY, best_grams = 0; size_t bt = 0;
                    for (size_t t = 0; t + w <= s.size(); t++) {
                        double g = grams_in_window(s, t, stride, fold);
                        if (g > kMaxGramsPerWindow * stride) continue;
                        // score: expected hits in the sample first, table growth second
                        double score = sample ? window_hits(s, t, stride, fold, *sample) * 1000.0 + g : g;
                        if (score < best) { best = score; best_grams = g; bt = t; }
                    }
                    if (std::isinf(best)) { ok = false; break; }
                    total += best_grams;
                    if (sample) hits += (best - best_grams) / 1000.0;
                    wins.push_back(Window{&s, bt, pi});
                    size_t lb = fs.before[pi] == SIZE_MAX ? SIZE_MAX : fs.before[pi] + bt + (size_t)stride - 1;
                    lookback = std::max(lookback, lb);
                }
                if (!ok) break;
            }
            // (the gram tables of a fixed-string set are global-memory tables: only the shared-memory bloom has a fixed size)
            if (!ok || (total > (double)kMaxGramsTotal && !fs.literal())) continue;
            if (!fold) {
                // prefer exact-case grams unless folding shrinks the table a lot (caseless sets)
                double folded_total = 0;
                for (auto& wn : wins) folded_total += grams_in_window(*wn.s, wn.start, stride, true);
                if (total > 3.0 * folded_total && total > 2048) continue;
            }
            GramList all;
            for (auto& wn : wins)
                for (int j = 0; j < stride; j++) all.add(*wn.s, wn.start + j, fold, mask_of(fs, wn.pattern));
            out.stride = stride;
            out.lookback = lookback > 4096 ? 0xffffffffu : (uint32_t)lookback;
            if (sample && sample->positions()) out.expected_hits_per_mib = hits * 1048576.0 / (double)sample->positions();
            finish_tables(all, fold, sample, out);
            out.note = describe(out, sample != nullptr);
            if (fs.literal()) build_literal_index(fs, wins, stride, fold, out);
            return;
        }
    }
    out.note = "gram expansion too large";
}

void build_prefilter(const FactorSet& fs, const GramHistogram* sample, Prefilter& out) {
    build_uniform(fs, sample, out);
    // A set that is sampled at stride 2 only because of ONE short factor does better with stride 4 plus two register
    // compares (half the shared-memory lookups of the streaming kernel; measured 0.54 -> 0.45 ms per 2 GiB), unless that
    // flags more text or makes the verification walks longer.  (Four compares were measured too: the streaming kernel
    // gains 8 %, verification loses more through the longer look-back of the 7-byte windows.)
    // (not for fixed-string sets: their literal index holds the grams of whole windows, which the register compares are not)
    if (out.enabled && out.stride == 2 && !fs.literal() && std::getenv("GPUGREP_NO_MIXED_STRIDE") == nullptr) {
        Prefilter mixed;
        if (build_mixed(fs, sample, out.fold_case, mixed) && mixed.enabled && mixed.lookback <= out.lookback + 4 &&
            (!sample || mixed.expected_hits_per_mib <= 1.1 * out.expected_hits_per_mib + 16.0))
            out = std::move(mixed);
    }
}

}  // namespace gpugrep
