// Pattern-set compilation driver.  See database.hpp.
#include "database.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string_view>
#include <list>
#include <future>
#include <map>
#include <mutex>

namespace gpugrep {
namespace {

constexpr size_t kMaxNfaInsts = 400000;    // per group
constexpr size_t kMaxPatternInsts = 70000;  // per pattern (bounded repeats are unrolled)

size_t env_size(const char* name, size_t dflt) {
    const char* v = std::getenv(name);
    if (!v || !*v) return dflt;
    return (size_t)std::strtoull(v, nullptr, 10);
}

// Build DFA groups for patterns[lo, hi) by recursive bisection until every group fits the state budget.
bool build_groups(const std::vector<NodePtr>& asts, const std::vector<int>& idx, size_t lo, size_t hi, bool simple,
                  size_t max_states, std::vector<DfaGroup>& out, std::vector<NfaPattern>& nfas, std::string& error, int depth = 0) {
    Nfa nfa;
    bool ok = true;
    for (size_t k = lo; k < hi && ok; k++) ok = nfa_add_pattern(nfa, *asts[idx[k]], (int)(k - lo), kMaxNfaInsts);
    const size_t mid = lo + (hi - lo) / 2;
    // A set this large may not fit one DFA: its halves are compiled on two more threads WHILE the union is attempted (three
    // levels deep, so at most 14 helper threads); whichever result is needed is there when the attempt ends.
    const bool speculate = depth < 3 && hi - lo >= 64 && (!ok || nfa.prog.size() * 4 > max_states);
    std::vector<DfaGroup> left_groups, right_groups;
    std::vector<NfaPattern> left_nfas, right_nfas;
    std::string left_error, right_error;
    std::future<bool> left, right;
    if (speculate) {
        left = std::async(std::launch::async, [&] { return build_groups(asts, idx, lo, mid, simple, max_states, left_groups, left_nfas, left_error, depth + 1); });
        right = std::async(std::launch::async, [&] { return build_groups(asts, idx, mid, hi, simple, max_states, right_groups, right_nfas, right_error, depth + 1); });
    }
    DfaGroup g;
    // A union DFA has about one state per distinct prefix of its patterns: with several times more NFA instructions than the
    // state budget the attempt cannot succeed, and running it to the budget costs seconds for a 10,000-pattern set.
    if (ok && hi - lo > 1 && nfa.prog.size() > 3 * max_states) ok = false;
    if (ok) {
        DfaBuildOptions opt;
        opt.simple = simple;
        opt.max_states = max_states;
        ok = build_dfa(nfa, opt, g.dfa);
    }
    bool left_ok = true, right_ok = true;
    if (speculate) {   // the helpers use this frame's vectors: always wait for them
        left_ok = left.get();
        right_ok = right.get();
    }
    if (ok) {
        for (size_t k = lo; k < hi; k++) g.members.push_back(idx[k]);
        out.push_back(std::move(g));
        return true;
    }
    if (hi - lo == 1) {
        // this pattern alone explodes as a DFA: bit-parallel NFA fallback
        Nfa single;
        NfaPattern np;
        np.pattern = idx[lo];
        if (!nfa_add_pattern(single, *asts[idx[lo]], 0, kMaxNfaInsts) || !build_nfa_tables(single, np.tables)) {
            error = "pattern " + std::to_string(idx[lo]) + " exceeds both the DFA state budget (" + std::to_string(max_states) +
                    " states) and the NFA position limit (4096)";
            return false;
        }
        nfas.push_back(std::move(np));
        return true;
    }
    if (!speculate)
        return build_groups(asts, idx, lo, mid, simple, max_states, out, nfas, error, depth + 1) &&
               build_groups(asts, idx, mid, hi, simple, max_states, out, nfas, error, depth + 1);
    if (!left_ok || !right_ok) {
        error = !left_ok ? left_error : right_error;
        return false;
    }
    for (auto& grp : left_groups) out.push_back(std::move(grp));    // pattern order is kept: left half first
    for (auto& grp : right_groups) out.push_back(std::move(grp));
    for (auto& np : left_nfas) nfas.push_back(std::move(np));
    for (auto& np : right_nfas) nfas.push_back(std::move(np));
    return true;
}

}  // namespace

int compile_database(const char* const* patterns, const unsigned* flags, const unsigned* ids, unsigned n,
                     std::shared_ptr<Database>& out, std::string& error) {
    const int kDbError = 4;  // HYPERSCANNER_DB (reference hyperscanner.c:29)
    if (n == 0 || !patterns) { error = "no patterns"; return kDbError; }
    auto db = std::make_shared<Database>();
    std::vector<NodePtr> asts;
    db->simple = true;
    for (unsigned i = 0; i < n; i++) {
        PatternInfo p;
        if (!patterns[i] || !patterns[i][0]) { error = "empty pattern"; return kDbError; }
        p.source = patterns[i];
        p.flags = flags ? flags[i] : 0;
        p.id = ids ? ids[i] : 0;
        if (p.flags & ~(FLAG_CASELESS | FLAG_DOTALL | FLAG_MULTILINE | FLAG_SINGLEMATCH)) {
            error = "pattern " + std::to_string(i) + ": unsupported flag bits";
            return kDbError;
        }
        ParseResult pr = parse_regex(p.source, p.flags);
        if (!pr.root) { error = "pattern " + std::to_string(i) + ": " + pr.error; return kDbError; }
        if (matches_empty_buffer(*pr.root)) { error = "pattern " + std::to_string(i) + " matches the empty buffer"; return kDbError; }
        {   // per-pattern size check (unrolled repeats)
            Nfa probe;
            if (!nfa_add_pattern(probe, *pr.root, 0, kMaxPatternInsts)) { error = "pattern " + std::to_string(i) + " is too large"; return kDbError; }
        }
        if (!(p.flags & FLAG_SINGLEMATCH) || p.id != (ids ? ids[0] : 0)) db->simple = false;
        asts.push_back(std::move(pr.root));
        db->patterns.push_back(std::move(p));
    }
    // hs_compile.h: expressions sharing a match id must agree on SINGLEMATCH
    {
        std::map<unsigned, unsigned> sm;
        for (auto& p : db->patterns) {
            unsigned v = p.flags & FLAG_SINGLEMATCH;
            auto it = sm.find(p.id);
            if (it == sm.end()) sm.emplace(p.id, v);
            else if (it->second != v) { error = "expressions sharing id " + std::to_string(p.id) + " disagree on SINGLEMATCH"; return kDbError; }
        }
    }
    db->simple_id = db->patterns[0].id;

    std::vector<int> idx(n);
    for (unsigned i = 0; i < n; i++) idx[i] = (int)i;
    size_t max_states = env_size("GPUGREP_MAX_DFA_STATES", 40000);
    if (!build_groups(asts, idx, 0, n, db->simple, max_states, db->groups, db->nfas, error)) return kDbError;

    // flatten accept sets into (id, singlematch) report lists
    db->report_begin.resize(db->groups.size());
    for (size_t g = 0; g < db->groups.size(); g++) {
        const DfaGroup& grp = db->groups[g];
        for (auto& set : grp.dfa.accept_sets) {
            db->report_begin[g].push_back((uint32_t)db->reports.size());
            std::vector<std::pair<unsigned, unsigned>> reps;
            for (int local : set) {
                const PatternInfo& p = db->patterns[grp.members[local]];
                reps.emplace_back(p.id, (p.flags & FLAG_SINGLEMATCH) ? 1u : 0u);
            }
            std::sort(reps.begin(), reps.end());
            reps.erase(std::unique(reps.begin(), reps.end()), reps.end());
            for (auto& r : reps) db->reports.push_back(ReportDesc{r.first, r.second});
        }
        db->report_begin[g].push_back((uint32_t)db->reports.size());
    }

    for (auto& np : db->nfas) {
        np.report_begin = (uint32_t)db->reports.size();
        const PatternInfo& p = db->patterns[np.pattern];
        db->reports.push_back(ReportDesc{p.id, (p.flags & FLAG_SINGLEMATCH) ? 1u : 0u});
    }

    std::vector<const Node*> raw;
    for (unsigned i = 0; i < n; i++) raw.push_back(asts[i].get());
    if (env_size("GPUGREP_NO_PREFILTER", 0) == 0) {
        db->factors = analyse_factors(raw);
        // which DFA group(s) a pattern's grams lead to: the verification kernel walks only those (prefilter.hpp)
        db->factors.group_mask.assign(n, 0u);
        for (size_t g = 0; g < db->groups.size(); g++)
            for (int member : db->groups[g].members) db->factors.group_mask[(size_t)member] |= 1u << (g & 31);
        // NFA-fallback patterns: bit 31 (shared with DFA groups 31, 63, ... - a superset, the NFA check then runs for nothing)
        for (auto& np : db->nfas) db->factors.group_mask[(size_t)np.pattern] = 0x80000000u;
        build_prefilter(db->factors, nullptr, db->prefilter);
    } else {
        db->prefilter.note = db->factors.note = "disabled by GPUGREP_NO_PREFILTER";
    }
    out = db;
    return 0;
}

namespace {

// Most recent first; a fixed-string set and a regex set never share an entry, whatever their keys.
std::shared_ptr<Database> cached(bool literal, std::string key, const std::function<int(std::shared_ptr<Database>&)>& compile, int& rc) {
    static std::mutex mu;
    static std::list<std::shared_ptr<Database>> cache;
    {
        std::lock_guard<std::mutex> lk(mu);
        for (auto it = cache.begin(); it != cache.end(); ++it) {
            if ((*it)->literal == literal && (*it)->key == key) {
                auto db = *it;
                cache.erase(it);
                cache.push_front(db);
                rc = 0;
                return db;
            }
        }
    }
    std::shared_ptr<Database> db;
    rc = compile(db);
    if (rc != 0) return nullptr;
    db->key = std::move(key);
    std::lock_guard<std::mutex> lk(mu);
    cache.push_front(db);
    while (cache.size() > 8) cache.pop_back();
    return db;
}

// (built for every scan call: 10,000 patterns are 300 KB of key, so no per-pattern formatting or allocation here)
std::string cache_key(const char* const* patterns, const unsigned* flags, const unsigned* ids, unsigned n) {
    std::string key;
    key.reserve((size_t)n * 48 + 64);
    for (unsigned i = 0; i < n; i++) {
        if (!patterns || !patterns[i]) break;
        key.append(patterns[i]);
        const unsigned tail[2] = {flags ? flags[i] : 0u, ids ? ids[i] : 0u};
        key.push_back('\0');
        key.append(reinterpret_cast<const char*>(tail), sizeof(tail));
    }
    key.append(std::getenv("GPUGREP_NO_PREFILTER") ? "np" : "");
    return key;
}

}  // namespace

std::shared_ptr<Database> cached_database(const char* const* patterns, const unsigned* flags, const unsigned* ids,
                                          unsigned n, int& rc, std::string& error) {
    std::string key = cache_key(patterns, flags, ids, n);
    if (const char* b = std::getenv("GPUGREP_MAX_DFA_STATES")) key.append(b);
    return cached(false, std::move(key), [&](std::shared_ptr<Database>& db) { return compile_database(patterns, flags, ids, n, db, error); }, rc);
}

// ---- fixed strings ----------------------------------------------------------------------------------------------
int check_literals(const char* const* literals, const unsigned* flags, unsigned n, std::string& error) {
    const int kDbError = 4;
    if (n == 0 || !literals) { error = "no literals"; return kDbError; }
    for (unsigned i = 0; i < n; i++) {
        if (!literals[i] || !literals[i][0]) { error = "literal " + std::to_string(i) + " is empty"; return kDbError; }
        if (flags && (flags[i] & ~(FLAG_CASELESS | FLAG_DOTALL | FLAG_MULTILINE | FLAG_SINGLEMATCH))) {
            error = "literal " + std::to_string(i) + ": unsupported flag bits";
            return kDbError;
        }
    }
    return 0;
}

int compile_literal_database(const char* const* literals, const unsigned* flags, unsigned n, std::shared_ptr<Database>& out,
                             std::string& error) {
    int rc = check_literals(literals, flags, n, error);
    if (rc) return rc;
    auto db = std::make_shared<Database>();
    db->simple = true;
    db->simple_id = 0;
    db->literal = true;
    LiteralSet& L = db->literals;
    L.given = n;
    // folded candidates per class, sorted; a literal with '\n' before its last byte can never lie inside a line
    struct Cand { std::string_view text; unsigned cls; };
    std::vector<std::string> folded(n);
    std::vector<Cand> cands;
    cands.reserve(n);
    for (unsigned i = 0; i < n; i++) {
        const size_t len = std::strlen(literals[i]);
        const char* nl = static_cast<const char*>(std::memchr(literals[i], '\n', len));
        if (nl && nl != literals[i] + len - 1) continue;
        const unsigned cls = flags && (flags[i] & FLAG_CASELESS) ? 1u : 0u;
        folded[i].assign(literals[i], len);
        if (cls) for (char& c : folded[i]) c = (char)fold_ascii((uint8_t)c);
        cands.push_back(Cand{folded[i], cls});
    }
    std::sort(cands.begin(), cands.end(), [](const Cand& a, const Cand& b) { return a.cls != b.cls ? a.cls < b.cls : a.text < b.text; });
    // prefix-free per class: in sorted order every string that has a kept prefix follows that prefix directly
    std::vector<Cand> kept;
    for (const Cand& c : cands) {
        if (!kept.empty() && kept.back().cls == c.cls && c.text.substr(0, kept.back().text.size()) == kept.back().text) continue;
        kept.push_back(c);
    }
    L.bucket.assign(2 * 65537, 0);
    L.one.assign(2 * 8, 0);
    size_t total = 0;
    for (const Cand& c : kept) total += c.text.size();
    L.bytes.reserve(total);
    std::vector<uint32_t> count(2 * 65536, 0);
    for (const Cand& c : kept) {
        const uint32_t id = (uint32_t)L.off.size();
        L.off.push_back((uint32_t)L.bytes.size());
        L.len.push_back((uint32_t)c.text.size());
        L.caseless.push_back((uint8_t)c.cls);
        L.bytes.insert(L.bytes.end(), c.text.begin(), c.text.end());
        const uint8_t b0 = (uint8_t)c.text[0];
        if (c.text.size() == 1) {
            L.one[c.cls * 8 + b0 / 32] |= 1u << (b0 % 32);
            L.rank.push_back(0);
        } else {
            L.rank.push_back((uint32_t)L.order.size());
            L.order.push_back(id);
            count[c.cls * 65536 + ((uint32_t)b0 << 8 | (uint8_t)c.text[1])]++;
        }
    }
    // (order is sorted by class, then bytes: the literals of one two-byte prefix are one range of it)
    uint32_t at = 0;
    for (unsigned cls = 0; cls < 2; cls++) {
        for (uint32_t k = 0; k < 65536; k++) {
            L.bucket[cls * 65537 + k] = at;
            at += count[cls * 65536 + k];
        }
        L.bucket[cls * 65537 + 65536] = at;
    }
    // one class-string per literal: the prefilter picks a rare window in each (caseless letters: both cases)
    const size_t m = L.off.size();
    FactorSet& fs = db->factors;
    fs.factors.resize(m);
    fs.before.assign(m, 0);
    fs.literal_rank = L.rank;
    fs.literal_class = L.caseless;
    size_t min_len = m ? SIZE_MAX : 0;
    for (size_t i = 0; i < m; i++) {
        ClassString s(L.len[i]);
        for (uint32_t k = 0; k < L.len[i]; k++) {
            const uint8_t b = L.bytes[L.off[i] + k];
            s[k].set(b);
            if (L.caseless[i] && (unsigned)b - 'a' < 26u) s[k].set(b & ~0x20u);
        }
        fs.factors[i].push_back(std::move(s));
        min_len = std::min<size_t>(min_len, L.len[i]);
    }
    fs.min_len = min_len;
    fs.usable = m > 0 && min_len >= 4;
    if (!fs.usable) fs.note = m ? "a literal is shorter than 4 bytes" : "no literal can match";
    if (fs.usable && env_size("GPUGREP_NO_PREFILTER", 0) != 0) {
        fs.usable = false;
        db->prefilter.note = fs.note = "disabled by GPUGREP_NO_PREFILTER";
    }
    if (fs.usable) build_prefilter(fs, nullptr, db->prefilter);
    else if (db->prefilter.note.empty()) db->prefilter.note = fs.note;
    PatternInfo info;
    info.source = "(" + std::to_string(n) + " literals)";
    db->patterns.push_back(std::move(info));
    out = db;
    return 0;
}

std::shared_ptr<Database> cached_literal_database(const char* const* literals, const unsigned* flags, unsigned n, int& rc,
                                                  std::string& error) {
    return cached(true, cache_key(literals, flags, nullptr, n),
                  [&](std::shared_ptr<Database>& db) { return compile_literal_database(literals, flags, n, db, error); }, rc);
}

// The report table (database.hpp LiteralReports) of the literals that can lie inside a line, and the (id, singlematch)
// descriptors of its nodes in db.reports.  The literals have passed check_literals.
static void build_literal_reports(const char* const* literals, const unsigned* flags, const unsigned* ids, unsigned n, Database& db) {
    LiteralReports& R = db.lit_reports;
    struct Given { std::string text; unsigned cls, id, sm; };
    std::vector<Given> given;
    given.reserve(n);
    for (unsigned i = 0; i < n; i++) {
        const size_t len = std::strlen(literals[i]);
        const char* nl = static_cast<const char*>(std::memchr(literals[i], '\n', len));
        if (nl && nl != literals[i] + len - 1) continue;   // can never lie inside a line
        Given g{std::string(literals[i], len), flags && (flags[i] & FLAG_CASELESS) ? 1u : 0u, ids ? ids[i] : 0u,
                flags && (flags[i] & FLAG_SINGLEMATCH) ? 1u : 0u};
        if (g.cls) for (char& c : g.text) c = (char)fold_ascii((uint8_t)c);
        given.push_back(std::move(g));
    }
    std::sort(given.begin(), given.end(), [](const Given& a, const Given& b) {
        if (a.cls != b.cls) return a.cls < b.cls;
        if (a.text != b.text) return a.text < b.text;
        return a.id != b.id ? a.id < b.id : a.sm < b.sm;
    });
    R.bucket.assign(2 * 65537, 0);
    R.one.assign(2 * 256, kNoLiteral);
    std::vector<uint32_t> count(2 * 65536, 0);
    std::vector<uint32_t> chain;   // the nodes that are prefixes of the last node, shortest first
    for (size_t i = 0; i < given.size(); i++) {
        const Given& g = given[i];
        const bool fresh = i == 0 || given[i - 1].cls != g.cls || given[i - 1].text != g.text;
        if (fresh) {
            const uint32_t node = (uint32_t)R.off.size();
            // (in byte order every node that is a prefix of this one comes before it, and is on the chain of its predecessor)
            while (!chain.empty()) {
                const uint32_t top = chain.back();
                const std::string_view t(reinterpret_cast<const char*>(R.bytes.data()) + R.off[top], R.len[top]);
                if (R.caseless[top] == g.cls && t.size() < g.text.size() && std::string_view(g.text).substr(0, t.size()) == t) break;
                chain.pop_back();
            }
            R.parent.push_back(chain.empty() ? kNoLiteral : chain.back());
            chain.push_back(node);
            R.off.push_back((uint32_t)R.bytes.size());
            R.len.push_back((uint32_t)g.text.size());
            R.caseless.push_back((uint8_t)g.cls);
            R.bytes.insert(R.bytes.end(), g.text.begin(), g.text.end());
            R.report_begin.push_back((uint32_t)db.reports.size());
            const uint8_t b0 = (uint8_t)g.text[0];
            if (g.text.size() == 1) {
                R.one[g.cls * 256 + b0] = node;
            } else {
                R.order.push_back(node);
                count[g.cls * 65536 + ((uint32_t)b0 << 8 | (uint8_t)g.text[1])]++;
            }
        }
        if (fresh || given[i - 1].id != g.id || given[i - 1].sm != g.sm) db.reports.push_back(ReportDesc{g.id, g.sm});
    }
    R.report_begin.push_back((uint32_t)db.reports.size());
    uint32_t at = 0;
    for (unsigned cls = 0; cls < 2; cls++) {
        for (uint32_t k = 0; k < 65536; k++) {
            R.bucket[cls * 65537 + k] = at;
            at += count[cls * 65536 + k];
        }
        R.bucket[cls * 65537 + 65536] = at;
    }
}

int compile_literal_report_database(const char* const* literals, const unsigned* flags, const unsigned* ids, unsigned n,
                                    std::shared_ptr<Database>& out, std::string& error) {
    const int kDbError = 4;
    int rc = check_literals(literals, flags, n, error);
    if (rc) return rc;
    {   // hs_compile.h: expressions sharing a match id must agree on SINGLEMATCH
        std::map<unsigned, unsigned> sm;
        for (unsigned i = 0; i < n; i++) {
            const unsigned id = ids ? ids[i] : 0u, v = flags ? flags[i] & FLAG_SINGLEMATCH : 0u;
            auto it = sm.emplace(id, v).first;
            if (it->second != v) { error = "literals sharing id " + std::to_string(id) + " disagree on SINGLEMATCH"; return kDbError; }
        }
    }
    rc = compile_literal_database(literals, flags, n, out, error);
    if (rc) return rc;
    build_literal_reports(literals, flags, ids, n, *out);
    out->literal_reports = true;
    return 0;
}

std::shared_ptr<Database> cached_literal_report_database(const char* const* literals, const unsigned* flags, const unsigned* ids,
                                                         unsigned n, int& rc, std::string& error) {
    // (the ids and every flag bit are part of the key; the tag keeps it apart from a selection set with ids 0)
    std::string key = cache_key(literals, flags, ids, n);
    key.append("\x01reports");
    return cached(true, std::move(key),
                  [&](std::shared_ptr<Database>& db) { return compile_literal_report_database(literals, flags, ids, n, db, error); }, rc);
}

int compile_literal_whole_database(const char* const* literals, const unsigned* flags, unsigned n, std::shared_ptr<Database>& out,
                                   std::string& error) {
    int rc = compile_literal_database(literals, flags, n, out, error);
    if (rc) return rc;
    // (ids and SINGLEMATCH do not matter here: the table only tells which literals occur where)
    build_literal_reports(literals, flags, nullptr, n, *out);
    out->literal_whole = true;
    return 0;
}

std::shared_ptr<Database> cached_literal_whole_database(const char* const* literals, const unsigned* flags, unsigned n, int& rc,
                                                        std::string& error) {
    // (one entry serves word and line scans: the mode is a slot setting; the tag keeps it apart from the other two kinds)
    std::string key = cache_key(literals, flags, nullptr, n);
    key.append("\x01whole");
    return cached(true, std::move(key),
                  [&](std::shared_ptr<Database>& db) { return compile_literal_whole_database(literals, flags, n, db, error); }, rc);
}

}  // namespace gpugrep
