// C ABI: check_patterns() and the compiled-database introspection entry points of include/gpugrep.h.
// Host only: nothing here touches CUDA, so it is safe to call before fork() (SURVEY.md §8b).
#include <cctype>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>

#include "../../include/gpugrep.h"
#include "automata.hpp"
#include "database.hpp"
#include "pike_vm.hpp"
#include "regex.hpp"

namespace gpugrep {
thread_local std::string g_last_error;
void set_last_error(const std::string& e) { g_last_error = e; }
}  // namespace gpugrep

namespace gpugrep {
namespace {

// Width of every match, or -1 when it varies.
int fixed_width(const Node& n) {
    switch (n.kind) {
        case NodeKind::Empty: return 0;
        case NodeKind::Assert: return 0;
        case NodeKind::Set: return 1;
        case NodeKind::Concat: {
            int total = 0;
            for (const NodePtr& k : n.kids) {
                const int w = fixed_width(*k);
                if (w < 0) return -1;
                total += w;
            }
            return total;
        }
        case NodeKind::Alt: {
            int width = -2;
            for (const NodePtr& k : n.kids) {
                const int w = fixed_width(*k);
                if (w < 0 || (width != -2 && w != width)) return -1;
                width = w;
            }
            return width == -2 ? 0 : width;
        }
        case NodeKind::Repeat: {
            const int w = n.kids.empty() ? 0 : fixed_width(*n.kids[0]);
            if (w < 0 || n.min != n.max || n.max < 0) return -1;
            return w * n.min;
        }
    }
    return -1;
}

// Conservative lexical screen: only syntax that Python's re (str pattern, no flags, ASCII text) and this compiler read
// the same way.  Everything else keeps the reference's re.finditer() path.
bool same_meaning_in_python(const std::string& p) {
    bool in_class = false;
    for (size_t i = 0; i < p.size(); i++) {
        const unsigned char c = (unsigned char)p[i];
        if (c < 0x20 || c > 0x7e) return false;
        if (c == '\\') {
            if (i + 1 >= p.size()) return false;
            const unsigned char e = (unsigned char)p[++i];
            if (e == 'x') {   // exactly two hex digits in Python
                if (i + 2 >= p.size() || !std::isxdigit((unsigned char)p[i + 1]) || !std::isxdigit((unsigned char)p[i + 2])) return false;
                i += 2;
                continue;
            }
            if (std::isalnum(e)) {
                if (in_class ? std::strchr("dDwWntrf", e) == nullptr : std::strchr("dDwWbBAntrf", e) == nullptr) return false;
            }
            continue;
        }
        if (in_class) {
            if (c == '[') return false;                  // POSIX classes / nested sets
            if (c == ']' && !(p[i - 1] == '[' || (p[i - 1] == '^' && i >= 2 && p[i - 2] == '['))) in_class = false;
            continue;
        }
        switch (c) {
            case '[': in_class = true; break;
            case '*': case '+': return false;
            case '?': if (i < 1 || p[i - 1] != '(') return false; if (i + 1 >= p.size() || p[i + 1] != ':') return false; break;   // only (?:
            case '{': {   // only {digits}
                size_t j = i + 1;
                while (j < p.size() && std::isdigit((unsigned char)p[j])) j++;
                if (j == i + 1 || j >= p.size() || p[j] != '}') return false;
                if (j + 1 < p.size() && (p[j + 1] == '?' || p[j + 1] == '+' || p[j + 1] == '{')) return false;
                i = j;
                break;
            }
            case '}': return false;
            case '$': return false;   // end-or-final-newline consumes the newline in the automaton
            default: break;
        }
    }
    return !in_class;
}

// Lexical screen of the span route: the syntax of same_meaning_in_python plus the quantifiers * + ? {m} {m,} {m,n} and their
// lazy forms.  Python reads {,n} as {0,n} where this compiler reads a literal; a quantifier after a quantifier is an error
// in Python (or possessive, from 3.11 on); Python's str \s includes 0x1C-0x1F; $, inline flags and POSIX classes differ too.
bool spans_mean_the_same_in_python(const std::string& p) {
    bool in_class = false;
    bool can_repeat = false;   // the previous item is an atom a quantifier may follow
    for (size_t i = 0; i < p.size(); i++) {
        const unsigned char c = (unsigned char)p[i];
        if (c < 0x20 || c > 0x7e) return false;
        if (c == '\\') {
            if (i + 1 >= p.size()) return false;
            const unsigned char e = (unsigned char)p[++i];
            if (e == 'x') {   // exactly two hex digits in Python
                if (i + 2 >= p.size() || !std::isxdigit((unsigned char)p[i + 1]) || !std::isxdigit((unsigned char)p[i + 2])) return false;
                i += 2;
            } else if (std::isalnum(e)) {
                if (in_class ? std::strchr("dDwWntrf", e) == nullptr : std::strchr("dDwWbBAntrf", e) == nullptr) return false;
            }
            if (!in_class) can_repeat = !(e == 'b' || e == 'B' || e == 'A');
            continue;
        }
        if (in_class) {
            if (c == '[') return false;                  // POSIX classes / nested sets
            if (c == ']' && !(p[i - 1] == '[' || (p[i - 1] == '^' && i >= 2 && p[i - 2] == '['))) { in_class = false; can_repeat = true; }
            continue;
        }
        size_t quantifier_end = 0;   // index of the last byte of a quantifier at i, 0 if none
        switch (c) {
            case '[': in_class = true; break;
            case '(':
                if (i + 1 < p.size() && p[i + 1] == '?') {   // only (?:
                    if (i + 2 >= p.size() || p[i + 2] != ':') return false;
                    i += 2;
                }
                can_repeat = false;
                continue;
            case ')': can_repeat = true; continue;
            case '|': case '^': can_repeat = false; continue;
            case '*': case '+': case '?': quantifier_end = i; break;
            case '{': {   // {m} {m,} {m,n}
                size_t j = i + 1;
                while (j < p.size() && std::isdigit((unsigned char)p[j])) j++;
                if (j == i + 1) return false;
                if (j < p.size() && p[j] == ',') {
                    j++;
                    while (j < p.size() && std::isdigit((unsigned char)p[j])) j++;
                }
                if (j >= p.size() || p[j] != '}') return false;
                quantifier_end = j;
                break;
            }
            case '}': return false;
            case '$': return false;
            default: can_repeat = true; continue;
        }
        if (c == '[') continue;
        if (!can_repeat) return false;
        i = quantifier_end;
        if (i + 1 < p.size() && p[i + 1] == '?') i++;   // lazy
        if (i + 1 < p.size() && (p[i + 1] == '*' || p[i + 1] == '+' || p[i + 1] == '?' || p[i + 1] == '{')) return false;
        can_repeat = false;
    }
    return !in_class;
}

// pike_vm.hpp cannot include regex.hpp (device code): its assertion codes are the AssertKind values
static_assert(kPikeBeginBuffer == (uint32_t)AssertKind::BeginBuffer && kPikeWordBoundary == (uint32_t)AssertKind::WordBoundary &&
                  kPikeNotWordBoundary == (uint32_t)AssertKind::NotWordBoundary,
              "pike_vm.hpp assertion codes must equal regex.hpp AssertKind values");

// A node that can match without consuming a byte (assertions count as empty).
bool nullable(const Node& n) { return matches_empty_buffer(n); }

bool repeats_consume(const Node& n) {
    if (n.kind == NodeKind::Repeat && (n.kids.empty() || nullable(*n.kids[0]))) return false;
    for (const NodePtr& k : n.kids)
        if (!repeats_consume(*k)) return false;
    return true;
}

// The span program of a screened pattern, or false.
bool span_program(const std::string& text, PikeProgram& out) {
    if (!spans_mean_the_same_in_python(text)) return false;
    ParseResult parsed = parse_regex(text, 0);
    if (!parsed.root || nullable(*parsed.root) || !repeats_consume(*parsed.root)) return false;
    Nfa nfa;
    if (!nfa_add_pattern(nfa, *parsed.root, 0, (size_t)kPikeMaxInsts, /*lazy=*/true)) return false;
    if (nfa.sets.size() > 256) return false;
    out.insts.clear();
    out.sets.clear();
    for (const NfaInst& in : nfa.prog) {
        switch (in.op) {
            case NfaInst::Byte: out.insts.push_back(pike_inst(kPikeByte, (uint32_t)in.arg, (uint32_t)in.x, 0)); break;
            case NfaInst::Split: out.insts.push_back(pike_inst(kPikeSplit, 0, (uint32_t)in.x, (uint32_t)in.y)); break;
            case NfaInst::Match: out.insts.push_back(pike_inst(kPikeMatch, 0, 0, 0)); break;
            case NfaInst::Assert: {
                const AssertKind k = (AssertKind)in.arg;
                if (k != AssertKind::BeginBuffer && k != AssertKind::WordBoundary && k != AssertKind::NotWordBoundary) return false;
                out.insts.push_back(pike_inst(kPikeAssert, (uint32_t)in.arg, (uint32_t)in.x, 0));
                break;
            }
        }
    }
    for (const ByteSet& s : nfa.sets)
        for (int w = 0; w < 4; w++) {
            out.sets.push_back((uint32_t)s.w[w]);
            out.sets.push_back((uint32_t)(s.w[w] >> 32));
        }
    out.start = nfa.starts[0];
    return true;
}

}  // namespace

bool build_pike_program(const char* pattern, PikeProgram& out) { return pattern && span_program(pattern, out); }

}  // namespace gpugrep

struct gpugrep_db {
    std::shared_ptr<gpugrep::Database> db;
};

extern "C" {

// Replaces reference hyperscanner.c:154-167.
int check_patterns(const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
                   const unsigned int elements) {
    int rc = 0;
    std::string err;
    auto db = gpugrep::cached_database(patterns, pattern_flags, pattern_ids, elements, rc, err);
    if (!db) {
        gpugrep::set_last_error(err);
        return GPUGREP_DB;
    }
    gpugrep::set_last_error("");
    return 0;
}

int gpugrep_check_literals(const char* const* literals, const unsigned int* literal_flags, unsigned int elements) {
    std::string err;
    const int rc = gpugrep::check_literals(literals, literal_flags, elements, err);
    gpugrep::set_last_error(err);
    return rc;
}

int gpugrep_span_width(const char* pattern) {
    if (!pattern) return -1;
    const std::string text(pattern);
    if (!gpugrep::same_meaning_in_python(text)) return -1;
    gpugrep::ParseResult parsed = gpugrep::parse_regex(text, 0);
    if (!parsed.root) return -1;
    const int width = gpugrep::fixed_width(*parsed.root);
    return width > 0 ? width : -1;
}

int gpugrep_span_exact(const char* pattern) {
    gpugrep::PikeProgram program;
    return gpugrep::build_pike_program(pattern, program) ? 1 : 0;
}

const char* gpugrep_last_error(void) { return gpugrep::g_last_error.c_str(); }
const char* gpugrep_version(void) { return "gpugrep 0.1.0 (sm_100a)"; }

gpugrep_db* gpugrep_db_compile(const char* const* patterns, const unsigned int* pattern_flags,
                               const unsigned int* pattern_ids, unsigned int elements, int* rc) {
    std::string err;
    std::shared_ptr<gpugrep::Database> db;
    int r = gpugrep::compile_database(patterns, pattern_flags, pattern_ids, elements, db, err);
    if (rc) *rc = r;
    gpugrep::set_last_error(err);
    if (r != 0) return nullptr;
    return new gpugrep_db{db};
}

void gpugrep_db_free(gpugrep_db* db) { delete db; }

int gpugrep_db_get_info(const gpugrep_db* h, gpugrep_db_info* out) {
    if (!h || !out) return -1;
    const gpugrep::Database& db = *h->db;
    std::memset(out, 0, sizeof(*out));
    out->patterns = (unsigned)db.patterns.size();
    out->groups = (unsigned)db.groups.size();
    out->simple = db.simple;
    out->simple_id = db.simple_id;
    out->prefilter = db.prefilter.enabled;
    out->prefilter_stride = (unsigned)db.prefilter.stride;
    out->prefilter_fold = db.prefilter.fold_case;
    out->prefilter_log2_bits = (unsigned)(db.prefilter.exact ? db.prefilter.log2_slots : db.prefilter.log2_bits);
    out->reserved = db.prefilter.exact ? 1u : 0u;
    out->prefilter_grams = (unsigned)db.prefilter.num_grams;
    out->prefilter_min_factor = (unsigned)db.prefilter.min_factor_len;
    out->prefilter_lookback = db.prefilter.lookback;
    for (auto& g : db.groups) out->total_states += (unsigned)g.dfa.num_states;
    return 0;
}

int gpugrep_db_get_group(const gpugrep_db* h, unsigned int group, gpugrep_group_info* out) {
    if (!h || !out || group >= h->db->groups.size()) return -1;
    const gpugrep::Dfa& d = h->db->groups[group].dfa;
    out->states = (unsigned)d.num_states;
    out->classes = (unsigned)d.num_classes;
    out->stride = (unsigned)d.stride;
    out->first_accept = (unsigned)d.first_accept;
    out->sink_match = d.sink_match;
    out->dead = d.dead;
    out->accept_sets = (unsigned)d.accept_sets.size();
    out->members = (unsigned)h->db->groups[group].members.size();
    out->entry_mid_other = (unsigned)d.entry_mid_other;
    out->entry_mid_word = (unsigned)d.entry_mid_word;
    out->idle_end = (unsigned)d.idle_end;
    out->reserved = 0;
    return 0;
}

int gpugrep_db_copy_group(const gpugrep_db* h, unsigned int group, uint8_t* byte_class, uint32_t* trans, uint32_t* accept_of) {
    if (!h || group >= h->db->groups.size()) return -1;
    const gpugrep::Dfa& d = h->db->groups[group].dfa;
    if (byte_class) std::memcpy(byte_class, d.byte_class, 256);
    if (trans) std::memcpy(trans, d.trans.data(), d.trans.size() * sizeof(uint32_t));
    if (accept_of) std::memcpy(accept_of, d.accept_of.data(), d.accept_of.size() * sizeof(uint32_t));
    return 0;
}

int gpugrep_db_accept_reports(const gpugrep_db* h, unsigned int group, unsigned int accept, unsigned int* ids,
                              unsigned int* singlematch, unsigned int cap) {
    if (!h || group >= h->db->groups.size()) return -1;
    const auto& rb = h->db->report_begin[group];
    if (accept + 1 >= rb.size()) return -1;
    unsigned n = 0;
    for (uint32_t k = rb[accept]; k < rb[accept + 1]; k++, n++) {
        if (n < cap) {
            if (ids) ids[n] = h->db->reports[k].id;
            if (singlematch) singlematch[n] = h->db->reports[k].singlematch;
        }
    }
    return (int)n;
}

size_t gpugrep_db_copy_depth(const gpugrep_db* h, unsigned int group, uint8_t* depth, size_t cap) {
    if (!h || group >= h->db->groups.size()) return 0;
    const auto& d = h->db->groups[group].dfa.depth;
    if (depth) std::memcpy(depth, d.data(), std::min(cap, d.size()));
    return d.size();
}

size_t gpugrep_db_copy_prefilter(const gpugrep_db* h, uint32_t* words, size_t cap_words, uint32_t* bloom_mul) {
    if (!h || !h->db->prefilter.enabled) return 0;
    const auto& pf = h->db->prefilter;
    size_t n = std::min(cap_words, pf.bitmap.size());
    if (words) std::memcpy(words, pf.bitmap.data(), n * sizeof(uint32_t));
    if (bloom_mul) *bloom_mul = pf.bloom_mul;   // the bitmap's multiplier (a tuned table picks it), not the exact table's
    return n;
}

size_t gpugrep_db_copy_grams(const gpugrep_db* h, uint32_t* out, size_t cap) {
    if (!h) return 0;
    const auto& g = h->db->prefilter.grams;
    size_t n = std::min(cap, g.size());
    if (out) std::memcpy(out, g.data(), n * sizeof(uint32_t));
    return g.size();
}

size_t gpugrep_db_copy_odd_compares(const gpugrep_db* h, uint32_t* out, size_t cap) {
    if (!h) return 0;
    const auto& odd = h->db->prefilter.odd;
    for (size_t k = 0; k < odd.size() && k < cap && out; k++) { out[2 * k] = odd[k].mul; out[2 * k + 1] = odd[k].add; }
    return odd.size();
}

int gpugrep_db_tune(gpugrep_db* h, const void* sample, size_t size) {
    if (!h || !h->db->factors.usable) return -1;
    gpugrep::GramHistogram hist;
    hist.add_sample((const uint8_t*)sample, size);
    gpugrep::build_prefilter(h->db->factors, &hist, h->db->prefilter);
    return h->db->prefilter.enabled ? 0 : -1;
}

const char* gpugrep_db_prefilter_note(const gpugrep_db* h) { return h ? h->db->prefilter.note.c_str() : ""; }

}  // extern "C"
