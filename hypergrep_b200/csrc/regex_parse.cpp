// Recursive-descent parser for the Hyperscan-supported PCRE subset (see regex.hpp).
// Accept/reject decisions follow Hyperscan's documented "Unsupported Constructs" list: anything that needs
// backtracking or sub-match state (look-around, back-references, atomic/possessive, conditionals, recursion,
// verbs, \C \R \K \X \G, callouts, unicode properties in byte mode) is a compile failure, surfaced by the
// C boundary as code 4 exactly like the reference (hyperscanner.c:162-164, 296-299).
#include "regex.hpp"

#include <cctype>

namespace gpugrep {

bool is_word_byte(unsigned b) { return (b >= '0' && b <= '9') || (b >= 'A' && b <= 'Z') || (b >= 'a' && b <= 'z') || b == '_'; }

namespace {

struct Flags {
    bool caseless, dotall, multiline, extended;
};

ByteSet fold_case(ByteSet s) {
    ByteSet r = s;
    for (unsigned c = 'a'; c <= 'z'; c++) {
        if (s.test(c)) r.set(c - 32);
        if (s.test(c - 32)) r.set(c);
    }
    return r;
}

ByteSet set_digit() { ByteSet s; s.set_range('0', '9'); return s; }
ByteSet set_word() { ByteSet s; for (unsigned b = 0; b < 256; b++) if (is_word_byte(b)) s.set(b); return s; }
ByteSet set_space() { ByteSet s; s.set_range(9, 13); s.set(32); return s; }
ByteSet set_hspace() { ByteSet s; s.set(9); s.set(32); s.set(0xA0); return s; }
ByteSet set_vspace() { ByteSet s; s.set_range(10, 13); s.set(0x85); return s; }

NodePtr mk(NodeKind k) { auto n = std::make_unique<Node>(); n->kind = k; return n; }
NodePtr mk_set(const ByteSet& s) { auto n = mk(NodeKind::Set); n->set = s; return n; }
NodePtr mk_assert(AssertKind a) { auto n = mk(NodeKind::Assert); n->assert_kind = a; return n; }

// `$` without MULTILINE and \Z: end of block, or before a '\n' that ends the block.  Every block this engine
// scans is one pseudo-line (reference hyperscanner.c:199,217), so a '\n' can only ever be the block's last byte
// and the assertion coincides with the MULTILINE `$` (EndLine): next symbol is '\n' or end of data.
NodePtr mk_end_or_final_newline() { return mk_assert(AssertKind::EndLine); }

class Parser {
public:
    Parser(const std::string& src, unsigned hs_flags) : s_(src) {
        top_.caseless = hs_flags & FLAG_CASELESS;
        top_.dotall = hs_flags & FLAG_DOTALL;
        top_.multiline = hs_flags & FLAG_MULTILINE;
        top_.extended = false;
    }

    ParseResult run() {
        ParseResult r;
        Flags f = top_;
        NodePtr n = parse_alternation(f, 0);
        if (!err_.empty()) { r.error = err_; return r; }
        if (i_ < s_.size()) { r.error = "unmatched ')'"; return r; }
        r.root = std::move(n);
        return r;
    }

private:
    const std::string& s_;
    size_t i_ = 0;
    Flags top_;
    std::string err_;
    int group_depth_ = 0;

    bool eof() const { return i_ >= s_.size(); }
    unsigned char peek(size_t k = 0) const { return i_ + k < s_.size() ? (unsigned char)s_[i_ + k] : 0; }
    bool fail(const char* msg) { if (err_.empty()) err_ = msg; return false; }

    void skip_extended(const Flags& f) {
        if (!f.extended) return;
        while (!eof()) {
            unsigned char c = peek();
            if (c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '\f' || c == '\v') { i_++; continue; }
            if (c == '#') { while (!eof() && peek() != '\n') i_++; continue; }
            break;
        }
    }

    NodePtr parse_alternation(Flags& f, int depth) {
        if (depth > 200) { fail("nesting too deep"); return nullptr; }
        std::vector<NodePtr> branches;
        branches.push_back(parse_branch(f, depth));
        while (err_.empty() && !eof() && peek() == '|') {
            i_++;
            branches.push_back(parse_branch(f, depth));
        }
        if (!err_.empty()) return nullptr;
        if (branches.size() == 1) return std::move(branches[0]);
        auto alt = mk(NodeKind::Alt);
        alt->kids = std::move(branches);
        return alt;
    }

    NodePtr parse_branch(Flags& f, int depth) {
        auto cat = mk(NodeKind::Concat);
        while (err_.empty()) {
            skip_extended(f);
            if (eof() || peek() == '|' || peek() == ')') break;
            bool quantifiable = true;
            NodePtr atom = parse_atom(f, depth, quantifiable);
            if (!err_.empty()) return nullptr;
            if (!atom) continue;  // option setting / comment
            skip_extended(f);
            atom = parse_quantifiers(std::move(atom), quantifiable, f);
            if (!err_.empty()) return nullptr;
            cat->kids.push_back(std::move(atom));
        }
        if (!err_.empty()) return nullptr;
        if (cat->kids.empty()) return mk(NodeKind::Empty);
        if (cat->kids.size() == 1) return std::move(cat->kids[0]);
        return cat;
    }

    // {n} {n,} {n,m}; anything else after '{' is a literal brace (PCRE)
    bool try_braces(int& mn, int& mx) {
        size_t j = i_ + 1;
        auto digits = [&](long& v) {
            size_t st = j; v = 0;
            while (j < s_.size() && std::isdigit((unsigned char)s_[j])) { v = v * 10 + (s_[j] - '0'); if (v > 100000) v = 100000; j++; }
            return j > st;
        };
        long a = 0, b = -1;
        if (!digits(a)) return false;
        if (j < s_.size() && s_[j] == ',') {
            j++;
            long t;
            if (digits(t)) b = t; else b = -1;
        } else {
            b = a;
        }
        if (j >= s_.size() || s_[j] != '}') return false;
        mn = (int)a; mx = (int)b;
        i_ = j + 1;
        return true;
    }

    NodePtr parse_quantifiers(NodePtr atom, bool quantifiable, const Flags& f) {
        while (!eof()) {
            unsigned char c = peek();
            int mn, mx;
            if (c == '*') { mn = 0; mx = -1; i_++; }
            else if (c == '+') { mn = 1; mx = -1; i_++; }
            else if (c == '?') { mn = 0; mx = 1; i_++; }
            else if (c == '{') { if (!try_braces(mn, mx)) break; }
            else break;
            if (!quantifiable) { fail("quantifier does not follow a repeatable item"); return nullptr; }
            if (mx >= 0 && mn > mx) { fail("numbers out of order in {} quantifier"); return nullptr; }
            if (mn > 32767 || mx > 32767) { fail("bounded repeat is too large"); return nullptr; }
            bool lazy = false;
            if (!eof() && peek() == '?') { i_++; lazy = true; }   // lazy: same language, recorded for the span program
            else if (!eof() && peek() == '+') { fail("possessive quantifiers are not supported"); return nullptr; }
            if (mx == 0) { atom = mk(NodeKind::Empty); }
            else if (!(mn == 1 && mx == 1)) {
                auto rep = mk(NodeKind::Repeat);
                rep->min = mn; rep->max = mx;
                rep->lazy = lazy;
                rep->kids.push_back(std::move(atom));
                atom = std::move(rep);
            }
            skip_extended(f);
            // a further quantifier applies to the repeated item (e.g. a{2}{3}); PCRE allows it
        }
        return atom;
    }

    NodePtr literal(unsigned char c, const Flags& f) {
        ByteSet s = ByteSet::of(c);
        if (f.caseless) s = fold_case(s);
        return mk_set(s);
    }

    bool parse_hex(int maxdigits, unsigned& v, int& nd) {
        v = 0; nd = 0;
        while (nd < maxdigits && !eof() && std::isxdigit(peek())) {
            unsigned char c = peek();
            v = v * 16 + (std::isdigit(c) ? c - '0' : (std::tolower(c) - 'a' + 10));
            nd++; i_++;
            if (v > 0xFFFF) return false;
        }
        return true;
    }

    // Parses the escape after '\\' (i_ points at the char after the backslash).
    // Outcomes: a byte set (class escape or literal), or an assertion (outside classes only).
    enum class EscKind { Set, Assert, EndOrFinalNewline, QuoteStart, Nothing, Error };
    EscKind parse_escape(bool in_class, const Flags& f, ByteSet& out, AssertKind& ak, bool& is_single) {
        is_single = false;
        if (eof()) { fail("\\ at end of pattern"); return EscKind::Error; }
        unsigned char c = peek();
        i_++;
        switch (c) {
            case 'd': out = set_digit(); return EscKind::Set;
            case 'D': out = ~set_digit(); return EscKind::Set;
            case 'w': out = set_word(); return EscKind::Set;
            case 'W': out = ~set_word(); return EscKind::Set;
            case 's': out = set_space(); return EscKind::Set;
            case 'S': out = ~set_space(); return EscKind::Set;
            case 'h': out = set_hspace(); return EscKind::Set;
            case 'H': out = ~set_hspace(); return EscKind::Set;
            case 'V': out = ~set_vspace(); return EscKind::Set;
            case 'v': out = set_vspace(); return EscKind::Set;
            case 'N': {
                if (in_class) { fail("\\N is not supported in a class"); return EscKind::Error; }
                // \N{U+hh..} names a code point (UTF mode only); any other '{' after \N must open a quantifier
                int mn, mx;
                const size_t at = i_;
                if (!eof() && peek() == '{' && !try_braces(mn, mx)) { fail("\\N{ is not a quantifier (\\N{U+..} needs UTF mode)"); return EscKind::Error; }
                i_ = at;
                out = ~ByteSet::of('\n'); return EscKind::Set;
            }
            case 'n': out = ByteSet::of('\n'); is_single = true; return EscKind::Set;
            case 'r': out = ByteSet::of('\r'); is_single = true; return EscKind::Set;
            case 't': out = ByteSet::of('\t'); is_single = true; return EscKind::Set;
            case 'f': out = ByteSet::of('\f'); is_single = true; return EscKind::Set;
            case 'a': out = ByteSet::of(7); is_single = true; return EscKind::Set;
            case 'e': out = ByteSet::of(27); is_single = true; return EscKind::Set;
            case 'E': return EscKind::Nothing;  // stray \E is ignored
            case 'Q': return EscKind::QuoteStart;
            case 'c': {
                if (eof()) { fail("\\c at end of pattern"); return EscKind::Error; }
                unsigned char x = peek(); i_++;
                if (x >= 'a' && x <= 'z') x -= 32;
                if (x < 32 || x > 126) { fail("\\c must be followed by a printable ASCII character"); return EscKind::Error; }
                out = ByteSet::of(x ^ 0x40); is_single = true; return EscKind::Set;
            }
            case 'x': {
                unsigned v; int nd;
                if (!eof() && peek() == '{') {
                    i_++;
                    if (!parse_hex(8, v, nd) || nd == 0 || eof() || peek() != '}') { fail("bad \\x{} escape"); return EscKind::Error; }
                    i_++;
                } else {
                    parse_hex(2, v, nd);
                }
                if (v > 255) { fail("character value in \\x{} escape is too large (no UTF-8 mode)"); return EscKind::Error; }
                out = ByteSet::of(v); is_single = true; return EscKind::Set;
            }
            case 'o': {
                if (eof() || peek() != '{') { fail("missing { after \\o"); return EscKind::Error; }
                i_++;
                unsigned v = 0; int nd = 0;
                while (!eof() && peek() >= '0' && peek() <= '7') { v = v * 8 + (peek() - '0'); nd++; i_++; if (v > 0xFFFF) break; }
                if (nd == 0 || eof() || peek() != '}' || v > 255) { fail("bad \\o{} escape"); return EscKind::Error; }
                i_++;
                out = ByteSet::of(v); is_single = true; return EscKind::Set;
            }
            case '0': {
                unsigned v = 0; int nd = 0;
                while (nd < 2 && !eof() && peek() >= '0' && peek() <= '7') { v = v * 8 + (peek() - '0'); nd++; i_++; }
                out = ByteSet::of(v & 255); is_single = true; return EscKind::Set;
            }
            default: break;
        }
        if (c >= '1' && c <= '9') {
            if (!in_class) { fail("back-references are not supported"); return EscKind::Error; }
            if (c >= '8') { out = ByteSet::of(c); is_single = true; return EscKind::Set; }   // [\8]: the digit itself
            unsigned v = c - '0'; int nd = 1;
            while (nd < 3 && !eof() && peek() >= '0' && peek() <= '7') { v = v * 8 + (peek() - '0'); nd++; i_++; }
            out = ByteSet::of(v & 255); is_single = true; return EscKind::Set;
        }
        if (in_class) {
            if (c == 'b') { out = ByteSet::of(8); is_single = true; return EscKind::Set; }
        } else {
            switch (c) {
                case 'b': ak = AssertKind::WordBoundary; return EscKind::Assert;
                case 'B': ak = AssertKind::NotWordBoundary; return EscKind::Assert;
                case 'A': ak = AssertKind::BeginBuffer; return EscKind::Assert;
                case 'z': ak = AssertKind::EndBuffer; return EscKind::Assert;
                case 'Z': return EscKind::EndOrFinalNewline;
                default: break;
            }
        }
        if (c == 'p' || c == 'P') { fail("unicode properties are not supported without UTF-8 mode"); return EscKind::Error; }
        if (c == 'C' || c == 'R' || c == 'K' || c == 'X' || c == 'G' || c == 'g' || c == 'k') { fail("unsupported escape sequence"); return EscKind::Error; }
        if (std::isalnum(c)) { fail("unrecognized character follows \\"); return EscKind::Error; }
        (void)f;
        out = ByteSet::of(c); is_single = true; return EscKind::Set;
    }

    bool posix_class(const std::string& name, ByteSet& s) {
        if (name == "alpha") { s.set_range('a', 'z'); s.set_range('A', 'Z'); }
        else if (name == "digit") s.set_range('0', '9');
        else if (name == "alnum") { s.set_range('a', 'z'); s.set_range('A', 'Z'); s.set_range('0', '9'); }
        else if (name == "upper") s.set_range('A', 'Z');
        else if (name == "lower") s.set_range('a', 'z');
        else if (name == "space") { s.set_range(9, 13); s.set(32); }
        else if (name == "blank") { s.set(9); s.set(32); }
        else if (name == "punct") { for (unsigned b = 33; b < 127; b++) if (!std::isalnum(b)) s.set(b); }
        else if (name == "print") s.set_range(32, 126);
        else if (name == "graph") s.set_range(33, 126);
        else if (name == "cntrl") { s.set_range(0, 31); s.set(127); }
        else if (name == "xdigit") { s.set_range('0', '9'); s.set_range('a', 'f'); s.set_range('A', 'F'); }
        else if (name == "word") s = set_word();
        else if (name == "ascii") s.set_range(0, 127);
        else return false;
        return true;
    }

    // '-' at i_ that is not the last character of the class
    bool dash_starts_range() const { return !eof() && peek() == '-' && i_ + 1 < s_.size() && peek(1) != ']'; }

    NodePtr parse_class(const Flags& f) {
        // i_ is just past '['
        bool negate = false;
        if (!eof() && peek() == '^') { negate = true; i_++; }
        ByteSet acc;
        bool first = true;
        bool have_prev = false; unsigned prev = 0;  // last single byte, candidate range start
        while (true) {
            if (eof()) { fail("missing terminating ] for character class"); return nullptr; }
            unsigned char c = peek();
            if (c == ']' && !first) { i_++; break; }
            first = false;
            ByteSet item; bool single = false; unsigned single_val = 0;
            if (c == '[' && (peek(1) == ':' || peek(1) == '.' || peek(1) == '=')) {
                unsigned char kind = peek(1);
                size_t close = s_.find(std::string(1, (char)kind) + "]", i_ + 2);
                if (close != std::string::npos) {
                    if (kind != ':') { fail("POSIX collating elements are not supported"); return nullptr; }
                    std::string name = s_.substr(i_ + 2, close - (i_ + 2));
                    bool neg = false;
                    if (!name.empty() && name[0] == '^') { neg = true; name = name.substr(1); }
                    ByteSet ps;
                    if (!posix_class(name, ps)) { fail("unknown POSIX class name"); return nullptr; }
                    if (neg) ps = ~ps;
                    item = ps;
                    i_ = close + 2;
                    acc |= item; have_prev = false;
                    if (dash_starts_range()) { fail("invalid range in character class"); return nullptr; }
                    continue;
                }
                // no closing :] -> literal '['
                i_++; single = true; single_val = '[';
            } else if (c == '\\') {
                i_++;
                AssertKind ak; bool is_single = false; ByteSet es;
                EscKind k = parse_escape(true, f, es, ak, is_single);
                if (k == EscKind::Error) return nullptr;
                if (k == EscKind::Nothing) continue;
                if (k == EscKind::QuoteStart) {
                    // \Q..\E inside a class: literal bytes
                    while (!eof() && !(peek() == '\\' && peek(1) == 'E')) { acc.set(peek()); i_++; }
                    if (!eof()) i_ += 2;
                    have_prev = false;
                    continue;
                }
                if (k != EscKind::Set) { fail("invalid escape in class"); return nullptr; }
                if (is_single) { single = true; for (unsigned b = 0; b < 256; b++) if (es.test(b)) single_val = b; }
                else {
                    // a class escape (\d, \h, ...) can bound no range: PCRE2 faults "[\d-z]" where Perl only warns
                    if (dash_starts_range()) { fail("invalid range in character class"); return nullptr; }
                    acc |= es; have_prev = false; continue;
                }
            } else {
                i_++; single = true; single_val = c;
            }
            // single byte: maybe the start or the end of a range
            if (single) {
                if (have_prev && false) {}
                // range "a-z": look ahead for '-' followed by a non-']' item
                if (!eof() && peek() == '-' && peek(1) != ']' && i_ + 1 < s_.size()) {
                    size_t save = i_;
                    i_++;  // past '-'
                    unsigned hi = 0; bool hi_ok = false;
                    unsigned char d = peek();
                    if (d == '\\') {
                        i_++;
                        AssertKind ak; bool is_single = false; ByteSet es;
                        EscKind k = parse_escape(true, f, es, ak, is_single);
                        if (k == EscKind::Error) return nullptr;
                        if (k == EscKind::Set && is_single) { for (unsigned b = 0; b < 256; b++) if (es.test(b)) hi = b; hi_ok = true; }
                        else if (k == EscKind::Set) { fail("invalid range in character class"); return nullptr; }   // "a-\d"
                        else { i_ = save; }   // "a-\Q..": '-' is literal; re-parse from '-'
                    } else if (d == '[' && peek(1) == ':' && s_.find(":]", i_ + 2) != std::string::npos) {
                        fail("invalid range in character class"); return nullptr;   // "a-[:digit:]"
                    } else {
                        i_++; hi = d; hi_ok = true;
                    }
                    if (hi_ok) {
                        if (hi < single_val) { fail("range out of order in character class"); return nullptr; }
                        acc.set_range(single_val, hi);
                        have_prev = false;
                        continue;
                    }
                }
                acc.set(single_val);
                prev = single_val; have_prev = true;
                (void)prev;
            }
        }
        if (f.caseless) acc = fold_case(acc);
        if (negate) acc = ~acc;
        return mk_set(acc);
    }

    // returns nullptr with empty err_ for constructs that produce no node (option settings, comments)
    NodePtr parse_atom(Flags& f, int depth, bool& quantifiable) {
        unsigned char c = peek();
        quantifiable = true;
        switch (c) {
            case '(': return parse_group(f, depth, quantifiable);
            case '[': i_++; return parse_class(f);
            case '.': {
                i_++;
                return mk_set(f.dotall ? ByteSet::all() : ~ByteSet::of('\n'));
            }
            case '^': i_++; quantifiable = false; return mk_assert(f.multiline ? AssertKind::BeginLine : AssertKind::BeginBuffer);
            case '$': {
                i_++; quantifiable = false;
                if (f.multiline) return mk_assert(AssertKind::EndLine);
                return mk_end_or_final_newline();
            }
            case '*': case '+': case '?': fail("quantifier does not follow a repeatable item"); return nullptr;
            case '\\': {
                i_++;
                ByteSet es; AssertKind ak; bool is_single = false;
                EscKind k = parse_escape(false, f, es, ak, is_single);
                switch (k) {
                    case EscKind::Error: return nullptr;
                    case EscKind::Nothing: return nullptr;
                    case EscKind::Assert: quantifiable = false; return mk_assert(ak);
                    case EscKind::EndOrFinalNewline: quantifiable = false; return mk_end_or_final_newline();
                    case EscKind::QuoteStart: {
                        // \Q...\E : each byte is a literal atom; a quantifier after \E applies to the last byte
                        auto cat = mk(NodeKind::Concat);
                        NodePtr last;
                        while (!eof() && !(peek() == '\\' && peek(1) == 'E')) {
                            if (last) cat->kids.push_back(std::move(last));
                            last = literal(peek(), f);
                            i_++;
                        }
                        if (!eof()) i_ += 2;
                        if (!last) return nullptr;
                        // apply a following quantifier to the last literal only
                        last = parse_quantifiers(std::move(last), true, f);
                        if (!err_.empty()) return nullptr;
                        cat->kids.push_back(std::move(last));
                        quantifiable = true;
                        if (cat->kids.size() == 1) return std::move(cat->kids[0]);
                        // further quantifiers directly after would be rejected by PCRE as well ("a{2}{3}" is legal
                        // but acts on the repeat); harmless here
                        return cat;
                    }
                    case EscKind::Set:
                        if (is_single && f.caseless) es = fold_case(es);
                        return mk_set(es);
                }
                return nullptr;
            }
            default:
                i_++;
                return literal(c, f);
        }
    }

    NodePtr parse_group(Flags& f, int depth, bool& quantifiable) {
        // i_ at '('
        i_++;
        Flags inner = f;
        if (!eof() && peek() == '*') { fail("backtracking control verbs are not supported"); return nullptr; }
        if (!eof() && peek() == '?') {
            i_++;
            if (eof()) { fail("unrecognized character after (?"); return nullptr; }
            unsigned char c = peek();
            if (c == '#') {  // comment
                while (!eof() && peek() != ')') i_++;
                if (eof()) { fail("missing ) after (?# comment"); return nullptr; }
                i_++;
                quantifiable = false;
                return nullptr;
            }
            if (c == ':') { i_++; }
            else if (c == '=' || c == '!') { fail("look-ahead assertions are not supported"); return nullptr; }
            else if (c == '>') { fail("atomic groups are not supported"); return nullptr; }
            else if (c == '(') { fail("conditional groups are not supported"); return nullptr; }
            else if (c == '|') { fail("branch reset groups are not supported"); return nullptr; }
            else if (c == 'R' || c == '&' || c == '+' || std::isdigit(c)) { fail("recursion / subroutine calls are not supported"); return nullptr; }
            else if (c == 'C') { fail("callouts are not supported"); return nullptr; }
            else if (c == '<' || c == 'P' || c == '\'') {
                unsigned char term = '>';
                if (c == 'P') {
                    i_++;
                    if (eof()) { fail("unrecognized character after (?P"); return nullptr; }
                    if (peek() == '=' || peek() == '>') { fail("named back-references / subroutines are not supported"); return nullptr; }
                    if (peek() != '<') { fail("unrecognized character after (?P"); return nullptr; }
                    i_++;
                } else if (c == '<') {
                    if (peek(1) == '=' || peek(1) == '!') { fail("look-behind assertions are not supported"); return nullptr; }
                    i_++;
                } else { i_++; term = '\''; }
                size_t st = i_;
                while (!eof() && (std::isalnum(peek()) || peek() == '_')) i_++;
                if (i_ == st || eof() || peek() != term || std::isdigit((unsigned char)s_[st])) { fail("bad group name"); return nullptr; }
                i_++;
            } else {
                // option letters: (?imsxUJ-imsx) or (?imsx-imsx:...)
                bool on = true; bool any = false;
                while (!eof() && peek() != ')' && peek() != ':') {
                    unsigned char o = peek();
                    if (o == '-') { if (!on) { fail("bad option setting"); return nullptr; } on = false; }
                    else if (o == 'i') inner.caseless = on;
                    else if (o == 's') inner.dotall = on;
                    else if (o == 'm') inner.multiline = on;
                    else if (o == 'x') inner.extended = on;
                    else if (o == 'U' || o == 'J') {}
                    else if (o == '^') { inner.caseless = inner.dotall = inner.multiline = inner.extended = false; }
                    else { fail("unrecognized character after (? or (?-"); return nullptr; }
                    any = true; i_++;
                }
                (void)any;
                if (eof()) { fail("missing )"); return nullptr; }
                if (peek() == ')') {
                    i_++;
                    f = inner;  // applies to the rest of the enclosing group
                    quantifiable = false;
                    return nullptr;
                }
                i_++;  // ':'
            }
        }
        NodePtr body = parse_alternation(inner, depth + 1);
        if (!err_.empty()) return nullptr;
        if (eof() || peek() != ')') { fail("missing )"); return nullptr; }
        i_++;
        quantifiable = true;
        return body;
    }
};

}  // namespace

ParseResult parse_regex(const std::string& pattern, unsigned flags) {
    Parser p(pattern, flags);
    return p.run();
}

bool matches_empty_buffer(const Node& n) {
    switch (n.kind) {
        case NodeKind::Empty: return true;
        case NodeKind::Set: return false;
        case NodeKind::Assert:
            // structural test (a start->accept path that consumes nothing), as in Hyperscan: assertions do not count
            return true;
        case NodeKind::Concat:
            for (auto& k : n.kids) if (!matches_empty_buffer(*k)) return false;
            return true;
        case NodeKind::Alt:
            for (auto& k : n.kids) if (matches_empty_buffer(*k)) return true;
            return false;
        case NodeKind::Repeat:
            return n.min == 0 || matches_empty_buffer(*n.kids[0]);
    }
    return false;
}

}  // namespace gpugrep
