// AST -> Thompson NFA -> DFA (subset construction, Moore minimisation, byte-class merging).  See automata.hpp.
#include "automata.hpp"

#include <algorithm>
#include <map>
#include <unordered_map>

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// Thompson construction, continuation style: emit(node, next) returns the entry instruction of `node`
// followed by `next`.  Bounded repeats are unrolled by re-emitting the child.
// ------------------------------------------------------------------------------------------------------------
namespace {

struct NfaBuilder {
    Nfa& nfa;
    size_t max_insts;
    bool lazy = false;   // honour Node::lazy (span programs only)
    bool overflow = false;
    std::map<ByteSet, int> set_ids;

    int add(NfaInst::Op op, int x, int y, int arg) {
        if (nfa.prog.size() >= max_insts) { overflow = true; return 0; }
        NfaInst in; in.op = op; in.x = x; in.y = y; in.arg = arg;
        nfa.prog.push_back(in);
        return (int)nfa.prog.size() - 1;
    }
    int set_id(const ByteSet& s) {
        auto it = set_ids.find(s);
        if (it != set_ids.end()) return it->second;
        int id = (int)nfa.sets.size();
        nfa.sets.push_back(s);
        set_ids.emplace(s, id);
        return id;
    }
    int emit(const Node& n, int next) {
        if (overflow) return 0;
        switch (n.kind) {
            case NodeKind::Empty: return next;
            case NodeKind::Set: return add(NfaInst::Byte, next, -1, set_id(n.set));
            case NodeKind::Assert: {
                switch (n.assert_kind) {
                    case AssertKind::BeginBuffer: case AssertKind::BeginLine: nfa.uses_line_ctx = true; break;
                    case AssertKind::WordBoundary: case AssertKind::NotWordBoundary: nfa.uses_word_ctx = true; nfa.uses_lookahead = true; break;
                    case AssertKind::EndBuffer: case AssertKind::EndLine: nfa.uses_lookahead = true; break;
                }
                return add(NfaInst::Assert, next, -1, (int)n.assert_kind);
            }
            case NodeKind::Concat: {
                int cur = next;
                for (size_t k = n.kids.size(); k-- > 0;) cur = emit(*n.kids[k], cur);
                return cur;
            }
            case NodeKind::Alt: {
                std::vector<int> entry;
                for (auto& k : n.kids) entry.push_back(emit(*k, next));
                int cur = entry.back();
                for (size_t k = entry.size() - 1; k-- > 0;) cur = add(NfaInst::Split, entry[k], cur, 0);
                return cur;
            }
            case NodeKind::Repeat: {
                const Node& c = *n.kids[0];
                int cur;
                const bool swap = lazy && n.lazy;   // prefer leaving the repeat
                if (n.max < 0) {
                    int loop = add(NfaInst::Split, -1, -1, 0);
                    int body = emit(c, loop);
                    if (overflow) return 0;
                    nfa.prog[loop].x = swap ? next : body;
                    nfa.prog[loop].y = swap ? body : next;
                    cur = (n.min == 0) ? loop : body;
                    for (int k = 1; k < n.min; k++) cur = emit(c, cur);
                } else {
                    cur = next;
                    for (int k = 0; k < n.max - n.min; k++) {
                        int b = emit(c, cur);
                        cur = swap ? add(NfaInst::Split, next, b, 0) : add(NfaInst::Split, b, next, 0);
                        if (overflow) return 0;
                    }
                    for (int k = 0; k < n.min; k++) cur = emit(c, cur);
                }
                return cur;
            }
        }
        return next;
    }
};

}  // namespace

bool nfa_add_pattern(Nfa& nfa, const Node& ast, int index, size_t max_insts, bool lazy) {
    NfaBuilder b{nfa, max_insts, lazy};
    for (size_t i = 0; i < nfa.sets.size(); i++) b.set_ids.emplace(nfa.sets[i], (int)i);
    size_t mark_prog = nfa.prog.size(), mark_sets = nfa.sets.size();
    int m = b.add(NfaInst::Match, -1, -1, index);
    int start = b.emit(ast, m);
    if (b.overflow) {
        nfa.prog.resize(mark_prog);
        nfa.sets.resize(mark_sets);
        return false;
    }
    nfa.starts.push_back(start);
    return true;
}

// ------------------------------------------------------------------------------------------------------------
// Subset construction
// ------------------------------------------------------------------------------------------------------------
namespace {

enum Look : int { LookWord = 0, LookOther = 1, LookNewline = 2, LookEod = 3 };

struct Ctx {
    bool at_start, prev_nl, prev_word;
};

struct VecHash {
    size_t operator()(const std::vector<int>& v) const {
        uint64_t h = 1469598103934665603ull;
        for (int x : v) { h ^= (uint32_t)x; h *= 1099511628211ull; h ^= h >> 29; }
        return (size_t)h;
    }
};

struct Determinizer {
    const Nfa& nfa;
    const DfaBuildOptions& opt;
    int ncls = 0;
    uint8_t byte_class[256];
    std::vector<int> class_look;                   // Look per class
    std::vector<std::vector<uint64_t>> set_classes;  // per set: bitset over classes
    // closure scratch
    std::vector<uint32_t> seen_strong, seen_weak;
    uint32_t stamp = 0;
    std::vector<int> stack;

    Determinizer(const Nfa& n, const DfaBuildOptions& o) : nfa(n), opt(o) {}

    void build_classes() {
        // partition refinement of 0..255 by every byte set in use (+ newline / word sets when context matters)
        std::vector<int> cls(256, 0);
        int n = 1;
        auto refine = [&](const ByteSet& s) {
            std::map<std::pair<int, bool>, int> remap;
            std::vector<int> out(256);
            int m = 0;
            for (int b = 0; b < 256; b++) {
                auto key = std::make_pair(cls[b], s.test(b));
                auto it = remap.find(key);
                if (it == remap.end()) it = remap.emplace(key, m++).first;
                out[b] = it->second;
            }
            cls.swap(out);
            n = m;
        };
        for (auto& s : nfa.sets) refine(s);
        if (nfa.uses_line_ctx || nfa.uses_lookahead) refine(ByteSet::of('\n'));
        if (nfa.uses_word_ctx) { ByteSet w; for (unsigned b = 0; b < 256; b++) if (is_word_byte(b)) w.set(b); refine(w); }
        ncls = n;
        for (int b = 0; b < 256; b++) byte_class[b] = (uint8_t)cls[b];
        class_look.assign(ncls, LookOther);
        std::vector<int> rep(ncls, -1);
        for (int b = 0; b < 256; b++) if (rep[cls[b]] < 0) rep[cls[b]] = b;
        for (int c = 0; c < ncls; c++) {
            int b = rep[c];
            if (b == '\n' && (nfa.uses_line_ctx || nfa.uses_lookahead)) class_look[c] = LookNewline;
            else if (nfa.uses_word_ctx && is_word_byte(b)) class_look[c] = LookWord;
        }
        size_t words = (ncls + 63) / 64;
        set_classes.assign(nfa.sets.size(), std::vector<uint64_t>(words, 0));
        for (size_t s = 0; s < nfa.sets.size(); s++)
            for (int c = 0; c < ncls; c++)
                if (nfa.sets[s].test(rep[c])) set_classes[s][c >> 6] |= 1ull << (c & 63);
    }

    bool assert_holds(AssertKind k, const Ctx& ctx, int look) const {
        switch (k) {
            case AssertKind::BeginBuffer: return ctx.at_start;
            // Hyperscan: a multiline ^ holds at offset 0 and after ANY newline, also the one that ends the block (a streaming
            // engine cannot tell that a newline is the last byte).  PCRE's default excludes that position; the oracle
            // compiles with PCRE2_ALT_CIRCUMFLEX to agree (SURVEY.md Appendix A; DESIGN.md section 2).
            case AssertKind::BeginLine: return ctx.at_start || ctx.prev_nl;
            case AssertKind::EndBuffer: return look == LookEod;
            case AssertKind::EndLine: return look == LookEod || look == LookNewline;
            case AssertKind::WordBoundary: return ctx.prev_word != (look == LookWord);
            case AssertKind::NotWordBoundary: return ctx.prev_word == (look == LookWord);
        }
        return false;
    }

    // Epsilon closure.  `strong` items descend from consumed bytes (their Match counts); `weak` items are the
    // fresh ".*" restarts whose zero-width matches must not be reported.
    void closure(const std::vector<int>& kernel, const Ctx& ctx, int look, std::vector<int>& bytes, std::vector<int>& matched,
                 bool with_kernel = true, bool with_starts = true) {
        bytes.clear(); matched.clear();
        stamp++;
        if (stamp == 0) { std::fill(seen_strong.begin(), seen_strong.end(), 0); std::fill(seen_weak.begin(), seen_weak.end(), 0); stamp = 1; }
        auto run = [&](int root, bool strong) {
            stack.clear();
            stack.push_back(root);
            while (!stack.empty()) {
                int pc = stack.back(); stack.pop_back();
                if (seen_strong[pc] == stamp) continue;
                if (!strong && seen_weak[pc] == stamp) continue;
                if (strong) seen_strong[pc] = stamp; else seen_weak[pc] = stamp;
                const NfaInst& in = nfa.prog[pc];
                switch (in.op) {
                    case NfaInst::Byte: bytes.push_back(pc); break;
                    case NfaInst::Split: stack.push_back(in.y); stack.push_back(in.x); break;
                    case NfaInst::Assert: if (assert_holds((AssertKind)in.arg, ctx, look)) stack.push_back(in.x); break;
                    case NfaInst::Match: if (strong) matched.push_back(in.arg); break;
                }
            }
        };
        if (with_kernel) for (int pc : kernel) run(pc, true);
        if (with_starts) for (int pc : nfa.starts) run(pc, false);
        std::sort(bytes.begin(), bytes.end());
        bytes.erase(std::unique(bytes.begin(), bytes.end()), bytes.end());
        std::sort(matched.begin(), matched.end());
        matched.erase(std::unique(matched.begin(), matched.end()), matched.end());
    }
};

}  // namespace

static void minimise(Dfa& d, const std::vector<char>& idle);
static std::vector<uint8_t> nfa_longest_paths(const Nfa& nfa);

bool build_nfa_tables(const Nfa& nfa, NfaTables& out) {
    DfaBuildOptions opt;
    Determinizer det(nfa, opt);
    det.seen_strong.assign(nfa.prog.size(), 0);
    det.seen_weak.assign(nfa.prog.size(), 0);
    std::vector<int> pos_of(nfa.prog.size(), -1);
    std::vector<int> pcs;
    for (size_t pc = 0; pc < nfa.prog.size(); pc++)
        if (nfa.prog[pc].op == NfaInst::Byte) { pos_of[pc] = (int)pcs.size(); pcs.push_back((int)pc); }
    const int P = (int)pcs.size();
    if (P == 0 || P > 128 * 32) return false;
    const int W = (P + 31) / 32;
    out = NfaTables();
    out.positions = P;
    out.words = W;
    out.reach.assign((size_t)256 * W, 0);
    out.follow.assign((size_t)P * 12 * W, 0);
    out.follow_match.assign((size_t)P * 12, 0);
    out.restart.assign((size_t)16 * W, 0);
    for (int p = 0; p < P; p++) {
        const ByteSet& set = nfa.sets[nfa.prog[pcs[p]].arg];
        for (int b = 0; b < 256; b++) if (set.test(b)) out.reach[(size_t)b * W + (p >> 5)] |= 1u << (p & 31);
    }
    std::vector<int> bytes, matched;
    for (int p = 0; p < P; p++) {
        std::vector<int> kernel = {nfa.prog[pcs[p]].x};
        for (int kind = 0; kind < 3; kind++) {          // the byte just consumed: word / other / newline
            Ctx ctx{false, kind == 2, kind == 0};
            for (int look = 0; look < 4; look++) {      // Look enum order: word, other, newline, end of data
                det.closure(kernel, ctx, look, bytes, matched, true, false);
                size_t combo = (size_t)kind * 4 + look;
                uint32_t* f = &out.follow[((size_t)p * 12 + combo) * W];
                for (int pc : bytes) { int q = pos_of[pc]; f[q >> 5] |= 1u << (q & 31); }
                out.follow_match[(size_t)p * 12 + combo] = matched.empty() ? 0u : 1u;
            }
        }
    }
    for (int prev = 0; prev < 4; prev++) {              // word / other / newline / start of block
        Ctx ctx{prev == 3, prev == 2, prev == 0};
        for (int look = 0; look < 4; look++) {
            det.closure({}, ctx, look, bytes, matched, false, true);
            uint32_t* r = &out.restart[((size_t)prev * 4 + look) * W];
            for (int pc : bytes) { int q = pos_of[pc]; r[q >> 5] |= 1u << (q & 31); }
        }
    }
    return true;
}

bool build_dfa(const Nfa& nfa, const DfaBuildOptions& opt, Dfa& out) {
    Determinizer det(nfa, opt);
    det.build_classes();
    det.seen_strong.assign(nfa.prog.size(), 0);
    det.seen_weak.assign(nfa.prog.size(), 0);
    const int ncls = det.ncls;
    const int stride = ncls + 1;

    // state key: kernel items..., then ctx bits, then accept-set id.  Terminal (post end-of-data) states use a
    // kernel of {-1}.
    std::unordered_map<std::vector<int>, int, VecHash> ids;
    std::vector<std::vector<int>> kernels;
    std::vector<Ctx> ctxs;
    std::vector<uint32_t> accept_of;
    std::map<std::vector<int>, int> accept_ids;
    std::vector<std::vector<int>> accept_sets;
    accept_sets.push_back({});
    accept_ids[{}] = 0;
    std::vector<uint32_t> trans;
    int sink_state = -1;  // simple mode only

    auto accept_id = [&](const std::vector<int>& m) {
        auto it = accept_ids.find(m);
        if (it != accept_ids.end()) return it->second;
        int id = (int)accept_sets.size();
        accept_sets.push_back(m);
        accept_ids.emplace(m, id);
        return id;
    };
    auto intern = [&](const std::vector<int>& kernel, const Ctx& ctx, int acc) -> int {
        std::vector<int> key = kernel;
        key.push_back(-2);
        key.push_back((ctx.at_start ? 1 : 0) | (ctx.prev_nl ? 2 : 0) | (ctx.prev_word ? 4 : 0));
        key.push_back(acc);
        auto it = ids.find(key);
        if (it != ids.end()) return it->second;
        int id = (int)kernels.size();
        ids.emplace(std::move(key), id);
        kernels.push_back(kernel);
        ctxs.push_back(ctx);
        accept_of.push_back((uint32_t)acc);
        trans.resize((size_t)(id + 1) * stride, 0);
        return id;
    };

    Ctx start_ctx{true, false, false};
    if (!nfa.uses_line_ctx) start_ctx.at_start = false;  // nobody can observe it: fewer states
    intern({}, start_ctx, 0);
    const int mid_other = intern({}, Ctx{false, false, false}, 0);
    const int mid_word = intern({}, Ctx{false, false, nfa.uses_word_ctx}, 0);
    if (opt.simple) {
        sink_state = intern({-1, -1}, Ctx{false, false, false}, accept_id({0}));
    }

    std::vector<int> bytes, matched, next_kernel;
    std::vector<int> look_bytes[4], look_matched[4];
    // per (context, look-ahead): for every byte class, the kernel items contributed by matches that START here
    std::map<int, std::vector<std::vector<int>>> start_cache;
    auto start_targets = [&](int ctx_bits, const Ctx& ctx, int slot, int look) -> const std::vector<std::vector<int>>& {
        int key = ctx_bits * 4 + slot;
        auto it = start_cache.find(key);
        if (it != start_cache.end()) return it->second;
        std::vector<int> sb, sm;
        det.closure({}, ctx, look, sb, sm, false, true);
        std::vector<std::vector<int>> per_class(ncls);
        for (int c = 0; c < ncls; c++) {
            for (int pc : sb) {
                const NfaInst& in = nfa.prog[pc];
                if ((det.set_classes[in.arg][c >> 6] >> (c & 63)) & 1) per_class[c].push_back(in.x);
            }
            std::sort(per_class[c].begin(), per_class[c].end());
            per_class[c].erase(std::unique(per_class[c].begin(), per_class[c].end()), per_class[c].end());
        }
        return start_cache.emplace(key, std::move(per_class)).first->second;
    };
    for (int s = 0; s < (int)kernels.size(); s++) {
        if ((size_t)kernels.size() > opt.max_states) return false;
        if (opt.simple && s == sink_state) {
            for (int c = 0; c < stride; c++) trans[(size_t)s * stride + c] = (uint32_t)sink_state;
            continue;
        }
        std::vector<int> kernel = kernels[s];
        Ctx ctx = ctxs[s];
        if (!kernel.empty() && kernel[0] == -1) {  // terminal: absorbing
            for (int c = 0; c < stride; c++) trans[(size_t)s * stride + c] = (uint32_t)s;
            continue;
        }
        bool have[4] = {false, false, false, false};
        auto get = [&](int look) {
            int slot = nfa.uses_lookahead ? look : 0;
            // only the items that descend from consumed bytes: the ".*" restarts are the same for every state with this
            // context and are merged in from start_targets() below (what keeps large pattern sets tractable)
            if (!have[slot]) { det.closure(kernel, ctx, look, look_bytes[slot], look_matched[slot], true, false); have[slot] = true; }
            return slot;
        };
        const int ctx_bits = (ctx.at_start ? 1 : 0) | (ctx.prev_nl ? 2 : 0) | (ctx.prev_word ? 4 : 0);
        for (int c = 0; c < ncls; c++) {
            int look = det.class_look[c];
            int slot = get(look);
            const std::vector<int>& m = look_matched[slot];
            int target;
            if (opt.simple && !m.empty()) {
                target = sink_state;
            } else {
                next_kernel.clear();
                for (int pc : look_bytes[slot]) {
                    const NfaInst& in = nfa.prog[pc];
                    if ((det.set_classes[in.arg][c >> 6] >> (c & 63)) & 1) next_kernel.push_back(in.x);
                }
                const std::vector<int>& fresh = start_targets(ctx_bits, ctx, nfa.uses_lookahead ? look : 0, look)[c];
                next_kernel.insert(next_kernel.end(), fresh.begin(), fresh.end());
                std::sort(next_kernel.begin(), next_kernel.end());
                next_kernel.erase(std::unique(next_kernel.begin(), next_kernel.end()), next_kernel.end());
                Ctx nctx{false, nfa.uses_line_ctx && look == LookNewline, nfa.uses_word_ctx && look == LookWord};
                target = intern(next_kernel, nctx, accept_id(m));
            }
            trans[(size_t)s * stride + c] = (uint32_t)target;
        }
        {   // end-of-data column
            int slot = get(LookEod);
            if (!nfa.uses_lookahead) {
                // closure is look-independent; matches found are the same set
            }
            const std::vector<int>& m = look_matched[slot];
            int target;
            if (opt.simple && !m.empty()) target = sink_state;
            else target = intern({-1}, Ctx{false, false, false}, accept_id(m));
            trans[(size_t)s * stride + ncls] = (uint32_t)target;
        }
    }

    out = Dfa();
    std::memcpy(out.byte_class, det.byte_class, 256);
    out.num_classes = ncls;
    out.stride = stride;
    out.trans = std::move(trans);
    out.num_states = (int)kernels.size();
    out.accept_of = std::move(accept_of);
    out.accept_sets = std::move(accept_sets);
    out.simple = opt.simple;
    out.sink_match = opt.simple ? sink_state : -1;
    out.entry_mid_other = mid_other;
    out.entry_mid_word = mid_word;
    // idle = empty kernel (no partial match in progress); recorded per state for minimise() to carry over
    out.idle_end = 0;
    std::vector<char> idle(kernels.size(), 0);
    for (size_t k = 0; k < kernels.size(); k++) idle[k] = kernels[k].empty() && out.accept_of[k] == 0;
    // depth: bytes consumed on the longest NFA path to any item of the kernel (terminal kernels: nothing in progress)
    const std::vector<uint8_t> longest = nfa_longest_paths(nfa);
    out.depth.assign(kernels.size(), 0);
    for (size_t k = 0; k < kernels.size(); k++)
        for (int pc : kernels[k])
            if (pc >= 0) out.depth[k] = std::max(out.depth[k], longest[(size_t)pc]);
    minimise(out, idle);
    return true;
}

// Longest path, in consumed bytes, from a pattern start to every instruction; 255 = unbounded (reachable through a loop).
static std::vector<uint8_t> nfa_longest_paths(const Nfa& nfa) {
    const size_t n = nfa.prog.size();
    std::vector<uint8_t> len(n, 0);
    std::vector<char> reached(n, 0), queued(n, 0);
    std::vector<int> work;
    for (int st : nfa.starts)
        if (st >= 0 && (size_t)st < n && !reached[(size_t)st]) { reached[(size_t)st] = 1; queued[(size_t)st] = 1; work.push_back(st); }
    // relaxation with a cap: a node on a byte-consuming loop climbs to 255 and stays there (at most 255 rises per node)
    while (!work.empty()) {
        const int pc = work.back();
        work.pop_back();
        queued[(size_t)pc] = 0;
        const NfaInst& in = nfa.prog[(size_t)pc];
        const int targets[2] = {in.op == NfaInst::Match ? -1 : in.x, in.op == NfaInst::Split ? in.y : -1};
        const int weight = in.op == NfaInst::Byte ? 1 : 0;
        for (int to : targets) {
            if (to < 0 || (size_t)to >= n) continue;
            const int cand = std::min(255, (int)len[(size_t)pc] + weight);
            if (!reached[(size_t)to] || cand > (int)len[(size_t)to]) {
                reached[(size_t)to] = 1;
                len[(size_t)to] = (uint8_t)cand;
                if (!queued[(size_t)to]) { queued[(size_t)to] = 1; work.push_back(to); }
            }
        }
    }
    return len;
}

// ------------------------------------------------------------------------------------------------------------
// Moore partition refinement + merging of identical alphabet columns + renumbering (accepting states last)
// ------------------------------------------------------------------------------------------------------------
static void minimise(Dfa& d, const std::vector<char>& idle) {
    const int n = d.num_states, stride = d.stride;
    std::vector<int> blk(n);
    {
        std::map<uint32_t, int> m;
        for (int s = 0; s < n; s++) {
            auto it = m.find(d.accept_of[s]);
            if (it == m.end()) it = m.emplace(d.accept_of[s], (int)m.size()).first;
            blk[s] = it->second;
        }
    }
    int nblk = 0;
    for (int s = 0; s < n; s++) nblk = std::max(nblk, blk[s] + 1);
    struct Key { uint64_t a, b; bool operator==(const Key& o) const { return a == o.a && b == o.b; } };
    struct KeyHash { size_t operator()(const Key& k) const { return (size_t)(k.a ^ (k.b * 0x9E3779B97F4A7C15ull)); } };
    std::vector<int> nb(n);
    while (true) {
        std::unordered_map<Key, int, KeyHash> sig;
        sig.reserve((size_t)n * 2);
        int cnt = 0;
        for (int s = 0; s < n; s++) {
            uint64_t a = 0xcbf29ce484222325ull ^ (uint64_t)blk[s], b = 0x9ae16a3b2f90404full + (uint64_t)blk[s];
            const uint32_t* row = &d.trans[(size_t)s * stride];
            for (int c = 0; c < stride; c++) {
                uint64_t v = (uint64_t)blk[row[c]] + 1;
                a = (a ^ v) * 0x100000001b3ull; a ^= a >> 32;
                b = (b + v * 0xff51afd7ed558ccdull); b = (b << 13) | (b >> 51); b *= 0xc4ceb9fe1a85ec53ull;
            }
            auto it = sig.find(Key{a, b});
            if (it == sig.end()) it = sig.emplace(Key{a, b}, cnt++).first;
            nb[s] = it->second;
        }
        if (cnt == nblk) break;
        nblk = cnt;
        blk.swap(nb);
    }
    // representative per block
    std::vector<int> rep(nblk, -1);
    for (int s = 0; s < n; s++) if (rep[blk[s]] < 0) rep[blk[s]] = s;
    // order: start block first, then other non-accepting, then accepting
    std::vector<int> order;  // new index -> block
    std::vector<int> newid(nblk, -1);
    order.push_back(blk[0]);
    newid[blk[0]] = 0;
    bool start_accepting = d.accept_of[0] != 0;
    (void)start_accepting;  // the start state never accepts (reports are delayed by one symbol)
    // a block is idle if it contains an idle state: equivalent states have the same future, so none of the block's
    // partial matches can matter
    std::vector<char> blk_idle(nblk, 0);
    for (int s = 0; s < n; s++) if (idle[s]) blk_idle[blk[s]] = 1;
    for (int b = 0; b < nblk; b++) if (newid[b] < 0 && d.accept_of[rep[b]] == 0 && blk_idle[b]) { newid[b] = (int)order.size(); order.push_back(b); }
    int idle_end = (int)order.size();
    for (int b = 0; b < nblk; b++) if (newid[b] < 0 && d.accept_of[rep[b]] == 0) { newid[b] = (int)order.size(); order.push_back(b); }
    int first_accept = (int)order.size();
    for (int b = 0; b < nblk; b++) if (newid[b] < 0) { newid[b] = (int)order.size(); order.push_back(b); }

    // merge identical columns (keep end-of-data as the last column)
    const int ncls = d.num_classes;
    std::vector<int> colmap(ncls, -1);
    std::vector<int> cols;  // new class -> old class
    for (int c = 0; c < ncls; c++) {
        for (size_t k = 0; k < cols.size() && colmap[c] < 0; k++) {
            bool same = true;
            for (int b = 0; b < nblk && same; b++) {
                const uint32_t* row = &d.trans[(size_t)rep[b] * stride];
                same = blk[row[c]] == blk[row[cols[k]]];
            }
            if (same) colmap[c] = (int)k;
        }
        if (colmap[c] < 0) { colmap[c] = (int)cols.size(); cols.push_back(c); }
    }
    const int ncls2 = (int)cols.size(), stride2 = ncls2 + 1;
    std::vector<uint32_t> t2((size_t)nblk * stride2);
    std::vector<uint32_t> acc2(nblk);
    for (int i = 0; i < nblk; i++) {
        int s = rep[order[i]];
        const uint32_t* row = &d.trans[(size_t)s * stride];
        for (int c = 0; c < ncls2; c++) t2[(size_t)i * stride2 + c] = (uint32_t)newid[blk[row[cols[c]]]];
        t2[(size_t)i * stride2 + ncls2] = (uint32_t)newid[blk[row[ncls]]];
        acc2[i] = d.accept_of[s];
    }
    for (int b = 0; b < 256; b++) d.byte_class[b] = (uint8_t)colmap[d.byte_class[b]];
    d.num_classes = ncls2;
    d.stride = stride2;
    d.trans.swap(t2);
    d.accept_of.swap(acc2);
    if (d.depth.size() == (size_t)n) {
        std::vector<uint8_t> blk_depth((size_t)nblk, 0);
        for (int st = 0; st < n; st++) blk_depth[(size_t)blk[st]] = std::max(blk_depth[(size_t)blk[st]], d.depth[(size_t)st]);
        std::vector<uint8_t> depth2((size_t)nblk, 0);
        for (int i = 0; i < nblk; i++) depth2[(size_t)i] = blk_depth[(size_t)order[i]];
        d.depth.swap(depth2);
    }
    d.num_states = nblk;
    d.first_accept = first_accept;
    if (d.sink_match >= 0) d.sink_match = newid[blk[d.sink_match]];
    d.entry_mid_other = newid[blk[d.entry_mid_other]];
    d.entry_mid_word = newid[blk[d.entry_mid_word]];
    d.idle_end = idle_end;
    d.dead = -1;
    for (int s = 0; s < nblk; s++) {
        if (d.accept_of[s] != 0) continue;
        bool self = true;
        for (int c = 0; c < stride2 && self; c++) self = d.trans[(size_t)s * stride2 + c] == (uint32_t)s;
        if (self) { d.dead = s; break; }
    }
}

}  // namespace gpugrep
