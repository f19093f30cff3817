// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with fixed strings (grep -F), inverted scans and context lines.
//
// The CPU engine of tests/mock_engine (included unchanged) finds the matched pseudo-lines of regex sets.  For a slot
// switched to fixed strings, a pseudo-line matches by the definition of include/gpugrep.h itself: its scanned block
// (leading NULs skipped, cut at the next NUL) contains one of the literals passed in, found with memmem, caseless ones on
// an ASCII-folded copy.  It reads the literals from the database's pattern cache key, not from the kept, prefix-free set,
// so that the host's pruning is checked too.  Inverted scans and context lines then select and widen the matched lines as
// tests/mock_engine_context does.  This lets `pytest -m "not gpu"` exercise the host logic of fixed-string scans (capi.cpp:
// the database, segments, limits, batching, shards, ingest; the Python layer and the CLI) without a GPU.  The kernels run
// on the GPU in libgpugrep.so (k_literal.cuh) and are checked by the `-m gpu` tests.
#include <mutex>
#include <string>
#include <unordered_map>

#define slot_collect matched_slot_collect
#include "../mock_engine/engine_cpu_mock.cpp"
#undef slot_collect

namespace gpugrep {

namespace {
struct Mode {
    bool invert = false, literal = false;
    uint32_t before = 0, after = 0;
};
std::mutex g_mode_mu;
std::unordered_map<const ScanSlot*, Mode> g_mode;   // set by the boundary on every slot it acquires

// The literals of a fixed-string database, parsed back from its cache key (literal, NUL, flags, ids; then options).
std::vector<std::pair<std::string, bool>> literals_of(const Database& db) {
    std::vector<std::pair<std::string, bool>> out;
    const std::string& k = db.key;
    size_t pos = 0;
    while (out.size() < db.literals.given) {
        const size_t nul = k.find('\0', pos);
        unsigned flags = 0;
        std::memcpy(&flags, k.data() + nul + 1, sizeof(flags));
        std::string text = k.substr(pos, nul - pos);
        const bool caseless = flags & 1u;
        if (caseless) for (char& c : text) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
        out.emplace_back(text, caseless);
        pos = nul + 1 + 2 * sizeof(unsigned);
    }
    return out;
}

bool block_has_literal(const uint8_t* p, size_t len, const std::vector<std::pair<std::string, bool>>& lits) {
    size_t a = 0;
    while (a < len && p[a] == 0) a++;
    const void* nul = std::memchr(p + a, 0, len - a);
    const size_t e = nul ? (size_t)((const uint8_t*)nul - p) : len;
    std::string raw((const char*)p + a, e - a), folded(raw);
    for (char& c : folded) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
    for (const auto& l : lits) {
        const std::string& hay = l.second ? folded : raw;
        if (memmem(hay.data(), hay.size(), l.first.data(), l.first.size())) return true;
    }
    return false;
}
}  // namespace

void slot_set_invert(ScanSlot* s, bool invert) {
    std::lock_guard<std::mutex> lk(g_mode_mu);
    g_mode[s].invert = invert;
}

void slot_set_context(ScanSlot* s, uint32_t before, uint32_t after) {
    std::lock_guard<std::mutex> lk(g_mode_mu);
    g_mode[s].before = before;
    g_mode[s].after = after;
}

void slot_set_literals(ScanSlot* s, bool literal) {
    std::lock_guard<std::mutex> lk(g_mode_mu);
    g_mode[s].literal = literal;
}

int slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    Mode w;
    {
        std::lock_guard<std::mutex> lk(g_mode_mu);
        auto it = g_mode.find(s);
        if (it != g_mode.end()) w = it->second;
    }
    const Database& db = *s->ddb->db;
    if (w.literal != db.literal) { error = "mock engine: fixed-string mode and database disagree"; return 7; }
    // every pseudo-line of the segment, split as the stand-in splits them
    std::vector<LineRec> lines;
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    for (size_t pos = 0; pos < s->n;) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        lines.push_back(LineRec{(uint32_t)lines.size(), (uint32_t)pos, (uint32_t)len});
        pos += len;
    }
    if (w.literal) {
        out = SegmentResult();
        s->recs.clear();
        const auto lits = literals_of(db);
        for (const LineRec& r : lines)
            if (block_has_literal(s->data + r.start, r.len, lits)) s->recs.push_back(r);
        out.num_lines = lines.size();
        out.stats.path = 2;
    } else {
        int rc = matched_slot_collect(s, out, error, split_above);
        if (rc) return rc;
    }
    if (!w.invert && w.before == 0 && w.after == 0) {
        out.lines = s->recs.data();
        out.num_line_recs = s->recs.size();
        return 0;
    }
    const size_t nlines = lines.size();
    std::vector<uint8_t> selected(nlines, 0);
    for (const LineRec& r : s->recs) selected[r.line] = 1;
    if (w.invert)
        for (auto& v : selected) v ^= 1;
    std::vector<size_t> P(nlines + 1, 0);
    for (size_t i = 0; i < nlines; i++) P[i + 1] = P[i] + selected[i];
    std::vector<LineRec> output;
    for (size_t i = 0; i < nlines; i++) {
        const bool edge = (w.before || w.after) && (i < w.after || i + w.before >= nlines);
        if (!edge && P[std::min(nlines, i + w.before + 1)] == P[i >= w.after ? i - w.after : 0]) continue;
        LineRec r = lines[i];
        if (!selected[i]) r.len |= kLineContext;
        output.push_back(r);
    }
    s->recs.swap(output);
    out.lines = s->recs.data();
    out.num_line_recs = out.num_valid_recs = s->recs.size();
    return 0;
}

}  // namespace gpugrep
