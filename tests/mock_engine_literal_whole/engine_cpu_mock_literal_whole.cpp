// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with whole-word / whole-line fixed strings
// (gpugrep_literal_whole_scan_*).
//
// The stand-in of tests/mock_engine_literal (included unchanged) selects the lines that hold a literal.  For a slot
// switched to whole words or lines, each of those lines is then kept by the definition of include/gpugrep.h itself: every
// literal passed in, read back with its flags from the database's cache key, is searched in the scanned block (leading
// NULs skipped, cut at the next NUL) with memmem, caseless ones on an ASCII-folded copy, and each occurrence is checked
// for a non-word byte (or the block edge) on both sides; a line is kept in line mode when the block without its final
// '\n' equals a literal.  Inversion and context lines then follow from the kept lines, as in that stand-in.  So the
// host's database, segments, limits, batching, shards and delivery are under test without a GPU.  The kernels run on the
// GPU in libgpugrep.so (k_literal_whole.cuh) and are checked by the `-m gpu` tests.
#include "../mock_engine_literal/engine_cpu_mock_literal.cpp"

// That stand-in's slot_collect is the selection; the boundary's calls to it are routed here instead by the linker
// (-Wl,--wrap, see the Makefile), and this file calls it directly.
#define GPUGREP_SLOT_COLLECT "_ZN7gpugrep12slot_collectEPNS_8ScanSlotERNS_13SegmentResultERNSt7__cxx1112basic_stringIcSt11char_traitsIcESaIcEEEm"

namespace gpugrep {

namespace {
std::mutex g_whole_mu;
std::unordered_map<const ScanSlot*, unsigned> g_whole;

bool word_byte(unsigned char c) { return (c >= '0' && c <= '9') || (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || c == '_'; }

bool block_passes(const uint8_t* p, size_t len, const std::vector<std::pair<std::string, bool>>& lits, unsigned whole) {
    size_t a = 0;
    while (a < len && p[a] == 0) a++;
    const void* nul = std::memchr(p + a, 0, len - a);
    const size_t e = nul ? (size_t)((const uint8_t*)nul - p) : len;
    std::string raw((const char*)p + a, e - a), folded(raw);
    for (char& c : folded) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
    for (const auto& l : lits) {
        const std::string& hay = l.second ? folded : raw;
        if (whole == 2) {
            const size_t n = !hay.empty() && hay.back() == '\n' ? hay.size() - 1 : hay.size();
            if (hay.compare(0, n, l.first) == 0 && l.first.size() == n) return true;
            continue;
        }
        for (size_t at = 0; at + l.first.size() <= hay.size(); at++) {
            const void* hit = memmem(hay.data() + at, hay.size() - at, l.first.data(), l.first.size());
            if (!hit) break;
            at = (size_t)((const char*)hit - hay.data());
            const size_t end = at + l.first.size();
            if ((at == 0 || !word_byte((unsigned char)raw[at - 1])) && (end == raw.size() || !word_byte((unsigned char)raw[end]))) return true;
        }
    }
    return false;
}
}  // namespace

void slot_set_literal_whole(ScanSlot* s, unsigned whole) {
    std::lock_guard<std::mutex> lk(g_whole_mu);
    g_whole[s] = whole;
}

int whole_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) __asm__("__wrap_" GPUGREP_SLOT_COLLECT);
int whole_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    unsigned whole = 0;
    {
        std::lock_guard<std::mutex> lk(g_whole_mu);
        auto it = g_whole.find(s);
        if (it != g_whole.end()) whole = it->second;
    }
    if (!whole) return slot_collect(s, out, error, split_above);
    const Database& db = *s->ddb->db;
    if (!db.literal_whole) { error = "mock engine: whole-word / whole-line scan of a database not compiled for it"; return 7; }
    Mode w;
    {   // the plain fixed-string selection first: no inversion, no context
        std::lock_guard<std::mutex> lk(g_mode_mu);
        w = g_mode[s];
        g_mode[s] = Mode{false, true, 0, 0};
    }
    int rc = slot_collect(s, out, error, split_above);
    {
        std::lock_guard<std::mutex> lk(g_mode_mu);
        g_mode[s] = w;
    }
    if (rc) return rc;
    const auto lits = literals_of(db);
    std::vector<LineRec> kept;
    for (size_t i = 0; i < out.num_line_recs; i++)
        if (block_passes(s->data + out.lines[i].start, out.lines[i].len, lits, whole)) kept.push_back(out.lines[i]);
    const size_t nlines = (size_t)out.num_lines;
    std::vector<uint8_t> selected(nlines, 0);
    for (const LineRec& r : kept) selected[r.line] = 1;
    if (w.invert)
        for (auto& v : selected) v ^= 1;
    // every pseudo-line's extents, split as the stand-in splits them
    std::vector<LineRec> lines;
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    for (size_t pos = 0; pos < s->n;) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        lines.push_back(LineRec{(uint32_t)lines.size(), (uint32_t)pos, (uint32_t)len});
        pos += len;
    }
    std::vector<size_t> P(nlines + 1, 0);
    for (size_t i = 0; i < nlines; i++) P[i + 1] = P[i] + selected[i];
    s->recs.clear();
    for (size_t i = 0; i < nlines; i++) {
        const bool edge = (w.before || w.after) && (i < w.after || i + w.before >= nlines);
        if (!edge && P[std::min(nlines, i + w.before + 1)] == P[i >= w.after ? i - w.after : 0]) continue;
        LineRec r = lines[i];
        if (!selected[i]) r.len |= kLineContext;
        s->recs.push_back(r);
    }
    out.lines = s->recs.data();
    out.num_line_recs = out.num_valid_recs = s->recs.size();
    return 0;
}

}  // namespace gpugrep
