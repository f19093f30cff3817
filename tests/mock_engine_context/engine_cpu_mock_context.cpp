// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with context lines (grep -A/-B/-C).
//
// The CPU engine of tests/mock_engine (included unchanged) finds the matched pseudo-lines; the selected ones are those, or
// for an inverted scan the others, as in tests/mock_engine_invert.  For a slot switched to context lines, slot_collect
// returns the per-segment superset the CUDA engine returns (engine.hpp
// slot_set_context): every pseudo-line with a selected line within `after` lines before or `before` lines after it, and the
// segment's first `after` and last `before` lines, with kLineContext on the ones that are not selected.  This lets
// `pytest -m "not gpu"` exercise the host logic of context scans (capi.cpp: the context filter across segments and shards,
// the trailing context after max_match_count, batching; the Python layer and the CLI) without a GPU.  The stage itself runs
// on the GPU in libgpugrep.so (k_context.cuh) and is checked by the `-m gpu` tests.
#include <mutex>
#include <unordered_map>

#define slot_collect matched_slot_collect
#include "../mock_engine/engine_cpu_mock.cpp"
#undef slot_collect

namespace gpugrep {

namespace {
struct Mode {
    bool invert = false;
    uint32_t before = 0, after = 0;
};
std::mutex g_mode_mu;
std::unordered_map<const ScanSlot*, Mode> g_mode;   // set by the boundary on every slot it acquires
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

int slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    int rc = matched_slot_collect(s, out, error, split_above);
    Mode w;
    {
        std::lock_guard<std::mutex> lk(g_mode_mu);
        auto it = g_mode.find(s);
        if (it != g_mode.end()) w = it->second;
    }
    if (rc || (!w.invert && w.before == 0 && w.after == 0)) return rc;
    // every pseudo-line of the segment, split as the stand-in splits them; the selected ones and their prefix count P (the
    // boundary scans these sets as simple-mode databases: one record per matched line)
    std::vector<LineRec> lines;
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    for (size_t pos = 0; pos < s->n;) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        lines.push_back(LineRec{(uint32_t)lines.size(), (uint32_t)pos, (uint32_t)len});
        pos += len;
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
        if (!edge && P[i + w.before + 1] == P[i - w.after]) continue;
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
