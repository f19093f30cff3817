// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with inverted scans (grep -v).
//
// The CPU engine of tests/mock_engine (included unchanged) finds the matched pseudo-lines; for a slot switched to inverted
// scanning, slot_collect replaces them with the pseudo-lines that did not match, split exactly as the stand-in splits them.
// This lets `pytest -m "not gpu"` exercise the host logic of inverted scans (capi.cpp: batching, max_match_count, the
// sharded merge, ingest; the Python layer and the CLI) without a GPU.  The complement itself runs on the GPU in
// libgpugrep.so (k_invert.cuh) and is checked by the `-m gpu` tests.
#include <mutex>
#include <unordered_map>

#define slot_collect matched_slot_collect
#include "../mock_engine/engine_cpu_mock.cpp"
#undef slot_collect

namespace gpugrep {

namespace {
std::mutex g_invert_mu;
std::unordered_map<const ScanSlot*, bool> g_invert;   // set by the boundary on every slot it acquires
}  // namespace

void slot_set_invert(ScanSlot* s, bool invert) {
    std::lock_guard<std::mutex> lk(g_invert_mu);
    g_invert[s] = invert;
}

int slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    int rc = matched_slot_collect(s, out, error, split_above);
    {
        std::lock_guard<std::mutex> lk(g_invert_mu);
        auto it = g_invert.find(s);
        if (rc || it == g_invert.end() || !it->second) return rc;
    }
    // the boundary scans inverted sets as simple-mode databases: one record per matched line, in line order
    std::vector<LineRec> selected;
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    size_t pos = 0, next = 0;
    for (uint32_t line = 0; pos < s->n; line++) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        if (next < s->recs.size() && s->recs[next].line == line) next++;
        else selected.push_back(LineRec{line, (uint32_t)pos, (uint32_t)len});
        pos += len;
    }
    s->recs.swap(selected);
    out.lines = s->recs.data();
    out.num_line_recs = out.num_valid_recs = s->recs.size();
    return 0;
}

}  // namespace gpugrep
