// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with the span stage (grep -o, gpugrep_match_spans).
//
// The CPU engine of tests/mock_engine (included unchanged) serves every other scan.  For a slot switched to spans
// (slot_set_spans), slot_collect splits the segment into pseudo-lines as that engine does and runs the span program of
// pike_vm.hpp - the function the CUDA kernel k_spans runs - over each stripped block on the CPU.  This lets
// `pytest -m "not gpu"` check the program, the exactness screen and the host logic (capi.cpp, the Python layer) against
// Python's re without a GPU; the kernel itself is checked by the `-m gpu` tests.
#include <mutex>
#include <unordered_map>

#define slot_collect matched_slot_collect
#include "../mock_engine/engine_cpu_mock.cpp"
#undef slot_collect

#include "pike_vm.hpp"

namespace gpugrep {

namespace {
std::mutex g_spans_mu;
std::unordered_map<const ScanSlot*, const PikeProgram*> g_program;   // set by the boundary on every slot it acquires
std::unordered_map<const ScanSlot*, std::vector<SpanRec>> g_spans;
}  // namespace

void slot_set_spans(ScanSlot* s, const PikeProgram* program) {
    std::lock_guard<std::mutex> lk(g_spans_mu);
    g_program[s] = program;
}

int slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    const PikeProgram* program = nullptr;
    std::vector<SpanRec>* spans = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_spans_mu);
        auto it = g_program.find(s);
        if (it != g_program.end()) program = it->second;
        spans = &g_spans[s];
    }
    if (!program) return matched_slot_collect(s, out, error, split_above);
    out = SegmentResult();
    spans->clear();
    const PikeView view = program->view();
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    uint32_t line = 0;
    for (size_t pos = 0; pos < s->n; line++) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        const uint8_t* p = s->data + pos;
        size_t a = 0;
        while (a < len && p[a] == 0) a++;
        size_t e = a;
        while (e < len && p[e] != 0) e++;
        const size_t first = spans->size();
        const bool ok = pike_spans(view, p + a, (uint32_t)(e - a), [&](uint32_t st, uint32_t en) { spans->push_back(SpanRec{line, st, en}); });
        if (!ok) {
            spans->resize(first);
            spans->push_back(SpanRec{line, kSpanOverBudget, kSpanOverBudget});
        }
        pos += len;
    }
    out.num_lines = line;
    out.spans = spans->data();
    out.num_spans = spans->size();
    out.stats.path = 2;
    return 0;
}

}  // namespace gpugrep
