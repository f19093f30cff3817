// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with the fixed-string report stage (gpugrep_literal_report_scan_*).
//
// The stand-in of tests/mock_engine_literal (included unchanged) selects the lines.  For a slot switched to reports, every
// selected pseudo-line then yields its reports by the definition of include/gpugrep.h itself: each literal passed in, read
// back with its flags and id from the database's cache key, is searched at every position of the scanned block (leading NULs
// skipped, cut at the next NUL) with memmem, caseless ones on an ASCII-folded copy.  An occurrence becomes an EventRec whose
// `report` is the node of the host's report table that holds that literal, so the host's table, its expansion of a node to
// ids, the de-duplication, SINGLEMATCH, the limit and the delivery are all under test.  The kernels run on the GPU in
// libgpugrep.so (k_literal_reports.cuh) and are checked by the `-m gpu` tests.
#include <map>

#include "../mock_engine_literal/engine_cpu_mock_literal.cpp"

// That stand-in's slot_collect is the selection; the boundary's calls to it are routed here instead by the linker
// (-Wl,--wrap, see the Makefile), and this file calls it directly.
#define GPUGREP_SLOT_COLLECT "_ZN7gpugrep12slot_collectEPNS_8ScanSlotERNS_13SegmentResultERNSt7__cxx1112basic_stringIcSt11char_traitsIcESaIcEEEm"

namespace gpugrep {

namespace {
std::mutex g_reports_mu;
std::unordered_map<const ScanSlot*, bool> g_reports;

struct Given {
    std::string text;   // folded when caseless
    bool caseless;
};

// The literals of a report database, parsed back from its cache key (literal, NUL, flags, id; then options).
std::vector<Given> given_of(const Database& db) {
    std::vector<Given> out;
    const std::string& k = db.key;
    size_t pos = 0;
    while (out.size() < db.literals.given) {
        const size_t nul = k.find('\0', pos);
        unsigned flags = 0;
        std::memcpy(&flags, k.data() + nul + 1, sizeof(flags));
        Given g{k.substr(pos, nul - pos), (flags & 1u) != 0};
        if (g.caseless) for (char& c : g.text) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
        out.push_back(std::move(g));
        pos = nul + 1 + 2 * sizeof(unsigned);
    }
    return out;
}
}  // namespace

void slot_set_literal_reports(ScanSlot* s, bool reports) {
    std::lock_guard<std::mutex> lk(g_reports_mu);
    g_reports[s] = reports;
}

int report_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) __asm__("__wrap_" GPUGREP_SLOT_COLLECT);
int report_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    bool reports = false;
    {
        std::lock_guard<std::mutex> lk(g_reports_mu);
        auto it = g_reports.find(s);
        if (it != g_reports.end()) reports = it->second;
    }
    int rc = slot_collect(s, out, error, split_above);
    if (rc || !reports) return rc;
    const Database& db = *s->ddb->db;
    if (!db.literal_reports) { error = "mock engine: report scan of a database without a report table"; return 7; }
    const LiteralReports& R = db.lit_reports;
    std::map<std::pair<bool, std::string>, uint32_t> node_of;
    for (uint32_t k = 0; k < R.off.size(); k++)
        node_of[{R.caseless[k] != 0, std::string((const char*)R.bytes.data() + R.off[k], R.len[k])}] = k;
    std::vector<std::pair<Given, uint32_t>> lits;
    for (Given& g : given_of(db)) {
        auto it = node_of.find({g.caseless, g.text});
        if (it != node_of.end()) lits.emplace_back(g, it->second);
        else if (g.text.find('\n') == g.text.size() - 1 || g.text.find('\n') == std::string::npos) {
            error = "mock engine: a literal that can match has no node";
            return 7;
        }
    }
    s->events.clear();
    for (size_t i = 0; i < out.num_line_recs; i++) {
        const LineRec& r = out.lines[i];
        const uint8_t* p = s->data + r.start;
        size_t a = 0;
        while (a < r.len && p[a] == 0) a++;
        const void* nul = std::memchr(p + a, 0, r.len - a);
        const size_t e = nul ? (size_t)((const uint8_t*)nul - p) : r.len;
        std::string raw((const char*)p + a, e - a), folded(raw);
        for (char& c : folded) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
        for (const auto& [g, node] : lits) {
            const std::string& hay = g.caseless ? folded : raw;
            for (size_t at = 0; at + g.text.size() <= hay.size(); at++) {
                const void* hit = memmem(hay.data() + at, hay.size() - at, g.text.data(), g.text.size());
                if (!hit) break;
                at = (size_t)((const char*)hit - hay.data());
                s->events.push_back(EventRec{r.line, r.start, r.len, (uint32_t)(at + g.text.size()), node});
            }
        }
    }
    out.lines = nullptr;
    out.num_line_recs = out.num_valid_recs = 0;
    out.events = s->events.data();
    out.num_events = s->events.size();
    return 0;
}

}  // namespace gpugrep
