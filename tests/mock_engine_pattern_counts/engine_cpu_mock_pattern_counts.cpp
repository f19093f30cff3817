// TEST-ONLY stand-in for hypergrep_b200/csrc/engine.cu with per-pattern line counts (gpugrep_pattern_counts_*).
//
// The stand-in of tests/mock_engine_literal (included unchanged) scans everything else.  For a slot switched to pattern
// counts, every pseudo-line of the segment (split as that stand-in splits them) gets the set of ids that report in it
// from the attribution database: regex sets through the stand-in's own automaton walk in event mode, each event expanded
// to its ids through the host's report lists; fixed strings by the definition of include/gpugrep.h itself, each literal
// passed in (read back with its flags from the database's cache key; its id is its index) searched with memmem in the
// scanned block (leading NULs skipped, cut at the next NUL), caseless ones on an ASCII-folded copy.  Each id of the set
// adds 1 to the slot's count of that id, which slot_read_pattern_counts hands over, as the engine keeps them on the device.  So the host's databases, segments, summing, shards and return codes are under test without a
// GPU.  The kernels run on the GPU in libgpugrep.so (k_pattern_counts.cuh) and are checked by the `-m gpu` tests.
#include <set>

#include "../mock_engine_literal/engine_cpu_mock_literal.cpp"

// That stand-in's slot_collect scans every other slot; the boundary's calls to it are routed here instead by the linker
// (-Wl,--wrap, see the Makefile), and this file calls it directly.
#define GPUGREP_SLOT_COLLECT "_ZN7gpugrep12slot_collectEPNS_8ScanSlotERNS_13SegmentResultERNSt7__cxx1112basic_stringIcSt11char_traitsIcESaIcEEEm"

namespace gpugrep {

namespace {
std::mutex g_counts_mu;
std::unordered_map<const ScanSlot*, const DeviceDb*> g_counts;
std::unordered_map<const ScanSlot*, std::vector<unsigned long long>> g_count_sum;   // since slot_set_pattern_counts

// The literals of a fixed-string database in the order given, parsed back from its cache key (literal, NUL, flags, id).
std::vector<std::pair<std::string, bool>> given_literals(const Database& db) {
    std::vector<std::pair<std::string, bool>> out;
    const std::string& k = db.key;
    size_t pos = 0;
    while (out.size() < db.literals.given) {
        const size_t nul = k.find('\0', pos);
        unsigned flags = 0;
        std::memcpy(&flags, k.data() + nul + 1, sizeof(flags));
        std::string text = k.substr(pos, nul - pos);
        if (flags & 1u) for (char& c : text) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
        out.emplace_back(std::move(text), (flags & 1u) != 0);
        pos = nul + 1 + 2 * sizeof(unsigned);
    }
    return out;
}
}  // namespace

// The report stage itself is not simulated here: fixed-string pattern counts only need the switch.
void slot_set_literal_reports(ScanSlot*, bool) {}

void slot_set_pattern_counts(ScanSlot* s, const DeviceDb* attribution) {
    std::lock_guard<std::mutex> lk(g_counts_mu);
    g_counts[s] = attribution;
    g_count_sum[s].clear();
}

int slot_read_pattern_counts(ScanSlot* s, std::vector<unsigned long long>& sum, std::string&) {
    std::lock_guard<std::mutex> lk(g_counts_mu);
    std::vector<unsigned long long>& mine = g_count_sum[s];
    for (size_t i = 0; i < std::min(mine.size(), sum.size()); i++) sum[i] += mine[i];
    mine.clear();
    return 0;
}

int counts_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) __asm__("__wrap_" GPUGREP_SLOT_COLLECT);
int counts_slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    const DeviceDb* attribution = nullptr;
    std::vector<unsigned long long>* counts = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_counts_mu);
        auto it = g_counts.find(s);
        if (it != g_counts.end()) attribution = it->second;
        counts = &g_count_sum[s];
    }
    if (!attribution) return slot_collect(s, out, error, split_above);
    const Database& db = *attribution->db;
    if (db.simple && !db.literal_reports) { error = "mock engine: pattern counts need an event-mode or report database"; return 7; }
    out = SegmentResult();
    std::vector<std::pair<std::string, bool>> lits;
    std::vector<std::pair<uint32_t, uint32_t>> flat;   // regex sets: flat report -> [begin, end) of db.reports
    if (db.literal_reports) {
        lits = given_literals(db);
        counts->resize(lits.size(), 0);
    } else {
        for (const auto& rb : db.report_begin)
            for (size_t k = 0; k + 1 < rb.size(); k++) flat.emplace_back(rb[k], rb[k + 1]);
        for (const auto& np : db.nfas) flat.emplace_back(np.report_begin, np.report_begin + 1);
        counts->resize(db.patterns.size(), 0);
    }
    const size_t limit = (size_t)std::max(1, s->buffer_size - 1);
    uint32_t line = 0;
    size_t matched = 0;
    std::vector<EventRec> events;
    for (size_t pos = 0; pos < s->n; line++) {
        const size_t avail = std::min(limit, s->n - pos);
        const void* nl = std::memchr(s->data + pos, '\n', avail);
        const size_t len = nl ? (size_t)((const uint8_t*)nl - (s->data + pos)) + 1 : avail;
        const uint8_t* p = s->data + pos;
        std::set<unsigned> ids;
        if (db.literal_reports) {
            size_t a = 0;
            while (a < len && p[a] == 0) a++;
            const void* nul = std::memchr(p + a, 0, len - a);
            const size_t e = nul ? (size_t)((const uint8_t*)nul - p) : len;
            std::string raw((const char*)p + a, e - a), folded(raw);
            for (char& c : folded) if ((unsigned)(unsigned char)c - 'A' < 26u) c |= 0x20;
            for (size_t i = 0; i < lits.size(); i++) {
                const std::string& hay = lits[i].second ? folded : raw;
                if (memmem(hay.data(), hay.size(), lits[i].first.data(), lits[i].first.size())) ids.insert((unsigned)i);
            }
        } else {
            bool hit = false;
            events.clear();
            walk(db, p, len, line, (uint32_t)pos, false, hit, events);
            for (const EventRec& ev : events)
                for (uint32_t k = flat[ev.report].first; k < flat[ev.report].second; k++) ids.insert(db.reports[k].id);
        }
        for (unsigned id : ids) (*counts)[id]++;
        matched += !ids.empty();
        pos += len;
    }
    out.num_lines = line;
    out.pattern_counts = true;
    out.num_valid_recs = matched;
    out.stats.path = 2;
    return 0;
}

}  // namespace gpugrep
