// C ABI: hyperscan() and the buffer/file scan entry points of include/gpugrep.h.
//
// Host driver around the CUDA engine.  It restates the control flow of the reference shim
//   hyperscan()     reference hyperscanner.c:248-326  (batch clamp, compile, scan, tail flush, return codes)
//   hyperscan_gz()  reference hyperscanner.c:179-231  (line loop, max_match_count stop rule)
//   hs_callback()   reference hyperscanner.c:83-102   (result slots, full batches then the remainder)
// with the per-line work moved to the GPU: the file is cut into segments that begin and end on pseudo-line
// boundaries, two segments are kept in flight (read/H2D of k+1 overlaps kernels and delivery of k), and the
// matched-line records that come back are turned into callbacks on the calling thread, in file order.
#include <cuda_runtime.h>
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <functional>
#include <list>
#include <mutex>
#include <thread>
#include <utility>
#include <string>
#include <vector>

#include "../../include/gpugrep.h"
#include "database.hpp"
#include "engine.hpp"
#include "ingest.hpp"
#include "pike_vm.hpp"

namespace gpugrep {
void set_last_error(const std::string& e);

namespace {

std::atomic<int> g_device_override{-1};
thread_local int t_device_override = -1;   // set by the shard workers of a scan that is split over several GPUs

// Outstanding bytes per device (files being scanned): a new scan goes to the least loaded GPU, so that one large file
// next to many small ones does not leave the other devices idle (SURVEY.md section 8f-3: placement by size).
constexpr int kMaxLoadDevices = 64;
std::atomic<unsigned long long> g_device_load[kMaxLoadDevices];

// `charged`: set when the choice was made by load (the caller gives the weight back through release_device).
int pick_device(unsigned long long weight, bool* charged) {
    *charged = false;
    if (t_device_override >= 0) return t_device_override;
    int d = g_device_override.load();
    if (d >= 0) return d;
    if (const char* e = std::getenv("GPUGREP_DEVICE")) return std::atoi(e);
    if (const char* e = std::getenv("LOCAL_RANK")) return std::atoi(e);
    // no explicit choice: spread the scans (one per file in multiscanner) over all visible GPUs
    const int count = std::min(engine_device_count(), kMaxLoadDevices);
    if (count <= 1) return 0;
    static std::mutex mu;
    static unsigned next = 0;
    std::lock_guard<std::mutex> lk(mu);
    int best = 0;
    unsigned long long best_load = ~0ull;
    for (int k = 0; k < count; k++) {   // ties go round-robin
        const int dev = (int)((next + (unsigned)k) % (unsigned)count);
        const unsigned long long load = g_device_load[dev].load();
        if (load < best_load) { best_load = load; best = dev; }
    }
    next = (unsigned)best + 1;
    g_device_load[best].fetch_add(weight + 1);
    *charged = true;
    return best;
}
void release_device(int device, unsigned long long weight) { g_device_load[device].fetch_sub(weight + 1); }

size_t env_mb(const char* name, size_t dflt_mb) {
    if (const char* b = std::getenv("GPUGREP_CHUNK_BYTES")) {   // test hook: tiny segments exercise the cut logic
        if (*b) return (size_t)std::strtoull(b, nullptr, 10);
    }
    const char* v = std::getenv(name);
    if (!v || !*v) return dflt_mb << 20;
    return (size_t)std::strtoull(v, nullptr, 10) << 20;
}

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Host batcher: the result slots of hyperscanner_state_t (hyperscanner.c:64-72) and hs_callback (:83-102).
// The reference keeps buffer_count slots of buffer_size bytes and strcpy()s every matched line into one; here the
// lines of a batch are packed into pooled blocks (stable addresses until the batch has been delivered).
// One result of a shard, kept until the shards before it have been delivered (scans split over several GPUs).
struct ShardRecord {
    unsigned id;
    unsigned long long line;   // pseudo-line index inside the shard
    size_t offset;             // of the delivered text in ShardResults::text (NUL-terminated there)
};
struct ShardResults {
    std::vector<ShardRecord> records;
    std::vector<char> text;
};

// Sink of gpugrep_match_ends(): (line, id, end) records instead of lines.
struct EndsSink {
    gpugrep_match_end* out;
    size_t capacity;
    size_t count = 0;
};

// Sink of gpugrep_match_spans(): (line, start, end) records.
struct SpansSink {
    gpugrep_match_span* out;
    size_t capacity;
    size_t count = 0;
};

class Deliverer {
public:
    Deliverer(hs_event cb, int buffer_count) : cb_(cb), cap_(std::max(1, buffer_count)) {
        if (cb_) results_.resize((size_t)cap_);
    }
    // collecting deliverer of a shard worker: results are stored, not called back
    explicit Deliverer(ShardResults* collect) : cb_(nullptr), cap_(1), collect_(collect) {}
    // `bytes`/`len`: the pseudo-line as it sits in the file.  The delivered text is what the reference strcpy()s:
    // leading NULs skipped, cut at the next NUL (hyperscanner.c:205-214, :92).  `counted`: false for context lines, which
    // count() leaves out.
    void emit(unsigned id, unsigned long long line_number, const uint8_t* bytes, size_t len, bool may_have_nul = true, bool counted = true) {
        if (counted) count_++;
        if (!cb_ && !collect_) return;
        size_t a = 0, b = len;
        if (may_have_nul) strip(bytes, len, a, b);
        if (collect_) {
            collect_->records.push_back(ShardRecord{id, line_number, collect_->text.size()});
            collect_->text.insert(collect_->text.end(), (const char*)bytes + a, (const char*)bytes + b);
            collect_->text.push_back('\0');
            return;
        }
        char* dst = place(b - a + 1);
        std::memcpy(dst, bytes + a, b - a);
        dst[b - a] = '\0';
        hyperscanner_result_t& r = results_[(size_t)fill_];
        r.id = id;
        r.line_number = line_number;
        r.line = dst;
        fill_++;
        if (fill_ == cap_) flush();
    }
    void emit_count_only(unsigned long long n) { count_ += n; }
    void set_ends(EndsSink* sink) { ends_ = sink; }
    bool wants_ends() const { return ends_ != nullptr; }
    void emit_end(unsigned id, unsigned long long line_number, unsigned end) {
        count_++;
        if (ends_->count < ends_->capacity) ends_->out[ends_->count] = gpugrep_match_end{line_number, id, end};
        ends_->count++;
    }
    void set_spans(SpansSink* sink) { spans_ = sink; }
    bool wants_spans() const { return spans_ != nullptr; }
    void emit_span(unsigned long long line_number, unsigned start, unsigned end) {
        count_++;
        if (spans_->count < spans_->capacity) spans_->out[spans_->count] = gpugrep_match_span{line_number, start, end};
        spans_->count++;
    }
    void flush() {
        if (cb_ && fill_ > 0) cb_(results_.data(), fill_);
        fill_ = 0;
        block_ = 0;
        used_ = 0;
    }
    unsigned long long count() const { return count_; }
    bool wants_lines() const { return cb_ != nullptr || collect_ != nullptr; }
    // a stored result of a shard, already stripped: straight into the result slots
    void emit_text(unsigned id, unsigned long long line_number, const char* text) {
        emit(id, line_number, (const uint8_t*)text, std::strlen(text), false);
    }
    // the delivered text of a pseudo-line is [a, b)
    static void strip(const uint8_t* bytes, size_t len, size_t& a, size_t& b) {
        a = 0;
        b = len;
        while (a < len && bytes[a] == 0) a++;
        const void* z = std::memchr(bytes + a, 0, len - a);
        if (z) b = (size_t)((const uint8_t*)z - bytes);
    }
private:
    static constexpr size_t kBlock = (size_t)1 << 20;
    char* place(size_t bytes) {
        while (true) {
            if (block_ == blocks_.size()) blocks_.emplace_back(std::max(bytes, kBlock));
            std::vector<char>& blk = blocks_[block_];
            if (used_ + bytes <= blk.size()) { char* p = blk.data() + used_; used_ += bytes; return p; }
            if (used_ == 0) { blk.resize(bytes); continue; }   // an over-long line gets the whole (grown) block
            block_++;
            used_ = 0;
        }
    }
    hs_event cb_;
    int cap_;
    ShardResults* collect_ = nullptr;
    EndsSink* ends_ = nullptr;
    SpansSink* spans_ = nullptr;
    int fill_ = 0;
    unsigned long long count_ = 0;
    std::vector<hyperscanner_result_t> results_;
    std::vector<std::vector<char>> blocks_;
    size_t block_ = 0, used_ = 0;
};

// Context lines (grep -A/-B/-C) on the delivering thread.  It is fed, in file order, the selected lines and the context
// candidates of the engine: a superset of the context lines (the output lines of each segment and the segment's edge
// lines, see slot_set_context).  It delivers each output line once, selected lines with id 0 and context lines with
// GPUGREP_CONTEXT_ID.  It applies max_match_count to the selected lines; after the line that reaches the limit, the next
// `after` lines still go out, all as context.  `tag_only` (the shard workers of a scan over several GPUs): every record is
// passed on, tagged, for the merge to filter; only the limit applies.
class ContextFilter {
public:
    ContextFilter(Deliverer* out, uint32_t before, uint32_t after, unsigned long long max_match, bool tag_only)
        : out_(out), before_(before), after_(after), max_(max_match), tag_only_(tag_only) {}
    // false: the limit has been reached and `line` lies past the trailing context: nothing more will be delivered
    bool feed(bool selected, unsigned long long line, const uint8_t* bytes, size_t len, bool may_have_nul) {
        if (limit_reached()) {
            if (line - last_ > after_) return false;
            out_->emit(GPUGREP_CONTEXT_ID, line, bytes, len, may_have_nul, false);
            return true;
        }
        if (selected) {
            for (const Held& h : held_)
                if (line - h.line <= before_) out_->emit(GPUGREP_CONTEXT_ID, h.line, (const uint8_t*)h.text.data(), h.text.size(), false, false);
            held_.clear();
            out_->emit(0, line, bytes, len, may_have_nul);
            last_ = line;
            any_ = true;
            selected_++;
        } else if (tag_only_ || (any_ && line - last_ <= after_)) {
            out_->emit(GPUGREP_CONTEXT_ID, line, bytes, len, may_have_nul, false);
        } else if (before_) {
            // held until a selected line within `before` lines follows; at most `before` lines can be wanted
            size_t a = 0, b = len;
            if (may_have_nul) Deliverer::strip(bytes, len, a, b);
            held_.push_back(Held{line, std::string((const char*)bytes + a, b - a)});
            if (held_.size() > before_) held_.pop_front();
        }
        return true;
    }
    // the limit has been reached and every line from `next_line` on lies past the trailing context
    bool finished(unsigned long long next_line) const { return limit_reached() && next_line - last_ > after_; }

private:
    bool limit_reached() const { return max_ > 0 && selected_ >= max_; }
    struct Held {
        unsigned long long line;
        std::string text;   // stripped
    };
    Deliverer* out_;
    uint32_t before_, after_;
    unsigned long long max_;
    bool tag_only_;
    bool any_ = false;
    unsigned long long last_ = 0, selected_ = 0;
    std::deque<Held> held_;
};

constexpr size_t kSampleBytes = 512 << 10;   // head of the input used to tune the prefilter windows
std::mutex g_plain_mu;                       // admission of plain-file scans (see scan_file)
std::condition_variable g_plain_cv;
constexpr int kMaxDevices = 64;              // power of two
int g_plain_scans[kMaxDevices] = {};
constexpr int kMaxPlainScans = 4;            // per device

// Sample-tuned prefilter tables, cached per (database, device, sample fingerprint).  `sample` must hold the first
// min(len, 64 KiB) bytes (the fingerprint); `fetch_full`, if given, returns a pointer to all `len` bytes and is only
// called on a cache miss (device-resident inputs copy the rest of the sample only then).
std::shared_ptr<DevicePrefilter> tuned_prefilter(const std::shared_ptr<Database>& db, const uint8_t* sample, size_t len, std::string& error,
                                                 const std::function<const uint8_t*()>& fetch_full = nullptr, bool reuse_sibling = false) {
    if (!db->simple || !db->factors.usable) return nullptr;
    struct Entry { const Database* db; int device; uint64_t fp; std::shared_ptr<Database> keep; std::shared_ptr<DevicePrefilter> pf; };
    static std::mutex mu;
    static std::list<Entry> cache;
    len = std::min(len, kSampleBytes);
    uint64_t fp = 1469598103934665603ull ^ len;
    for (size_t i = 0; i + 8 <= std::min<size_t>(len, 64 << 10); i += 8) {
        uint64_t w;
        std::memcpy(&w, sample + i, 8);
        fp = (fp ^ w) * 1099511628211ull;
    }
    // a sample that is fully at hand (no fetch_full) is also told apart by its tail: a re-tuning sample shares its head
    // with the one it replaces
    if (!fetch_full && len > ((size_t)64 << 10)) {
        for (size_t i = len - ((size_t)64 << 10); i + 8 <= len; i += 8) {
            uint64_t w;
            std::memcpy(&w, sample + i, 8);
            fp = (fp ^ w) * 1099511628211ull;
        }
    }
    const int device = engine_current_device();
    {
        std::lock_guard<std::mutex> lk(mu);
        for (auto it = cache.begin(); it != cache.end(); ++it) {
            if (it->db == db.get() && it->device == device && it->fp == fp) {
                cache.splice(cache.begin(), cache, it);
                return cache.front().pf;
            }
        }
        // Another input of the same scan (multiscanner: many files, one pattern set): the table that was tuned on a
        // sibling file is taken as it is - building the gram histogram of every file's head costs milliseconds per file,
        // more than scanning a small file does.  If this text is different after all, the first segments flag more chunks
        // than the sample promised and the windows are chosen again (Job::drifted / retune).
        if (reuse_sibling && std::getenv("GPUGREP_NO_TUNE") == nullptr) {
            for (auto it = cache.begin(); it != cache.end(); ++it)
                if (it->db == db.get() && it->device == device && prefilter_expected_hits(it->pf.get()) >= 0) return it->pf;
        }
    }
    Prefilter pf;
    if (len >= 4096 && std::getenv("GPUGREP_NO_TUNE") == nullptr) {
        if (fetch_full) sample = fetch_full();
        if (!sample) { error = "could not read the tuning sample"; return nullptr; }
        GramHistogram hist;
        hist.add_sample(sample, len);
        build_prefilter(db->factors, &hist, pf);
    } else {
        pf = db->prefilter;
    }
    auto dpf = engine_upload_prefilter(pf, error);
    if (!dpf) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    cache.push_front(Entry{db.get(), device, fp, db, dpf});
    while (cache.size() > 16) cache.pop_back();
    return dpf;
}

struct Job {
    int device = 0;
    unsigned long long device_weight = 0;
    bool device_charged = false;
    ~Job() { if (device_charged) release_device(device, device_weight); }
    std::shared_ptr<Database> db;
    std::shared_ptr<DeviceDb> ddb;
    std::shared_ptr<DevicePrefilter> dpf;   // null: general path
    int buffer_size = 0;
    unsigned long long max_match = 0;
    Deliverer* out = nullptr;
    ContextFilter* context = nullptr;   // scans with context lines: every record goes through it (it applies max_match)
    unsigned long long line_base = 0;
    bool stop = false;
    gpugrep_stats stats{};
    std::string error;
    // flattened accept-set lookup for general mode
    std::vector<uint32_t> report_begin_flat;
    // Drift of the text: the prefilter windows were chosen against the head of the input.  When a segment flags far more
    // chunks than that sample promised, the windows are chosen again against a sample that also holds text of the
    // drifting region (the filter is a superset filter: results do not change, only the number of candidates does).
    std::vector<uint8_t> tune_head;   // head of the input the current table was tuned on (at most 256 KiB)
    int retunes = 0;
    bool drifted(const SegmentResult& r, size_t segment_bytes) const {
        if (!dpf || retunes >= 3 || segment_bytes < ((size_t)1 << 20) || !(r.stats.path & 1)) return false;
        if (std::getenv("GPUGREP_NO_RETUNE") != nullptr) return false;
        const double expected = prefilter_expected_hits(dpf.get());
        if (expected < 0) return false;
        const double seen = (double)r.stats.candidates / ((double)segment_bytes / 1048576.0);
        return seen > 2.0 * std::max(expected, 500.0) + 1000.0;
    }
    // `region`: host bytes of the drifting text (a few hundred KiB are used)
    void retune(const uint8_t* region, size_t len) {
        std::vector<uint8_t> sample(tune_head);
        const size_t take = std::min<size_t>(len, kSampleBytes - std::min(kSampleBytes / 2, sample.size()));
        sample.resize(std::min(sample.size(), kSampleBytes / 2));
        sample.insert(sample.end(), region, region + take);
        std::string err;
        auto fresh = tuned_prefilter(db, sample.data(), sample.size(), err);
        if (fresh) dpf = fresh;
        retunes++;
    }

    // events, not line records: general-mode sets and fixed-string sets compiled for reports
    bool wants_events() const { return !db->simple || db->literal_reports; }

    void prepare() {
        if (db->literal_reports) {   // device events carry the node of the report table
            const auto& rb = db->lit_reports.report_begin;
            report_begin_flat.assign(rb.begin(), rb.end() - 1);
            report_end_flat.assign(rb.begin() + 1, rb.end());
            return;
        }
        if (db->simple) return;   // the flat report ranges are only read when events are expanded to ids
        for (auto& rb : db->report_begin) {
            // every group's list ends with a sentinel; keep [begin, next begin) pairs addressable by flat index
            for (size_t k = 0; k + 1 < rb.size(); k++) { report_begin_flat.push_back(rb[k]); report_end_flat.push_back(rb[k + 1]); }
        }
        // NFA-fallback patterns follow, one report each (engine: NfaView::report)
        for (auto& np : db->nfas) { report_begin_flat.push_back(np.report_begin); report_end_flat.push_back(np.report_begin + 1); }
    }
    std::vector<uint32_t> report_end_flat;

    bool limit_reached() const { return max_match > 0 && out->count() >= max_match; }

    // Turn one segment's records into callbacks.  `host` is the segment's bytes on the host, or nullptr when the
    // input lives on the device only (then matched lines are gathered through the slot).
    int deliver(const SegmentResult& r, const uint8_t* host, ScanSlot* slot) {
        stats.lines += r.num_lines;
        stats.gpu_ms += r.stats.gpu_ms;
        stats.stream_kernel_ms += r.stats.stream_ms;
        stats.launches += r.stats.launches;
        stats.stream_launches += r.stats.stream_launches;
        stats.candidates += r.stats.candidates;
        stats.h2d_bytes += r.stats.h2d_bytes;
        stats.d2h_bytes += r.stats.d2h_bytes;
        stats.path |= r.stats.path;
        stats.segments++;
        stats.nul_segments += r.stats.nul ? 1u : 0u;
        if (stop) return 0;
        int rc = out->wants_spans() ? deliver_spans(r) : (wants_events() ? deliver_events(r, host, slot) : deliver_simple(r, host, slot));
        line_base += r.num_lines;
        return rc;
    }

    int deliver_simple(const SegmentResult& r, const uint8_t* host, ScanSlot* slot) {
        const LineRec* recs = r.lines;
        size_t count = r.num_line_recs;
        const bool fast_rec = (r.stats.path & 1) != 0;   // fast-path records: NUL hint in len, dropped ones marked kLineInvalid
        if (fast_rec) {
            if (!out->wants_lines() && max_match == 0) { out->emit_count_only(r.num_valid_recs); return 0; }
            if (r.num_valid_recs != count) {
                unique_.clear();
                unique_.reserve(r.num_valid_recs);
                for (size_t i = 0; i < count; i++) if (recs[i].len != kLineInvalid) unique_.push_back(recs[i]);
                recs = unique_.data();
                count = unique_.size();
            }
        }
        size_t take = count;
        if (max_match > 0 && !context) {
            unsigned long long room = max_match > out->count() ? max_match - out->count() : 0;
            if ((unsigned long long)take >= room) { take = (size_t)room; stop = true; }
        }
        if (!out->wants_lines()) { out->emit_count_only(take); return 0; }
        std::vector<uint8_t> gathered;
        std::vector<unsigned long long> goff;
        if (!host && take) {
            std::vector<uint32_t> starts(take), lens(take);
            unsigned long long total = 0;
            goff.resize(take);
            for (size_t i = 0; i < take; i++) { starts[i] = recs[i].start; lens[i] = recs[i].len & kLineLenMask; goff[i] = total; total += lens[i] + 1ull; }
            gathered.resize((size_t)total);
            int rc = slot_gather_lines(slot, starts.data(), lens.data(), take, gathered.data(), error);
            if (rc) return rc;
        }
        for (size_t i = 0; i < take; i++) {
            const LineRec& lr = recs[i];
            if (host && i + 8 < take) {   // matched lines are scattered over the (pinned) input: hide the cache misses
                const uint8_t* ahead = host + recs[i + 8].start;
                __builtin_prefetch(ahead);
                __builtin_prefetch(ahead + 64);
                __builtin_prefetch(ahead + 128);
            }
            const uint8_t* bytes = host ? host + lr.start : gathered.data() + goff[i];
            const bool may_have_nul = fast_rec ? (lr.len & kLineHasNul) != 0 : true;
            if (!context) {
                out->emit(db->simple_id, line_base + lr.line, bytes, lr.len & kLineLenMask, may_have_nul);
            } else if (!context->feed((lr.len & kLineContext) == 0, line_base + lr.line, bytes, lr.len & kLineLenMask, may_have_nul)) {
                stop = true;
                break;
            }
        }
        // the reader goes on past the limit while trailing context is owed
        if (context && context->finished(line_base + r.num_lines)) stop = true;
        return 0;
    }

    std::vector<LineRec> unique_;

    int deliver_spans(const SegmentResult& r) {
        for (size_t i = 0; i < r.num_spans; i++) out->emit_span(line_base + r.spans[i].line, r.spans[i].start, r.spans[i].end);
        return 0;
    }

    int deliver_events(const SegmentResult& r, const uint8_t* host, ScanSlot* slot) {
        // events arrive grouped by pseudo-line in file order; inside a line they are grouped by DFA group
        struct Ev { uint32_t end; unsigned id; unsigned sm; };
        std::vector<Ev> evs;
        std::vector<unsigned> fired;
        // device-resident input: gather the distinct lines once
        std::vector<uint8_t> gathered;
        std::vector<unsigned long long> goff;
        std::vector<size_t> line_slot;   // per event -> index of its line in the gathered set
        if (!host && out->wants_lines() && r.num_events) {
            std::vector<uint32_t> starts, lens;
            unsigned long long total = 0;
            line_slot.resize(r.num_events);
            for (size_t i = 0; i < r.num_events; i++) {
                if (i == 0 || r.events[i].line != r.events[i - 1].line) {
                    starts.push_back(r.events[i].start); lens.push_back(r.events[i].len); goff.push_back(total); total += r.events[i].len + 1ull;
                }
                line_slot[i] = starts.size() - 1;
            }
            gathered.resize((size_t)total);
            int rc = slot_gather_lines(slot, starts.data(), lens.data(), starts.size(), gathered.data(), error);
            if (rc) return rc;
        }
        size_t i = 0;
        while (i < r.num_events && !stop) {
            size_t j = i;
            evs.clear();
            while (j < r.num_events && r.events[j].line == r.events[i].line) {
                uint32_t flat = r.events[j].report;
                for (uint32_t k = report_begin_flat[flat]; k < report_end_flat[flat]; k++)
                    evs.push_back(Ev{r.events[j].end, db->reports[k].id, db->reports[k].singlematch});
                j++;
            }
            // hs_scan order: by end offset (ties: by id); one report per (id, end); SINGLEMATCH ids once per block
            std::sort(evs.begin(), evs.end(), [](const Ev& a, const Ev& b) { return a.end != b.end ? a.end < b.end : a.id < b.id; });
            fired.clear();
            const EventRec& e0 = r.events[i];
            const uint8_t* bytes = host ? host + e0.start : (gathered.empty() ? nullptr : gathered.data() + goff[line_slot[i]]);
            for (size_t k = 0; k < evs.size(); k++) {
                if (k && evs[k].end == evs[k - 1].end && evs[k].id == evs[k - 1].id) continue;
                if (evs[k].sm) {
                    if (std::find(fired.begin(), fired.end(), evs[k].id) != fired.end()) continue;
                    fired.push_back(evs[k].id);
                }
                if (out->wants_ends()) out->emit_end(evs[k].id, line_base + e0.line, evs[k].end);
                else if (out->wants_lines()) out->emit(evs[k].id, line_base + e0.line, bytes, e0.len);
                else out->emit_count_only(1);
            }
            // hyperscanner.c:222: the limit is checked after all reports of the line
            if (limit_reached()) stop = true;
            i = j;
        }
        return 0;
    }
};

struct Params {
    const char* const* patterns;
    const unsigned* flags;
    const unsigned* ids;
    unsigned elements;
    hs_event cb;
    int buffer_size;
    int buffer_count;
    unsigned long long max_match;
    void* user_stream;
    EndsSink* ends = nullptr;   // gpugrep_match_ends(): end offsets instead of lines
    SpansSink* spans = nullptr;             // gpugrep_match_spans(): match spans of `span_program` instead of lines
    const PikeProgram* span_program = nullptr;
    bool invert = false;        // gpugrep_invert_scan_*(): deliver the pseudo-lines in which no pattern reports
    bool context_scan = false;  // gpugrep_context_scan_*(): lines around the selected ones too
    bool literal = false;       // gpugrep_literal_scan_*(): `patterns` are fixed strings (flags: CASELESS only, no ids)
    bool literal_reports = false;   // gpugrep_literal_report_scan_*(): fixed strings with ids, one record per (id, end)
    unsigned whole = 0;         // gpugrep_literal_whole_scan_*(): GPUGREP_WHOLE_WORD or GPUGREP_WHOLE_LINE
    uint32_t before = 0, after = 0;
    // the context stage runs only when lines are delivered (count-only scans ignore context)
    bool context() const { return context_scan && cb != nullptr && (before || after); }
};

// Largest prefix of [p, p+have) that ends on a pseudo-line boundary; 0 if none exists yet.
// `final`: end of data, everything is scanned.  limit = buffer_size - 1 (gzgets reads at most that many bytes).
size_t cut_point(const uint8_t* p, size_t have, bool final, size_t limit) {
    if (final) return have;
    const void* nl = memrchr(p, '\n', have);
    size_t cut = nl ? (size_t)((const uint8_t*)nl - p) + 1 : 0;
    size_t tail = have - cut;
    if (tail >= limit) cut += (tail / limit) * limit;
    return cut;
}

// slot_set_invert is weak (engine.hpp): absent only from CPU stand-ins of the engine without inverted scans (setup_job refuses
// inverted scans there).
void set_invert(ScanSlot* slot, bool invert) {
    if (slot_set_invert) slot_set_invert(slot, invert);
}
void set_context(ScanSlot* slot, const Params& pr) {
    if (slot_set_context) slot_set_context(slot, pr.context() ? pr.before : 0u, pr.context() ? pr.after : 0u);
}
void set_spans(ScanSlot* slot, const Params& pr) {
    if (slot_set_spans) slot_set_spans(slot, pr.span_program);
}
void set_literals(ScanSlot* slot, const Params& pr) {
    if (slot_set_literals) slot_set_literals(slot, pr.literal);
    if (slot_set_literal_reports) slot_set_literal_reports(slot, pr.literal_reports);
    if (slot_set_literal_whole) slot_set_literal_whole(slot, pr.whole);
}

int setup_job(const Params& pr, Job& job, Deliverer& out, unsigned long long weight = 0) {
    int rc = 0;
    if (pr.literal_reports) job.db = cached_literal_report_database(pr.patterns, pr.flags, pr.ids, pr.elements, rc, job.error);
    else if (pr.whole) job.db = cached_literal_whole_database(pr.patterns, pr.flags, pr.elements, rc, job.error);
    else if (pr.literal) job.db = cached_literal_database(pr.patterns, pr.flags, pr.elements, rc, job.error);
    else job.db = cached_database(pr.patterns, pr.flags, pr.ids, pr.elements, rc, job.error);
    if (job.db && !pr.literal && (pr.invert || pr.context_scan)) {
        // Which lines match does not depend on ids or SINGLEMATCH: once the set compiles as given, it is scanned as "every
        // pattern SINGLEMATCH, one id 0" (simple mode, so multi-id sets take the fast path too), CASELESS/DOTALL/MULTILINE kept.
        std::vector<unsigned> flags(pr.elements), ids(pr.elements, 0u);
        for (unsigned i = 0; i < pr.elements; i++) flags[i] = (pr.flags ? pr.flags[i] : 0u) | 8u;
        job.db = cached_database(pr.patterns, flags.data(), ids.data(), pr.elements, rc, job.error);
    }
    if (!job.db) {
        std::fprintf(stderr, "ERROR: Unable to create database. Exiting.\n");   // same text as hyperscanner.c:297
        return GPUGREP_DB;
    }
    if (pr.buffer_size < 2) { job.error = "buffer_size must be at least 2"; return GPUGREP_SCAN; }
    if (pr.invert && !slot_set_invert) { job.error = "this build of the engine has no inverted scan"; return GPUGREP_SCAN; }
    if (pr.context_scan && !slot_set_context) { job.error = "this build of the engine has no context lines"; return GPUGREP_SCAN; }
    if (pr.span_program && !slot_set_spans) { job.error = "this build of the engine has no span stage"; return GPUGREP_SCAN; }
    if (pr.literal && !slot_set_literals) { job.error = "this build of the engine has no fixed-string stage"; return GPUGREP_SCAN; }
    if (pr.literal_reports && !slot_set_literal_reports) { job.error = "this build of the engine has no fixed-string report stage"; return GPUGREP_SCAN; }
    if (pr.whole && !slot_set_literal_whole) { job.error = "this build of the engine has no whole-word / whole-line stage"; return GPUGREP_SCAN; }
    job.device_weight = weight;
    job.device = pick_device(weight, &job.device_charged);
    if (engine_select_device(job.device, job.error) != 0) {
        std::fprintf(stderr, "ERROR: Unable to allocate scratch space. Exiting. (%s)\n", job.error.c_str());
        return GPUGREP_SCRATCH;
    }
    job.ddb = engine_upload(job.db, job.error);
    if (!job.ddb) return GPUGREP_SCRATCH;
    job.buffer_size = pr.buffer_size;
    job.max_match = pr.max_match;
    job.out = &out;
    job.prepare();
    return 0;
}

int effective_batch(const Params& pr) {
    int bc = pr.buffer_count;
    if (pr.max_match > 0 && pr.max_match < (unsigned long long)(bc < 0 ? 0 : bc)) bc = (int)pr.max_match;   // hyperscanner.c:259-262
    return std::max(1, bc);
}

size_t clamp_limit(int buffer_size) {
    size_t limit = (size_t)buffer_size - 1;
    const size_t kMaxLimit = ((size_t)1 << 29);   // pseudo-lines longer than 512 MiB are split there (documented divergence)
    return std::min(limit, kMaxLimit);
}

// ---- file input -------------------------------------------------------------------------------------------
// Reader side of scan_file(): fills pinned slot buffers with consecutive segments (each ends on a pseudo-line boundary;
// the unfinished tail is carried into the next buffer) on its own thread, so that reading / inflating segment k+2
// overlaps the H2D + kernels of k+1 and the delivery of k.
struct SegmentQueue {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<int> free_slots;            // buffers the reader may fill
    std::vector<std::pair<int, size_t>> ready;   // (slot, segment bytes), FIFO
    bool done = false;                      // reader reached the end of the input
    bool abort = false;                     // consumer asked the reader to stop
};

// One shard of a scan: byte range [begin, end) of a plain file; its results go to `collect` (null: count only).
struct ShardSpec {
    size_t begin = 0, end = 0;
    ShardResults* collect = nullptr;
    bool count_only = false;
};

int scan_file(const char* path, const Params& pr, gpugrep_stats* stats_out, const ShardSpec* shard = nullptr) {
    double t0 = now_ms();
    Deliverer own(pr.cb, effective_batch(pr));
    Deliverer collecting(shard ? shard->collect : nullptr);
    Deliverer counting(nullptr, 1);
    Deliverer& out = !shard ? own : (shard->count_only ? counting : collecting);
    Job job;
    unsigned long long weight = 0;   // bytes on disk: the scan goes to the least loaded device
    {
        struct stat sb;
        if (::stat(path, &sb) == 0 && S_ISREG(sb.st_mode)) weight = shard ? shard->end - shard->begin : (unsigned long long)sb.st_size;
    }
    int rc = setup_job(pr, job, out, weight);
    if (rc) { set_last_error(job.error); return rc; }
    ContextFilter context(&out, pr.before, pr.after, pr.max_match, shard != nullptr);
    if (pr.context()) job.context = &context;
    std::string err;
    auto src = shard ? open_plain_range(path, shard->begin, shard->end, err) : open_byte_source(path, err);
    if (!src) { set_last_error(err); return GPUGREP_GZ_OPEN; }

    const size_t limit = clamp_limit(pr.buffer_size);
    // Segment (= pinned slot) size and admission.  Every slot costs pinned memory that has to be allocated and pinned first:
    // a cold process scanning 16 plain files at once (multiscanner: one host thread per file) paid seconds for 45 slots of
    // 64 MiB.  Four plain-file scans at a time already saturate the PCIe link, so the others wait their turn; compressed
    // sources deliver ~1 GB/s per file, all run at once (the decoders are the work) and take small slots.
    const bool plain = std::strcmp(src->kind(), "plain") == 0;
    struct Admission {   // per device: files are spread round-robin over the visible GPUs
        bool held;
        int device;
        explicit Admission(bool gate) : held(gate), device(engine_current_device() & (kMaxDevices - 1)) {
            if (!held) return;
            std::unique_lock<std::mutex> lk(g_plain_mu);
            g_plain_cv.wait(lk, [this] { return g_plain_scans[device] < kMaxPlainScans; });
            g_plain_scans[device]++;
        }
        ~Admission() {
            if (!held) return;
            { std::lock_guard<std::mutex> lk(g_plain_mu); g_plain_scans[device]--; }
            g_plain_cv.notify_all();
        }
    } admission(plain);
    size_t chunk = env_mb("GPUGREP_CHUNK_MB", plain ? 32 : 8);
    chunk = std::max(chunk, 2 * limit + 4096);
    chunk = std::min(chunk, kMaxSegmentBytes);
    constexpr int kSlots = 3;
    ScanSlot* slots[kSlots] = {nullptr, nullptr, nullptr};
    uint8_t* bufs[kSlots] = {nullptr, nullptr, nullptr};
    bool ok = true;
    for (int i = 0; i < kSlots && ok; i++) {
        slots[i] = engine_acquire_slot(err);
        ok = slots[i] != nullptr;
        if (ok) { bufs[i] = slot_host_buffer(slots[i], chunk, err); ok = bufs[i] != nullptr; }
    }
    if (!ok) {
        for (ScanSlot* sl : slots) engine_release_slot(sl);
        set_last_error(err);
        return GPUGREP_SCRATCH;
    }

    const bool count_only = !out.wants_lines() && pr.max_match == 0 && !job.wants_events();
    for (ScanSlot* sl : slots) {
        slot_set_want_records(sl, !count_only);
        set_invert(sl, pr.invert);
        set_context(sl, pr);
        set_spans(sl, pr);
        set_literals(sl, pr);
    }
    SegmentQueue q;
    for (int i = 0; i < kSlots; i++) q.free_slots.push_back(i);
    std::thread reader([&] {
        std::vector<uint8_t> carry;
        bool eof = false;
        // the first segments are short so that the copy engine and the kernels start early (a 128 MiB file would otherwise
        // spend a third of its time reading the first 64 MiB with the GPU idle)
        const size_t floor_bytes = 2 * limit + 4096;
        size_t target = std::min(chunk, std::max(floor_bytes, (size_t)8 << 20));
        while (!eof) {
            int slot;
            {
                std::unique_lock<std::mutex> lk(q.mu);
                q.cv.wait(lk, [&] { return q.abort || !q.free_slots.empty(); });
                if (q.abort) break;
                slot = q.free_slots.back();
                q.free_slots.pop_back();
            }
            uint8_t* buf = bufs[slot];
            if (!carry.empty()) std::memcpy(buf, carry.data(), carry.size());
            size_t have = carry.size();
            size_t cut = 0;
            while (true) {
                size_t got = src->read(buf + have, target - have);
                have += got;
                if (got == 0) eof = true;
                cut = cut_point(buf, have, eof, limit);
                if (cut > 0 || eof || have == target) break;
            }
            target = std::min(chunk, target * 4);
            if (cut == 0 && !eof) cut = have;   // cannot happen (chunk >= 2*limit): defensive
            carry.assign(buf + cut, buf + have);
            std::lock_guard<std::mutex> lk(q.mu);
            if (cut > 0) q.ready.emplace_back(slot, cut);
            else q.free_slots.push_back(slot);
            q.cv.notify_all();
        }
        std::lock_guard<std::mutex> lk(q.mu);
        q.done = true;
        q.cv.notify_all();
    });

    auto release = [&](int slot) {
        std::lock_guard<std::mutex> lk(q.mu);
        q.free_slots.push_back(slot);
        q.cv.notify_all();
    };
    int inflight = -1;
    size_t inflight_len = 0;
    bool tuned = false;
    while (!job.stop && rc == 0) {
        int slot = -1;
        size_t len = 0;
        {
            std::unique_lock<std::mutex> lk(q.mu);
            q.cv.wait(lk, [&] { return !q.ready.empty() || q.done; });
            if (q.ready.empty()) break;
            slot = q.ready.front().first;
            len = q.ready.front().second;
            q.ready.erase(q.ready.begin());
        }
        job.stats.bytes_scanned += len;
        if (!tuned) {
            job.dpf = tuned_prefilter(job.db, bufs[slot], len, job.error, nullptr, /*reuse_sibling=*/true);
            job.tune_head.assign(bufs[slot], bufs[slot] + std::min(len, kSampleBytes / 2));
            tuned = true;
        }
        rc = slot_submit(slots[slot], *job.ddb, job.dpf.get(), bufs[slot], nullptr, len, pr.buffer_size, nullptr, job.error);
        if (rc) { release(slot); break; }
        if (inflight >= 0) {
            SegmentResult res;
            rc = slot_collect(slots[inflight], res, job.error);
            if (rc == 0) rc = job.deliver(res, bufs[inflight], slots[inflight]);
            if (rc == 0 && job.drifted(res, inflight_len)) job.retune(bufs[inflight] + inflight_len / 2, inflight_len - inflight_len / 2);
            release(inflight);
        }
        inflight = slot;
        inflight_len = len;
    }
    if (inflight >= 0) {
        SegmentResult res;
        int rc2 = slot_collect(slots[inflight], res, job.error);   // always drain the GPU before the buffers are reused
        if (rc == 0) rc = rc2;
        if (rc == 0 && !job.stop) rc = job.deliver(res, bufs[inflight], slots[inflight]);
        release(inflight);
    }
    {
        std::lock_guard<std::mutex> lk(q.mu);
        q.abort = true;
        q.cv.notify_all();
    }
    reader.join();
    out.flush();   // hyperscanner.c:311-313
    for (ScanSlot* sl : slots) engine_release_slot(sl);
    job.stats.matches = out.count();
    job.stats.wall_ms = now_ms() - t0;
    if (stats_out) *stats_out = job.stats;
    if (rc) {
        std::fprintf(stderr, "ERROR: Unable to scan buffer. Exiting. (%s)\n", job.error.c_str());
        set_last_error(job.error);
    } else {
        set_last_error("");
    }
    return rc;
}

// ---- memory input -----------------------------------------------------------------------------------------
// Find the cut for a device-resident window by pulling its tail to the host.
int device_cut(const uint8_t* dev, size_t have, bool final, size_t limit, size_t& cut, std::string& error) {
    if (final) { cut = have; return 0; }
    std::vector<uint8_t> tail;
    size_t span = std::min<size_t>(have, 1 << 20);
    while (true) {
        tail.resize(span);
        if (cudaMemcpy(tail.data(), dev + have - span, span, cudaMemcpyDeviceToHost) != cudaSuccess) { error = "cudaMemcpy failed while locating a segment boundary"; return GPUGREP_SCAN; }
        // prefer a line end that leaves the next segment 16-byte aligned (the kernels use 16-byte loads)
        size_t base = have - span;
        size_t best = 0, any = 0;
        for (size_t p = span; p > 0; p--) {
            if (tail[p - 1] != '\n') continue;
            if (!any) any = base + p;
            if (((base + p) & 15) == 0) { best = base + p; break; }
            if (span - p > (64 << 10)) break;
        }
        if (best || any) {
            size_t c = best ? best : any;
            size_t rest = have - c;
            if (!best && rest >= limit) c += (rest / limit) * limit;
            cut = c;
            return 0;
        }
        if (span == have) { cut = (have / limit) * limit; return 0; }
        span = std::min(have, span * 8);
    }
}

int scan_memory(const uint8_t* data, size_t size, int location, const Params& pr, gpugrep_stats* stats_out, const ShardSpec* shard = nullptr) {
    double t0 = now_ms();
    Deliverer own(pr.cb, effective_batch(pr));
    own.set_ends(pr.ends);
    own.set_spans(pr.spans);
    Deliverer collecting(shard ? shard->collect : nullptr);
    Deliverer counting(nullptr, 1);
    Deliverer& out = !shard ? own : (shard->count_only ? counting : collecting);
    Job job;
    int rc = setup_job(pr, job, out, size);
    if (rc) { set_last_error(job.error); return rc; }
    ContextFilter context(&out, pr.before, pr.after, pr.max_match, shard != nullptr);
    if (pr.context()) job.context = &context;
    std::string err;
    const size_t limit = clamp_limit(pr.buffer_size);
    const bool on_device = location == GPUGREP_LOC_DEVICE;
    size_t chunk = on_device ? env_mb("GPUGREP_DEVICE_SEGMENT_MB", 2048) : env_mb("GPUGREP_CHUNK_MB", 64);
    chunk = std::max(chunk, 2 * limit + 4096);
    chunk = std::min(chunk, kMaxSegmentBytes);
    bool pinned = false;
    if (!on_device && size) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, data) == cudaSuccess) pinned = attr.type == cudaMemoryTypeHost;
        else cudaGetLastError();
    }
    ScanSlot* slots[2] = {engine_acquire_slot(err, location != GPUGREP_LOC_DEVICE), engine_acquire_slot(err, location != GPUGREP_LOC_DEVICE)};
    if (!slots[0] || !slots[1]) { engine_release_slot(slots[0]); engine_release_slot(slots[1]); set_last_error(err); return GPUGREP_SCRATCH; }
    const bool count_only = !out.wants_lines() && pr.max_match == 0 && !job.wants_events();
    for (ScanSlot* sl : slots) {
        slot_set_want_records(sl, !count_only);
        set_invert(sl, pr.invert);
        set_context(sl, pr);
        set_spans(sl, pr);
        set_literals(sl, pr);
    }
    const uint8_t* seg_host[2] = {nullptr, nullptr};
    const uint8_t* seg_dev[2] = {nullptr, nullptr};
    size_t seg_len[2] = {0, 0};
    int k = 0, inflight = -1;
    bool tuned = false;
    std::vector<uint8_t> sample;
    // device-resident input: all segment ends come from one small kernel instead of one synchronous copy per segment
    std::vector<size_t> dev_cuts;
    size_t dev_cut_index = 0;
    std::vector<uint8_t> head;   // device-resident input: its first 64 KiB, enough for the fingerprint of the tuning sample
    if (on_device && size) {
        if (size > chunk) chunk = std::min(chunk, kMaxSegmentBytes - ((size_t)16 << 20));
        head.resize(std::min<size_t>(size, 64 << 10));
        if (slot_probe_input(slots[0], data, size, chunk, dev_cuts, head.data(), head.size(), pr.user_stream, job.error) != 0) {
            engine_release_slot(slots[0]); engine_release_slot(slots[1]);
            set_last_error(job.error);
            return GPUGREP_SCAN;
        }
    }
    // Collect segment `idx` and deliver its results.  A large segment in which the fast path hit one of its bounds (a line
    // too long for it, a candidate / record overflow) is not sent down the general path as a whole: the same bytes are
    // scanned again in 64 MiB pieces on this slot, one after the other, and only the piece with the problem pays for it.
    // A general-path segment with more match events than one segment holds is cut the same way (device-resident input
    // comes in segments of up to 2 GiB; a 64 MiB piece is what host input gets anyway).
    constexpr size_t kSplitAbove = (size_t)128 << 20, kSplitPiece = (size_t)64 << 20;
    auto finish = [&](int idx) -> int {
        SegmentResult res;
        int r = slot_collect(slots[idx], res, job.error, kSplitAbove);
        if (r == kSplitSegment) {
            const uint8_t* base_host = seg_host[idx];
            const uint8_t* base_dev = seg_dev[idx];
            const size_t len = seg_len[idx];
            job.stats.split_segments++;
            for (size_t p = 0; p < len && !job.stop;) {
                const size_t have = std::min(kSplitPiece, len - p);
                const bool last = p + have == len;
                size_t cut = 0;
                if (on_device) {
                    r = device_cut(base_dev + p, have, last, limit, cut, job.error);
                    if (r) return r;
                } else {
                    cut = cut_point(base_host + p, have, last, limit);
                }
                if (cut == 0) cut = have;
                const uint8_t* host_src = nullptr;
                if (!on_device) {
                    host_src = base_host + p;
                    if (!pinned) {
                        uint8_t* stage = slot_host_buffer(slots[idx], std::max(chunk, kSplitPiece), job.error);
                        if (!stage) return GPUGREP_SCRATCH;
                        std::memcpy(stage, base_host + p, cut);
                        host_src = stage;
                    }
                }
                r = slot_submit(slots[idx], *job.ddb, job.dpf.get(), host_src, on_device ? base_dev + p : nullptr, cut, pr.buffer_size, pr.user_stream, job.error);
                if (r) return r;
                r = slot_collect(slots[idx], res, job.error);
                if (r == 0) r = job.deliver(res, on_device ? nullptr : base_host + p, slots[idx]);
                if (r) return r;
                p += cut;
            }
            return 0;
        }
        if (r == 0) r = job.deliver(res, seg_host[idx], slots[idx]);
        if (r == 0 && job.drifted(res, seg_len[idx])) {
            // sample of the drifting region: host bytes as they are, device-resident text through one small copy
            const size_t half = seg_len[idx] / 2, span = std::min(seg_len[idx] - half, kSampleBytes / 2);
            if (seg_host[idx]) {
                job.retune(seg_host[idx] + half, span);
            } else {
                std::vector<uint8_t> region(span);
                if (cudaMemcpy(region.data(), seg_dev[idx] + half, span, cudaMemcpyDeviceToHost) == cudaSuccess) {
                    job.stats.d2h_bytes += span;
                    job.retune(region.data(), span);
                }
            }
        }
        return r;
    };
    size_t pos = 0;
    while (pos < size && !job.stop && rc == 0) {
        size_t have = std::min(chunk, size - pos);
        bool final = pos + have == size;
        size_t cut = 0;
        if (on_device && !dev_cuts.empty()) {
            cut = dev_cuts[dev_cut_index++] - pos;
        } else if (on_device) {
            rc = device_cut(data + pos, have, final, limit, cut, job.error);
            if (rc) break;
        } else {
            cut = cut_point(data + pos, have, final, limit);
        }
        if (cut == 0) cut = have;   // defensive: chunk >= 2*limit guarantees progress
        const uint8_t* host_src = nullptr;
        if (!on_device) {
            if (pinned) host_src = data + pos;
            else {
                uint8_t* stage = slot_host_buffer(slots[k], chunk, job.error);
                if (!stage) { rc = GPUGREP_SCRATCH; break; }
                std::memcpy(stage, data + pos, cut);
                host_src = stage;
            }
        }
        if (!tuned) {
            tuned = true;
            if (on_device) {
                const size_t sample_len = std::min(cut, kSampleBytes);
                job.stats.d2h_bytes += head.size();
                job.tune_head.assign(head.begin(), head.begin() + std::min(head.size(), kSampleBytes / 2));
                job.dpf = tuned_prefilter(job.db, head.data(), sample_len, job.error, [&]() -> const uint8_t* {
                    sample.resize(sample_len);
                    if (cudaMemcpy(sample.data(), data, sample_len, cudaMemcpyDeviceToHost) != cudaSuccess) return nullptr;
                    job.stats.d2h_bytes += sample_len;
                    return sample.data();
                });
            } else {
                job.dpf = tuned_prefilter(job.db, data, cut, job.error);
                job.tune_head.assign(data, data + std::min(cut, kSampleBytes / 2));
            }
        }
        rc = slot_submit(slots[k], *job.ddb, job.dpf.get(), host_src, on_device ? data + pos : nullptr, cut, pr.buffer_size, pr.user_stream, job.error);
        if (rc) break;
        seg_host[k] = on_device ? nullptr : data + pos;
        job.stats.bytes_scanned += cut;
        pos += cut;
        if (inflight >= 0) {
            rc = finish(inflight);
            inflight = -1;
        }
        inflight = k;
        seg_len[k] = cut;
        seg_dev[k] = on_device ? data + (pos - cut) : nullptr;
        k ^= 1;
    }
    if (inflight >= 0) {
        int rc2 = finish(inflight);   // always drain the GPU
        if (rc == 0) rc = rc2;
    }
    out.flush();
    engine_release_slot(slots[0]);
    engine_release_slot(slots[1]);
    job.stats.matches = out.count();
    job.stats.wall_ms = now_ms() - t0;
    if (stats_out) *stats_out = job.stats;
    set_last_error(rc ? job.error : "");
    if (rc) std::fprintf(stderr, "ERROR: Unable to scan buffer. Exiting. (%s)\n", job.error.c_str());
    return rc;
}

// ---- one input over several GPUs (SURVEY.md section 8e-2) ----------------------------------------------------
// $GPUGREP_DEVICES = "all" or a comma-separated list: hyperscan(path) on a plain file and gpugrep_scan_buffer on host
// memory split the input into one newline-aligned byte range per device, scan the ranges concurrently (one host thread
// and one pipeline per device), and merge on the calling thread: exclusive prefix sum of the shard line counts, line
// numbers rebased, results in range order, the max_match_count rule applied to the merged sequence, callbacks batched
// exactly as for a single device.  The only data exchanged between the shards are G line counts.
std::vector<int> shard_devices() {
    std::vector<int> out;
    const char* e = std::getenv("GPUGREP_DEVICES");
    if (!e || !*e) return out;
    const int count = engine_device_count();
    if (count < 1) return out;
    if (std::strcmp(e, "all") == 0) {
        for (int d = 0; d < count; d++) out.push_back(d);
    } else {
        for (const char* p = e; *p;) {
            char* endp = nullptr;
            long v = std::strtol(p, &endp, 10);
            if (endp == p) break;
            if (v >= 0 && v < count) out.push_back((int)v);
            p = *endp == ',' ? endp + 1 : endp;
        }
    }
    if (out.size() < 2) out.clear();
    return out;
}

// below 32 MiB per shard a second device does not pay for its pipeline start ($GPUGREP_MIN_SHARD_BYTES: test hook)
size_t min_shard_bytes() {
    if (const char* e = std::getenv("GPUGREP_MIN_SHARD_BYTES")) {
        if (*e) return std::max<size_t>(1, (size_t)std::strtoull(e, nullptr, 10));
    }
    return (size_t)32 << 20;
}

// `bounds`: G+1 newline-aligned offsets; `run(g, spec, stats)` scans shard g.
int scan_sharded(const std::vector<int>& devices, const std::vector<size_t>& bounds, const Params& pr, gpugrep_stats* stats_out,
                 const std::function<int(size_t, const ShardSpec&, gpugrep_stats*)>& run) {
    const double t0 = now_ms();
    const size_t G = bounds.size() - 1;
    // a NULL callback without a limit only counts; everything else needs the results themselves for the ordered merge
    const bool count_only = pr.cb == nullptr && pr.max_match == 0;
    std::vector<ShardResults> results(G);
    std::vector<gpugrep_stats> stats(G);
    std::vector<int> rcs(G, 0);
    std::vector<std::string> errors(G);
    std::vector<std::thread> workers;
    for (size_t g = 0; g < G; g++) {
        workers.emplace_back([&, g] {
            t_device_override = devices[g % devices.size()];
            ShardSpec spec;
            spec.begin = bounds[g];
            spec.end = bounds[g + 1];
            spec.collect = &results[g];
            spec.count_only = count_only;
            std::memset(&stats[g], 0, sizeof(gpugrep_stats));
            rcs[g] = spec.end > spec.begin ? run(g, spec, &stats[g]) : 0;
            if (rcs[g]) errors[g] = gpugrep_last_error();
        });
    }
    for (auto& w : workers) w.join();
    gpugrep_stats total;
    std::memset(&total, 0, sizeof(total));
    for (size_t g = 0; g < G; g++) {
        if (rcs[g]) { set_last_error(errors[g]); return rcs[g]; }
        total.bytes_scanned += stats[g].bytes_scanned; total.lines += stats[g].lines; total.candidates += stats[g].candidates;
        total.h2d_bytes += stats[g].h2d_bytes; total.d2h_bytes += stats[g].d2h_bytes; total.gpu_ms += stats[g].gpu_ms;
        total.stream_kernel_ms += stats[g].stream_kernel_ms; total.launches += stats[g].launches;
        total.stream_launches += stats[g].stream_launches; total.segments += stats[g].segments; total.path |= stats[g].path;
        total.nul_segments += stats[g].nul_segments;
    }
    // ordered merge on the calling thread
    Deliverer out(pr.cb, effective_batch(pr));
    // context lines: the shards pass on every candidate (id GPUGREP_CONTEXT_ID), and the merge filters them, so that a
    // window may reach across a shard boundary
    ContextFilter context(&out, pr.before, pr.after, pr.max_match, false);
    unsigned long long line_base = 0;
    bool stop = false;
    for (size_t g = 0; g < G && !stop; g++) {
        if (count_only) {
            out.emit_count_only(stats[g].matches);
        } else if (pr.context()) {
            const auto& recs = results[g].records;
            for (size_t i = 0; i < recs.size() && !stop; i++) {
                const char* text = results[g].text.data() + recs[i].offset;
                stop = !context.feed(recs[i].id != GPUGREP_CONTEXT_ID, line_base + recs[i].line, (const uint8_t*)text, std::strlen(text), false);
            }
            if (context.finished(line_base + stats[g].lines)) stop = true;
        } else {
            const auto& recs = results[g].records;
            for (size_t i = 0; i < recs.size() && !stop;) {
                size_t j = i;
                for (; j < recs.size() && recs[j].line == recs[i].line; j++) {
                    if (pr.cb) out.emit_text(recs[j].id, line_base + recs[j].line, results[g].text.data() + recs[j].offset);
                    else out.emit_count_only(1);
                }
                // hyperscanner.c:222: the limit is checked after all reports of a line
                if (pr.max_match > 0 && out.count() >= pr.max_match) stop = true;
                i = j;
            }
        }
        line_base += stats[g].lines;
    }
    out.flush();
    total.matches = out.count();
    total.wall_ms = now_ms() - t0;
    if (stats_out) *stats_out = total;
    set_last_error("");
    return 0;
}

// Shard boundaries of a host buffer: k * size / G advanced to just past the next '\n'.
std::vector<size_t> buffer_bounds(const uint8_t* data, size_t size, size_t shards) {
    std::vector<size_t> b;
    for (size_t g = 0; g <= shards; g++) b.push_back(gpugrep_shard_begin(data, size, (unsigned)g, (unsigned)shards));
    return b;
}

// The same for a file, reading a window at every boundary.
std::vector<size_t> file_bounds(const char* path, size_t size, size_t shards) {
    std::vector<size_t> b{0};
    FILE* f = std::fopen(path, "rb");
    if (!f) return {};
    std::vector<char> window((size_t)1 << 20);
    for (size_t g = 1; g < shards; g++) {
        size_t pos = (size_t)(((unsigned __int128)size * g) / shards);
        size_t found = size;
        // the byte before pos may already be a newline
        if (pos > 0 && fseeko(f, (off_t)(pos - 1), SEEK_SET) == 0) {
            size_t at = pos - 1;
            while (true) {
                size_t got = std::fread(window.data(), 1, window.size(), f);
                if (got == 0) break;
                const void* nl = std::memchr(window.data(), '\n', got);
                if (nl) { found = at + (size_t)((const char*)nl - window.data()) + 1; break; }
                at += got;
            }
        }
        b.push_back(std::max(found, b.back()));
    }
    std::fclose(f);
    b.push_back(size);
    return b;
}

}  // namespace

// hyperscan(path): one device, or - plain files, $GPUGREP_DEVICES - one byte range per device.
static int scan_path(const char* path, const Params& pr, gpugrep_stats* stats) {
    const std::vector<int> devices = shard_devices();
    if (!devices.empty() && pr.buffer_size >= 2) {
        const size_t size = plain_regular_file_size(path);
        if (size >= 2 * min_shard_bytes()) {
            const size_t shards = std::min(devices.size(), size / min_shard_bytes());
            const std::vector<size_t> bounds = file_bounds(path, size, shards);
            if (bounds.size() == shards + 1)
                return scan_sharded(devices, bounds, pr, stats, [&](size_t, const ShardSpec& spec, gpugrep_stats* st) { return scan_file(path, pr, st, &spec); });
        }
    }
    return scan_file(path, pr, stats);
}

// gpugrep_scan_buffer / gpugrep_invert_scan_buffer: one device, or - host memory, $GPUGREP_DEVICES - one byte range per device.
static int scan_buffer(const void* data, size_t size, int location, const Params& pr, gpugrep_stats* stats) {
    if (location == GPUGREP_LOC_HOST) {
        const std::vector<int> devices = shard_devices();
        if (!devices.empty() && size >= 2 * min_shard_bytes() && pr.buffer_size >= 2) {
            const size_t shards = std::min(devices.size(), size / min_shard_bytes());
            const std::vector<size_t> bounds = buffer_bounds((const uint8_t*)data, size, shards);
            return scan_sharded(devices, bounds, pr, stats, [&](size_t, const ShardSpec& spec, gpugrep_stats* st) {
                return scan_memory((const uint8_t*)data + spec.begin, spec.end - spec.begin, GPUGREP_LOC_HOST, pr, st, &spec);
            });
        }
    }
    return scan_memory((const uint8_t*)data, size, location, pr, stats);
}
}  // namespace gpugrep

extern "C" {

// Replaces reference hyperscanner.c:248-326.
int hyperscan(char* file_name, const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
              const unsigned int elements, hs_event on_event, const int buffer_size, int buffer_count, unsigned long long max_match_count) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    return gpugrep::scan_path(file_name, pr, nullptr);
}

int gpugrep_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
                      unsigned int elements, hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                      gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_scan_buffer(const void* data, size_t size, int location, const char* const* patterns, const unsigned int* pattern_flags,
                        const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                        unsigned long long max_match_count, void* stream, gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_invert_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
                             unsigned int elements, hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                             gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    pr.invert = true;
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_invert_scan_buffer(const void* data, size_t size, int location, const char* const* patterns, const unsigned int* pattern_flags,
                               const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                               unsigned long long max_match_count, void* stream, gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    pr.invert = true;
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_context_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
                              unsigned int elements, hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                              unsigned int before, unsigned int after, int invert, gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_context_scan_buffer(const void* data, size_t size, int location, const char* const* patterns, const unsigned int* pattern_flags,
                                const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                                unsigned long long max_match_count, unsigned int before, unsigned int after, int invert, void* stream,
                                gpugrep_stats* stats) {
    gpugrep::Params pr{patterns, pattern_flags, pattern_ids, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_literal_scan_file(const char* file_name, const char* const* literals, const unsigned int* literal_flags, unsigned int elements,
                              hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count, unsigned int before,
                              unsigned int after, int invert, gpugrep_stats* stats) {
    gpugrep::Params pr{literals, literal_flags, nullptr, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    pr.literal = true;
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_literal_scan_buffer(const void* data, size_t size, int location, const char* const* literals, const unsigned int* literal_flags,
                                unsigned int elements, hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                                unsigned int before, unsigned int after, int invert, void* stream, gpugrep_stats* stats) {
    gpugrep::Params pr{literals, literal_flags, nullptr, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    pr.literal = true;
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_literal_whole_scan_file(const char* file_name, const char* const* literals, const unsigned int* literal_flags, unsigned int elements,
                                    unsigned int whole, hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                                    unsigned int before, unsigned int after, int invert, gpugrep_stats* stats) {
    if (whole != GPUGREP_WHOLE_WORD && whole != GPUGREP_WHOLE_LINE) { gpugrep::set_last_error("whole must be GPUGREP_WHOLE_WORD or GPUGREP_WHOLE_LINE"); return GPUGREP_DB; }
    gpugrep::Params pr{literals, literal_flags, nullptr, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    pr.literal = true;
    pr.whole = whole;
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_literal_whole_scan_buffer(const void* data, size_t size, int location, const char* const* literals, const unsigned int* literal_flags,
                                      unsigned int elements, unsigned int whole, hs_event on_event, int buffer_size, int buffer_count,
                                      unsigned long long max_match_count, unsigned int before, unsigned int after, int invert, void* stream,
                                      gpugrep_stats* stats) {
    if (whole != GPUGREP_WHOLE_WORD && whole != GPUGREP_WHOLE_LINE) { gpugrep::set_last_error("whole must be GPUGREP_WHOLE_WORD or GPUGREP_WHOLE_LINE"); return GPUGREP_DB; }
    gpugrep::Params pr{literals, literal_flags, nullptr, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    pr.literal = true;
    pr.whole = whole;
    pr.invert = invert != 0;
    pr.context_scan = true;
    pr.before = before;
    pr.after = after;
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_literal_report_scan_file(const char* file_name, const char* const* literals, const unsigned int* literal_flags,
                                     const unsigned int* literal_ids, unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                                     unsigned long long max_match_count, gpugrep_stats* stats) {
    gpugrep::Params pr{literals, literal_flags, literal_ids, elements, on_event, buffer_size, buffer_count, max_match_count, nullptr};
    pr.literal = true;
    pr.literal_reports = true;
    return gpugrep::scan_path(file_name, pr, stats);
}

int gpugrep_literal_report_scan_buffer(const void* data, size_t size, int location, const char* const* literals, const unsigned int* literal_flags,
                                       const unsigned int* literal_ids, unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                                       unsigned long long max_match_count, void* stream, gpugrep_stats* stats) {
    gpugrep::Params pr{literals, literal_flags, literal_ids, elements, on_event, buffer_size, buffer_count, max_match_count, stream};
    pr.literal = true;
    pr.literal_reports = true;
    return gpugrep::scan_buffer(data, size, location, pr, stats);
}

int gpugrep_match_ends(const void* data, size_t size, int location, const char* const* patterns, const unsigned int* pattern_flags,
                       const unsigned int* pattern_ids, unsigned int elements, int buffer_size, gpugrep_match_end* out, size_t capacity,
                       size_t* count, gpugrep_stats* stats) {
    // every end is wanted: without SINGLEMATCH the set is scanned on the general path, whose records carry the offsets
    std::vector<unsigned> flags(elements);
    for (unsigned i = 0; i < elements; i++) flags[i] = (pattern_flags ? pattern_flags[i] : 0u) & ~8u;
    gpugrep::EndsSink sink{out, out ? capacity : 0};
    gpugrep::Params pr{patterns, flags.data(), pattern_ids, elements, nullptr, buffer_size, 1, 0, nullptr, &sink};
    const int rc = gpugrep::scan_memory((const uint8_t*)data, size, location, pr, stats);
    if (count) *count = sink.count;
    return rc;
}

int gpugrep_match_spans(const void* data, size_t size, int location, const char* pattern, int buffer_size, gpugrep_match_span* out,
                        size_t capacity, size_t* count, gpugrep_stats* stats) {
    if (count) *count = 0;
    gpugrep::PikeProgram program;
    if (!gpugrep::build_pike_program(pattern, program)) {
        gpugrep::set_last_error("the pattern is not accepted by gpugrep_span_exact");
        return GPUGREP_DB;
    }
    // compiled like the reference's re.compile(pattern): no flags (the automata only check that the pattern compiles)
    const unsigned flags = 0, id = 0;
    gpugrep::SpansSink sink{out, out ? capacity : 0};
    gpugrep::Params pr{&pattern, &flags, &id, 1, nullptr, buffer_size, 1, 0, nullptr};
    pr.spans = &sink;
    pr.span_program = &program;
    const int rc = gpugrep::scan_memory((const uint8_t*)data, size, location, pr, stats);
    if (count) *count = sink.count;
    return rc;
}

size_t gpugrep_shard_begin(const void* data, size_t size, unsigned int rank, unsigned int world) {
    if (world == 0 || rank == 0) return 0;
    if (rank >= world) return size;
    size_t pos = (size_t)(((unsigned __int128)size * rank) / world);
    if (pos >= size) return size;
    if (pos > 0 && ((const uint8_t*)data)[pos - 1] == '\n') return pos;
    const void* nl = std::memchr((const uint8_t*)data + pos, '\n', size - pos);
    return nl ? (size_t)((const uint8_t*)nl - (const uint8_t*)data) + 1 : size;
}

// A callback that drops its batch: lets benchmarks exercise the full delivery path (line copies into result slots)
// without a Python frame per batch.
void gpugrep_discard_results(hyperscanner_result_t* results, int result_count) { (void)results; (void)result_count; }

// The host ingest alone (no GPU work): what the scan of `file_name` would read, as a byte count and an FNV-1a hash.
int gpugrep_ingest_probe(const char* file_name, unsigned long long* text_bytes, unsigned long long* text_hash) {
    std::string error;
    auto src = gpugrep::open_byte_source(file_name, error);
    if (!src) {
        gpugrep::set_last_error(error);
        return 6;
    }
    std::vector<uint8_t> buf((size_t)8 << 20);
    unsigned long long total = 0, hash = 1469598103934665603ull;
    for (;;) {
        const size_t got = src->read(buf.data(), buf.size());
        if (got == 0) break;
        // (eight bytes at a time: the hash must not be what limits the measurement)
        size_t i = 0;
        for (; i + 8 <= got; i += 8) {
            unsigned long long w;
            std::memcpy(&w, buf.data() + i, 8);
            hash = (hash ^ w) * 1099511628211ull;
        }
        for (; i < got; i++) hash = (hash ^ buf[i]) * 1099511628211ull;
        total += got;
    }
    if (text_bytes) *text_bytes = total;
    if (text_hash) *text_hash = hash;
    return 0;
}

void gpugrep_set_device(int device) { gpugrep::g_device_override.store(device); }
void gpugrep_set_zstd_path(const char* path) { if (path) gpugrep::set_zstd_library_path(path); }

}  // extern "C"
