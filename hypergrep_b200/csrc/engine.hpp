// CUDA engine interface (host side).  The kernels replace the reference's per-line loop
// gzgets -> hs_scan -> hs_callback (reference hyperscanner.c:198-226, 83-102) for one device-resident segment
// of (decompressed) file bytes that starts at a pseudo-line start and ends at a pseudo-line end.
#pragma once
#include <cstddef>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "database.hpp"

namespace gpugrep {

// One matched pseudo-line (simple mode: every pattern SINGLEMATCH, one shared id).
struct LineRec {
    uint32_t line;    // pseudo-line index inside the segment
    uint32_t start;   // byte offset of the pseudo-line inside the segment
    uint32_t len;     // bytes, trailing '\n' included when present; bit 31 (fast path only): the line contains NUL bytes;
                      // bit 30 (scans with context lines): an output line that is not selected
};
// (fast-path lines are shorter than 128 KiB and pseudo-lines at most 2^29 bytes: bit 30 is free)
constexpr uint32_t kLineLenMask = 0x3fffffffu;
constexpr uint32_t kLineHasNul = 0x80000000u;
constexpr uint32_t kLineContext = 0x40000000u;
constexpr uint32_t kLineInvalid = 0xffffffffu;   // fast path: repeat of a line already reported, or a failed NUL re-check

// One automaton report (general mode): some accept set fired at `end` inside pseudo-line `line`.
struct EventRec {
    uint32_t line, start, len;
    uint32_t end;      // match end offset relative to the scanned block (after leading-NUL stripping)
    uint32_t report;   // index into Database::report_begin flattened over groups (DeviceDb::accept_base)
};

// One match span (slot_set_spans): [start, end) relative to the scanned block of pseudo-line `line` (after leading-NUL
// stripping); start == end == kSpanOverBudget (pike_vm.hpp) marks a line whose search ran over its step budget.
struct SpanRec {
    uint32_t line, start, end;
};

struct SegmentStats {
    double gpu_ms = 0, stream_ms = 0;
    unsigned launches = 0, stream_launches = 0;
    unsigned long long candidates = 0;
    unsigned long long h2d_bytes = 0, d2h_bytes = 0;
    unsigned path = 0;   // bit0 fast path, bit1 general path
    bool nul = false;    // the streaming kernel found a NUL byte in the segment (it tests in count-only scans only)
};

struct SegmentResult {
    uint64_t num_lines = 0;        // pseudo-lines in the segment
    const LineRec* lines = nullptr;   // simple mode, file order (pinned host memory owned by the slot)
    size_t num_line_recs = 0;
    size_t num_valid_recs = 0;        // fast path: records whose len is not kLineInvalid (the others must be skipped)
    const EventRec* events = nullptr; // general mode, grouped by line in file order
    size_t num_events = 0;
    const SpanRec* spans = nullptr;   // span stage (slot_set_spans): by line, then start
    size_t num_spans = 0;
    SegmentStats stats;
};

struct PikeProgram;       // span program of one pattern (pike_vm.hpp)
struct DeviceDb;          // device-resident DFA tables of one Database on one device
struct DevicePrefilter;   // device-resident gram table of one (sample-tuned) Prefilter
class ScanSlot;    // stream + scratch + pinned result buffers for one in-flight segment

// All functions return 0 or a reference return code (3 = scratch allocation, 7 = CUDA failure) and set `error`.
int engine_select_device(int device, std::string& error);   // cudaSetDevice for the calling host thread
int engine_current_device();                                 // the calling thread's current device
int engine_device_count();

std::shared_ptr<DeviceDb> engine_upload(const std::shared_ptr<Database>& db, std::string& error);
std::shared_ptr<DevicePrefilter> engine_upload_prefilter(const Prefilter& pf, std::string& error);
// Gram hits per MiB that the tuning sample promised for this table (-1: built without a sample).
double prefilter_expected_hits(const DevicePrefilter* pf);

// Pooled per device; never returns a slot in use.  `for_host_input`: the caller will stage host bytes through the slot's pinned
// buffer (the slot with the largest pinned buffer is preferred: pinning is slow); else the one with the most device scratch.
ScanSlot* engine_acquire_slot(std::string& error, bool for_host_input = true);
void engine_release_slot(ScanSlot* slot);

// Pinned staging buffer of the slot (grow-only); used by host ingest to read file bytes into.
uint8_t* slot_host_buffer(ScanSlot* slot, size_t capacity, std::string& error);

// Enqueue the scan of one segment.  Exactly one of host_data / dev_data is non-null.
//  host_data: host memory (pinned => direct H2D; pageable => cudaMemcpyAsync stages it), n bytes.
//  dev_data : device pointer, 16-byte aligned, n bytes, stays valid until slot_collect returns.
//  user_stream: optional cudaStream_t to run on instead of the slot's own stream.
//  pf: gram table for the fast path, or nullptr (general path).
int slot_submit(ScanSlot* slot, const DeviceDb& ddb, const DevicePrefilter* pf, const uint8_t* host_data, const uint8_t* dev_data, size_t n,
                int buffer_size, void* user_stream, std::string& error);
// Count-only callers (no callback, no match limit) need no records on the host: the fast path counts the matched lines on
// the device without building records, SegmentResult::lines stays null and num_valid_recs is exact (num_line_recs is then
// the number of marked lines, repeats included).  Call before slot_submit.
void slot_set_want_records(ScanSlot* slot, bool want);
// Inverted scan (grep -v): the segment's results are the pseudo-lines in which NO pattern reports, as LineRecs of a simple-mode
// database (lines, num_line_recs, num_valid_recs; every record valid, kLineHasNul set conservatively).  num_lines is
// unchanged.  Count-only (no records wanted) costs nothing beyond the normal scan: lines - matched.  Call before slot_submit.
// Weak: a build of the host logic against a CPU stand-in of this engine that lacks inverted scans still links; the boundary
// then fails inverted scans with 7 (there is no host-side complement).  engine.cu always defines it.
__attribute__((weak)) void slot_set_invert(ScanSlot* slot, bool invert);
// Context lines (grep -A/-B/-C), for scans that want records: the segment's results are, in line order, every output line
// whose selected line (matched, or with invert unmatched) lies in the segment - within `after` lines after or `before`
// lines before it - plus the segment's first `after` and last `before` lines, the candidates for the selected lines of
// the neighbouring segments.  Records of lines that are not selected carry kLineContext; every record is valid.
// before == after == 0: no context stage.  Call before slot_submit.  Weak like slot_set_invert (a build without it fails
// context scans with 7).
__attribute__((weak)) void slot_set_context(ScanSlot* slot, uint32_t before, uint32_t after);
// Span stage (grep -o, gpugrep_match_spans): the segment takes the general path, and its results are the leftmost-first
// match spans of `program` in every pseudo-line (SegmentResult::spans) instead of lines or events; null switches it off.
// `program` stays valid until slot_collect returns.  Call before slot_submit.  Weak like slot_set_invert (a build without it
// fails span scans with 7).
__attribute__((weak)) void slot_set_spans(ScanSlot* slot, const PikeProgram* program);
// Fixed-string scan (grep -F, gpugrep_literal_scan_*): the database is a fixed-string set (Database::literal) and the segment
// is matched against its literals instead of automata, on both paths.  Call before slot_submit, which fails with 7 when the
// database is not of the kind the slot is set to.  Weak like slot_set_invert (a build without it fails such scans with 7).
__attribute__((weak)) void slot_set_literals(ScanSlot* slot, bool literal);
// Wait for the segment and expose its results (valid until the next slot_submit on this slot).
// Returns kSplitSegment (and no results) when the fast path hit one of its capacity bounds - a line too long for it, a
// candidate or record overflow - in a segment of more than `split_above` bytes: the caller then scans the same bytes again
// in smaller segments, so that only the piece with the problem takes the (much slower) general path.  The general path
// asks the same when such a segment has more match events than it can hold (2^27).  split_above == 0: never ask, take
// the general path for the whole segment (and fail with 7 over the event bound).
constexpr int kSplitSegment = -2;
int slot_collect(ScanSlot* slot, SegmentResult& out, std::string& error, size_t split_above = 0);

// Copy the bytes of matched lines to the host when the input lives only on the device (device-resident scans
// with a callback).  `recs` are LineRec-like (start,len) pairs already on the host; out must hold sum(len)+count.
int slot_gather_lines(ScanSlot* slot, const uint32_t* starts, const uint32_t* lens, size_t count, uint8_t* out,
                      std::string& error);

// Device-resident input, one round trip on the slot's own stream: the segment ends and the first `head_len` bytes of the
// input (fingerprint of the prefilter sample).  cuts[j] = offset just past the last '\n' before (j+1)*chunk that keeps the
// next segment 16-byte aligned (the last entry is `size`); left empty when the input is a single segment or some
// boundary has no such newline nearby (the caller then cuts sequentially).
// `user_stream`: the stream the caller's producer of dev_data runs on, or null; the probe is ordered behind it.
int slot_probe_input(ScanSlot* slot, const uint8_t* dev_data, size_t size, size_t chunk, std::vector<size_t>& cuts, uint8_t* head,
                     size_t head_len, void* user_stream, std::string& error);

constexpr size_t kMaxSegmentBytes = (size_t)3 << 30;   // offsets inside a segment are 32-bit

}  // namespace gpugrep
