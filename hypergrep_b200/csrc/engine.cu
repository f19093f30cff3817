// CUDA engine for sm_100a: streaming newline/prefilter kernel, scans, candidate verification (DFA), compaction.
//
// Replaces, for one device-resident segment of file bytes, the reference's per-line loop
//   gzgets (line split)  -> hs_scan (match)          -> hs_callback (record)
//   hyperscanner.c:199      hyperscanner.c:217           hyperscanner.c:83-102
// Two paths produce identical results:
//   FAST    (simple mode + literal prefilter + no over-long lines):
//           k_stream -> scan -> k_list_candidates [-> k_confirm] -> k_verify_smem | k_verify_local -> k_tile_offsets -> k_emit_nlm -> k_dedupe_records
//           (count-only: k_emit_nlm<*, true> -> k_count_keys, no records)
//   GENERAL (everything else, and the fallback when a fast-path capacity bound is hit):
//           k_stream(no filter) -> scan -> k_newline_positions -> pseudo-line table -> k_match_pl_* -> scan -> emit
// INVERTED scans (grep -v) select the lines without a match: the fast path adds a complement stage after the dedupe
// (k_invert.cuh, run from slot_collect), the general path negates the per-line flags of k_match_pl_simple.
// SPANS (grep -o, slot_set_spans): the general path up to the pseudo-line table, then k_spans (count) -> scan -> k_spans (write)
// instead of the automata (k_spans.cuh).
// FIXED STRINGS (grep -F, slot_set_literals): the same two paths without automata; k_verify_literals takes the place of the
// DFA verification (k_confirm always runs before it) and k_match_pl_literals that of k_match_pl_simple (k_literal.cuh).
// CONTEXT lines (grep -A/-B/-C, scans with records): a window test over the prefix count of the selected lines picks the
// output lines of a segment (k_context.cuh, after the dedupe on the fast path, after k_match_pl_simple on the general path).
// All byte offsets inside a segment are 32-bit (segments are < 4 GiB); line numbers are rebased on the host.
// Device code lives in the .cuh files included below (one translation unit); this file holds the host side: device
// tables, scan slots, the launch sequence of a segment and the collection of its results.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "engine.hpp"
#include "nfa_sim.hpp"

// device code, in dependency order
#include "device_types.cuh"
#include "swar.cuh"
#include "confirm.cuh"
#include "k_stream.cuh"
#include "scan.cuh"
#include "dfa_walk.cuh"
#include "k_literal.cuh"
#include "k_fast.cuh"
#include "k_general.cuh"
#include "k_invert.cuh"
#include "k_context.cuh"
#include "k_spans.cuh"

namespace gpugrep {

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
    ~DevBuf() { if (p) cudaFree(p); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
    ~PinBuf() { if (p) cudaFreeHost(p); }
};

std::mutex g_mu;
// SM count of the calling thread's current device (scans on different GPUs run concurrently on different host threads:
// nothing here may depend on "the" device of the process)
int device_sms() {
    static int cached[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        cached[dev] = sms;   // benign race: every writer stores the same value
    }
    return cached[dev];
}
// k_verify_smem: table + class map per block, two blocks per SM (227 KiB of shared memory)
constexpr size_t kMaxSharedTableBytes = (size_t)112 << 10;

// A kernel's dynamic shared-memory limit (cudaFuncAttributeMaxDynamicSharedMemorySize) belongs to the process and the
// device, not to one launch.  Scans run concurrently on host threads with different table sizes, so a scan that set a
// smaller limit would make another scan's larger launch fail.  The limit of each kernel is therefore only ever raised:
// one SmemLimit per kernel function (a static at its one launch site) holds the largest value set on each device.
constexpr int kMaxDevices = 64;
struct SmemLimit {
    std::atomic<int> bytes[kMaxDevices] = {};
};
std::mutex g_smem_mu;

template <class Kernel>
cudaError_t raise_smem_limit(SmemLimit& limit, Kernel kernel, size_t smem) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    std::atomic<int>& cur = limit.bytes[dev];
    if ((size_t)cur.load(std::memory_order_acquire) >= smem) return cudaSuccess;
    std::lock_guard<std::mutex> lk(g_smem_mu);
    if ((size_t)cur.load(std::memory_order_relaxed) >= smem) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) cur.store((int)smem, std::memory_order_release);
    return e;
}

}  // namespace

struct DeviceDb {
    std::shared_ptr<Database> db;
    int device = 0;
    std::vector<void*> allocs;
    GroupDev* d_groups = nullptr;
    int ngroups = 0;
    NfaView* d_nfas = nullptr;
    int nnfa = 0;
    bool simple = false;
    size_t smem_table_bytes = 0;   // single group with a class-compressed table (GroupDev::ctab): its size, else 0
    bool literal = false;          // fixed-string set: `lits` instead of groups
    LiteralView lits{};
    ~DeviceDb() { for (void* p : allocs) cudaFree(p); }
};

struct DevicePrefilter {
    int device = 0;
    uint32_t* d_table = nullptr;
    int table_words = 0;
    int stride = 4;
    bool fold = false;
    int mode = 0;        // 1 exact keys, 2 bloom byte table
    int nodd = 0;        // register compares at offsets 2 mod 4 (mixed sampling; bloom mode only)
    ProbeParams pp{};
    uint32_t lookback = 0xffffffffu;
    uint32_t* d_confirm = nullptr;   // exact gram set for the verification kernel (Prefilter::confirm_keys), or null
    uint32_t* d_confirm_groups = nullptr;
    uint32_t* d_confirm_ext = nullptr;            // Prefilter::confirm_ext, or null
    unsigned long long* d_ext_keys = nullptr;
    int ext_log2 = 0;
    unsigned long long ext_mul = 0, ext_mul2 = 0;
    int confirm_log2 = 0;
    uint32_t confirm_mul = 0, confirm_mul2 = 0;
    double bloom_false_rate = 0;     // expected share of 16-byte chunks flagged by bloom collisions alone
    double expected_hits_per_mib = -1;   // gram hits per MiB of the tuning sample (-1: no sample)
    LiteralIndex lit_index{};            // fixed-string sets: Prefilter::lit_begin / lit_entries (null otherwise)
    ~DevicePrefilter() {
        if (lit_index.begin) cudaFree((void*)lit_index.begin);
        if (lit_index.entries) cudaFree((void*)lit_index.entries);
        if (d_table) cudaFree(d_table);
        if (d_confirm) cudaFree(d_confirm);
        if (d_confirm_groups) cudaFree(d_confirm_groups);
        if (d_confirm_ext) cudaFree(d_confirm_ext);
        if (d_ext_keys) cudaFree(d_ext_keys);
    }
};

class ScanSlot {
public:
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // result D2H, so that it does not queue behind the next segment's kernels
    cudaEvent_t done = nullptr;           // all kernels of the segment + the totals copy have finished
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // 0/1: whole segment, 2/3: streaming kernel
    DevBuf d_input, d_meta, d_nlmask, d_gsum, d_prefix, d_sums, d_cand, d_res, d_recoff, d_recs, d_totals;
    DevBuf d_nlpos, d_npl, d_ploff, d_plstart, d_pllen, d_flags, d_counts, d_events, d_gather, d_gidx, d_hitinfo, d_survivors;
    DevBuf d_linebits, d_invrecs;   // inverted fast path: matched-line bitmap, selected-line records (context lines: output records)
    DevBuf d_outbits, d_outoff;     // context lines: output-line bitmap (general path: flags) and its prefix
    DevBuf d_pike;                  // span stage: the program and its byte sets
    PinBuf h_totals, h_recs, h_stage, h_gather, h_probe;
    // state of the in-flight segment
    const DeviceDb* ddb = nullptr;
    const uint8_t* data = nullptr;   // device pointer of the segment
    size_t n = 0, nblk = 0, cand_cap = 0, rec_cap = 0;
    int buffer_size = 0;
    bool fast = false;
    bool want_records = true;   // false: the caller only counts matches (no callback, no limit): the fast path counts without records
    bool invert = false;        // deliver the lines without a match (slot_set_invert)
    uint32_t ctx_before = 0, ctx_after = 0;   // context lines (slot_set_context)
    const PikeProgram* pike = nullptr;        // span stage (slot_set_spans)
    bool literal = false;                     // fixed-string scan (slot_set_literals)
    SegmentStats stats;
    bool in_use = false;

    int run_general(SegmentResult& out, std::string& error, size_t split_above);
    int run_spans(SegmentResult& out, size_t npl_total, std::string& error, size_t split_above);
    int run_complement(size_t nrec, size_t nlines, size_t selected, std::string& error);
    int run_context(size_t nrec, size_t nlines, size_t selected, size_t& count, std::string& error);
    bool context() const { return want_records && (ctx_before || ctx_after); }
};

int engine_select_device(int device, std::string& error) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        error = std::string("no CUDA device available: ") + cudaGetErrorString(e) + " (libgpugrep has no CPU fallback)";
        return 7;
    }
    if (device < 0 || device >= count) device = 0;
    CUDA_TRY(cudaSetDevice(device));   // per host thread
    return 0;
}

int engine_current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return dev;
}

int engine_device_count() {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return count;
}

std::shared_ptr<DeviceDb> engine_upload(const std::shared_ptr<Database>& db, std::string& error) {
    static std::mutex mu;
    static std::vector<std::pair<std::weak_ptr<Database>, std::shared_ptr<DeviceDb>>> cache;
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    cudaGetDevice(&dev);
    for (auto it = cache.begin(); it != cache.end();) {
        auto sp = it->first.lock();
        if (!sp) { it = cache.erase(it); continue; }
        if (sp == db && it->second->device == dev) return it->second;
        ++it;
    }
    auto out = std::make_shared<DeviceDb>();
    out->db = db;
    out->device = dev;
    out->simple = db->simple;
    auto upload = [&](const void* src, size_t bytes) -> void* {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr;
        out->allocs.push_back(p);
        if (bytes && cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        return p;
    };
    if (db->literal) {
        const LiteralSet& L = db->literals;
        std::vector<uint8_t> bytes(L.bytes);
        bytes.resize(bytes.size() + 16, 0);   // (k_literal.cuh lit_compare: 8-byte loads)
        LiteralView v{};
        v.bytes = (const uint8_t*)upload(bytes.data(), bytes.size());
        v.off = (const uint32_t*)upload(L.off.data(), L.off.size() * 4);
        v.len = (const uint32_t*)upload(L.len.data(), L.len.size() * 4);
        v.order = (const uint32_t*)upload(L.order.data(), L.order.size() * 4);
        v.bucket = (const uint32_t*)upload(L.bucket.data(), L.bucket.size() * 4);
        v.one = (const uint32_t*)upload(L.one.data(), L.one.size() * 4);
        for (uint8_t c : L.caseless) v.classes |= 1u << c;
        if (!v.bytes || !v.off || !v.len || !v.order || !v.bucket || !v.one) { error = "cudaMalloc/cudaMemcpy failed while uploading the literals"; return nullptr; }
        out->literal = true;
        out->lits = v;
    }
    std::vector<GroupDev> groups;
    for (size_t g = 0; g < db->groups.size(); g++) {
        const Dfa& d = db->groups[g].dfa;
        if (d.num_states > 65536) { error = "DFA group exceeds 65536 states"; return nullptr; }
        std::vector<uint16_t> t16(d.trans.size());
        for (size_t k = 0; k < d.trans.size(); k++) t16[k] = (uint16_t)d.trans[k];
        GroupDev G{};
        G.trans = (const uint16_t*)upload(t16.data(), t16.size() * sizeof(uint16_t));
        G.cls = (const uint8_t*)upload(d.byte_class, 256);
        G.accept_of = (const uint32_t*)upload(d.accept_of.data(), d.accept_of.size() * sizeof(uint32_t));
        std::vector<uint8_t> depth = d.depth;
        depth.resize((size_t)d.num_states, 255);   // (a table without depths: never stop early)
        G.depth = (const uint8_t*)upload(depth.data(), depth.size());
        if (!G.trans || !G.cls || !G.accept_of || !G.depth) { error = "cudaMalloc/cudaMemcpy failed while uploading DFA tables"; return nullptr; }
        if (db->simple && (size_t)d.num_states * 512 <= ((size_t)256 << 20)) {
            // Byte-indexed table for local verification with the line rules folded in (one load per byte, no special
            // cases in the walk): '\n' and NUL end the scanned block, so their columns hold either the absorbing
            // "matched" state (the block matched at its end) or state 0 (restart: next line / text after the NUL).
            std::vector<uint16_t> flat((size_t)d.num_states * 256), eod((size_t)d.num_states);
            // Every accepting state is replaced by ONE absorbing "matched" state that also survives '\n' and NUL: the
            // walk tests for it only where a line ends (see walk_local), never per byte.
            const uint16_t sink = (uint16_t)d.sink_match;
            for (int st = 0; st < d.num_states; st++) {
                const uint32_t at_eod = d.trans[(size_t)st * d.stride + d.num_classes];
                eod[st] = (uint16_t)at_eod;
                for (int b = 0; b < 256; b++) {
                    uint32_t nx = d.trans[(size_t)st * d.stride + d.byte_class[b]];
                    if (st >= d.first_accept) nx = sink;
                    else if (b == 0) nx = (int)at_eod >= d.first_accept ? sink : 0;
                    else if (b == '\n') nx = ((int)nx >= d.first_accept || (int)d.trans[(size_t)nx * d.stride + d.num_classes] >= d.first_accept) ? sink : 0;
                    else if ((int)nx >= d.first_accept) nx = sink;
                    flat[(size_t)st * 256 + b] = (uint16_t)nx;
                }
            }
            G.flat = (const uint16_t*)upload(flat.data(), flat.size() * sizeof(uint16_t));
            G.eod_next = (const uint16_t*)upload(eod.data(), eod.size() * sizeof(uint16_t));
            if (!G.flat || !G.eod_next) { error = "cudaMalloc/cudaMemcpy failed while uploading DFA tables"; return nullptr; }
            // Class-compressed copy for shared memory.  Bytes of one alphabet class have identical columns in `flat`,
            // except '\n' and NUL, whose columns carry the line rules: they get classes of their own.
            const int ncls = d.num_classes + 2;
            const size_t ctab_bytes = (size_t)d.num_states * ncls * 2;
            if (db->groups.size() == 1 && ncls <= 255 && ctab_bytes + (size_t)d.num_states + 32 <= kMaxSharedTableBytes) {   // (+ the depths)
                std::vector<uint8_t> cmap2(256);
                std::vector<int> rep((size_t)ncls, -1);
                for (int b = 255; b >= 0; b--) {
                    const int c = b == 0 ? d.num_classes : (b == '\n' ? d.num_classes + 1 : d.byte_class[b]);
                    cmap2[(size_t)b] = (uint8_t)c;
                    rep[(size_t)c] = b;
                }
                // the table rounded up to 16 bytes, the depths of the states behind it
                const size_t ctab_pad = (ctab_bytes + 15) / 16 * 16, depth_pad = ((size_t)d.num_states + 15) / 16 * 16;
                std::vector<uint16_t> ctab((ctab_pad + depth_pad) / 2, 0);
                for (int st = 0; st < d.num_states; st++)
                    for (int c = 0; c < ncls; c++)
                        if (rep[(size_t)c] >= 0) ctab[(size_t)st * ncls + c] = flat[(size_t)st * 256 + rep[(size_t)c]];
                std::memcpy(reinterpret_cast<uint8_t*>(ctab.data()) + ctab_pad, depth.data(), depth.size());
                G.cdepth_off = (uint32_t)(ctab_pad / 4);
                G.ctab = (const uint16_t*)upload(ctab.data(), ctab.size() * sizeof(uint16_t));
                G.cmap = (const uint8_t*)upload(cmap2.data(), 256);
                if (!G.ctab || !G.cmap) { error = "cudaMalloc/cudaMemcpy failed while uploading DFA tables"; return nullptr; }
                G.crow = (uint32_t)ncls * 2u;
                G.cstates = (uint32_t)d.num_states;
                out->smem_table_bytes = ctab_pad + depth_pad;
            }
        }
        G.stride = (uint32_t)d.stride;
        G.eod = (uint32_t)d.num_classes;
        G.first_accept = (uint32_t)d.first_accept;
        G.dead = d.dead >= 0 ? (uint32_t)d.dead : 0xffffffffu;
        G.idle_end = (uint32_t)d.idle_end;
        G.mid_other = (uint32_t)d.entry_mid_other;
        G.mid_word = (uint32_t)d.entry_mid_word;
        G.accept_base = db->report_begin.empty() ? 0u : 0u;
        groups.push_back(G);
    }
    // accept_base: flattened index of (group, accept set) = sum of accept-set counts of earlier groups
    uint32_t base = 0;
    for (size_t g = 0; g < groups.size(); g++) {
        groups[g].accept_base = base;
        base += (uint32_t)db->groups[g].dfa.accept_sets.size();
    }
    out->d_groups = (GroupDev*)upload(groups.data(), groups.size() * sizeof(GroupDev));
    out->ngroups = (int)groups.size();
    if (!out->d_groups) { error = "cudaMalloc failed for group table"; return nullptr; }
    std::vector<NfaView> nfas;
    for (size_t k = 0; k < db->nfas.size(); k++) {
        const NfaTables& t = db->nfas[k].tables;
        NfaView v;
        v.positions = t.positions;
        v.words = t.words;
        v.reach = (const uint32_t*)upload(t.reach.data(), t.reach.size() * 4);
        v.follow = (const uint32_t*)upload(t.follow.data(), t.follow.size() * 4);
        v.follow_match = (const uint32_t*)upload(t.follow_match.data(), t.follow_match.size() * 4);
        v.restart = (const uint32_t*)upload(t.restart.data(), t.restart.size() * 4);
        v.report = base + (uint32_t)k;   // flattened report index: after the accept sets of all DFA groups
        if (!v.reach || !v.follow || !v.follow_match || !v.restart) { error = "cudaMalloc failed for NFA tables"; return nullptr; }
        nfas.push_back(v);
    }
    out->d_nfas = (NfaView*)upload(nfas.data(), nfas.size() * sizeof(NfaView));
    out->nnfa = (int)nfas.size();
    cache.emplace_back(db, out);
    if (cache.size() > 8) cache.erase(cache.begin());
    return out;
}

std::shared_ptr<DevicePrefilter> engine_upload_prefilter(const Prefilter& pf, std::string& error) {
    if (!pf.enabled) return nullptr;
    auto out = std::make_shared<DevicePrefilter>();
    cudaGetDevice(&out->device);
    std::vector<uint32_t> replicated;
    const std::vector<uint32_t>* src = &pf.bitmap;
    const char* want = std::getenv("GPUGREP_FILTER");
    const bool use_exact = pf.exact && pf.odd.empty() && want && std::strcmp(want, "exact") == 0;
    out->stride = pf.stride;
    out->fold = pf.fold_case;
    out->mode = use_exact ? 1 : 2;
    out->pp.mul = use_exact ? pf.hash_mul : pf.bloom_mul;
    out->pp.mul2 = pf.hash_mul2;
    out->pp.shift = 32 - (pf.log2_bits - 3);   // bloom: product -> byte index
    out->lookback = pf.lookback;
    out->nodd = (int)std::min<size_t>(pf.odd.size(), 2);
    for (int k = 0; k < 2; k++) {
        const auto& c = pf.odd.empty() ? Prefilter::OddCompare{1u, 1u} : pf.odd[(size_t)k < pf.odd.size() ? (size_t)k : 0];
        out->pp.odd_mul[k] = c.mul;
        out->pp.odd_add[k] = c.add;
    }
    if (use_exact) {
        // replicate so that a lane reads copy (lane mod R): as many copies as fit ~160 KiB of shared memory, at most 32
        const size_t slots = (size_t)1 << pf.log2_slots;
        int rshift = 5;
        while (rshift > 0 && (3 * slots * 4) << rshift > 200 * 1024) rshift--;   // two halves + alignment slack of one half
        const size_t copies = (size_t)1 << rshift;
        replicated.resize(2 * slots * copies);
        for (size_t half = 0; half < 2; half++) {
            // An empty slot holds 0, which reads as a hit for the gram 0 ("\0\0\0\0": NUL runs and the zero padding after the
            // end of a segment), and that gram always probes slot 0.  An empty slot 0 gets a filler key that hashes elsewhere.
            uint32_t slot0 = pf.keys[half * slots];
            if (slot0 == 0) {
                const uint32_t mul = half == 0 ? pf.hash_mul : pf.hash_mul2;
                slot0 = 1;
                while (prefilter_hash(slot0, mul, pf.log2_slots) == 0) slot0++;
            }
            for (size_t h = 0; h < slots; h++)
                for (size_t r = 0; r < copies; r++) replicated[half * slots * copies + h * copies + r] = h == 0 ? slot0 : pf.keys[half * slots + h];
        }
        out->pp.rshift = rshift;
        out->pp.half_bytes = (uint32_t)(slots * copies * 4);
        // byte offset of slot h, copy r: ((h << rshift) | r) * 4.  h = product >> (32 - log2_slots), hence:
        out->pp.shift = 32 - pf.log2_slots - rshift - 2;
        out->pp.amask = (uint32_t)((slots - 1) << (rshift + 2));
        src = &replicated;
    }
    if (!pf.confirm_keys.empty() && pf.confirm_groups.size() == pf.confirm_keys.size()) {
        out->confirm_log2 = pf.confirm_log2;
        out->confirm_mul = pf.confirm_mul;
        out->confirm_mul2 = pf.confirm_mul2;
        if (cudaMalloc((void**)&out->d_confirm, pf.confirm_keys.size() * sizeof(uint32_t)) != cudaSuccess ||
            cudaMemcpy(out->d_confirm, pf.confirm_keys.data(), pf.confirm_keys.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMalloc((void**)&out->d_confirm_groups, pf.confirm_groups.size() * sizeof(uint32_t)) != cudaSuccess ||
            cudaMemcpy(out->d_confirm_groups, pf.confirm_groups.data(), pf.confirm_groups.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) != cudaSuccess) {
            error = "cudaMalloc/cudaMemcpy failed for the gram confirmation table";
            return nullptr;
        }
        if (pf.confirm_ext.size() == pf.confirm_keys.size() && !pf.ext_keys.empty()) {
            out->ext_log2 = pf.ext_log2;
            out->ext_mul = pf.ext_mul;
            out->ext_mul2 = pf.ext_mul2;
            if (cudaMalloc((void**)&out->d_confirm_ext, pf.confirm_ext.size() * sizeof(uint32_t)) != cudaSuccess ||
                cudaMemcpy(out->d_confirm_ext, pf.confirm_ext.data(), pf.confirm_ext.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) != cudaSuccess ||
                cudaMalloc((void**)&out->d_ext_keys, pf.ext_keys.size() * sizeof(uint64_t)) != cudaSuccess ||
                cudaMemcpy(out->d_ext_keys, pf.ext_keys.data(), pf.ext_keys.size() * sizeof(uint64_t), cudaMemcpyHostToDevice) != cudaSuccess) {
                error = "cudaMalloc/cudaMemcpy failed for the extended confirmation table";
                return nullptr;
            }
        }
    }
    if (!pf.lit_begin.empty() && out->d_confirm) {
        void* b = nullptr;
        void* e = nullptr;
        const bool ok = cudaMalloc(&b, pf.lit_begin.size() * 4) == cudaSuccess && (out->lit_index.begin = (const uint32_t*)b) &&
                        cudaMemcpy(b, pf.lit_begin.data(), pf.lit_begin.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
                        cudaMalloc(&e, std::max<size_t>(pf.lit_entries.size(), 1) * 8) == cudaSuccess &&
                        (out->lit_index.entries = (const unsigned long long*)e) &&
                        cudaMemcpy(e, pf.lit_entries.data(), pf.lit_entries.size() * 8, cudaMemcpyHostToDevice) == cudaSuccess;
        if (!ok) { error = "cudaMalloc/cudaMemcpy failed for the literal index"; return nullptr; }
    }
    out->bloom_false_rate = (double)pf.num_grams * (16.0 / pf.stride) / (double)((size_t)1 << pf.log2_bits);
    out->expected_hits_per_mib = pf.expected_hits_per_mib;
    out->table_words = (int)src->size();
    if (cudaMalloc((void**)&out->d_table, src->size() * sizeof(uint32_t)) != cudaSuccess ||
        cudaMemcpy(out->d_table, src->data(), src->size() * sizeof(uint32_t), cudaMemcpyHostToDevice) != cudaSuccess) {
        error = "cudaMalloc/cudaMemcpy failed for the prefilter table";
        return nullptr;
    }
    return out;
}

double prefilter_expected_hits(const DevicePrefilter* pf) { return pf ? pf->expected_hits_per_mib : -1.0; }

namespace {
std::vector<ScanSlot*> g_free_slots;
}

ScanSlot* engine_acquire_slot(std::string& error, bool for_host_input) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { error = "cudaGetDevice failed"; return nullptr; }
    {
        std::lock_guard<std::mutex> lk(g_mu);
        // The free slot that already owns what this scan needs - the largest pinned staging buffer for host inputs (pinning
        // 32 MiB costs milliseconds), the most device scratch for device-resident inputs - and the most recently released
        // one among equals: a small working set of slots is reused and grown once, instead of every pooled slot being
        // re-pinned or re-allocated in turn (growing a buffer frees the old one, which synchronises the device).
        auto weight = [for_host_input](const ScanSlot* sl) {
            const size_t device_scratch = sl->d_input.cap + sl->d_cand.cap + sl->d_hitinfo.cap + sl->d_recs.cap;
            return for_host_input ? std::make_pair(sl->h_stage.cap, device_scratch) : std::make_pair(device_scratch, sl->h_stage.cap);
        };
        size_t best = g_free_slots.size();
        for (size_t i = 0; i < g_free_slots.size(); i++)
            if (g_free_slots[i]->device == dev && (best == g_free_slots.size() || weight(g_free_slots[i]) >= weight(g_free_slots[best]))) best = i;
        if (best < g_free_slots.size()) {
            ScanSlot* s = g_free_slots[best];
            g_free_slots.erase(g_free_slots.begin() + best);
            s->in_use = true;
            return s;
        }
    }
    ScanSlot* s = new ScanSlot();
    s->device = dev;
    if (cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking) != cudaSuccess) { error = "cudaStreamCreate failed"; delete s; return nullptr; }
    for (auto& e : s->ev) if (cudaEventCreate(&e) != cudaSuccess) { error = "cudaEventCreate failed"; delete s; return nullptr; }
    if (cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming) != cudaSuccess) {
        error = "cudaStreamCreate/cudaEventCreate failed"; delete s; return nullptr;
    }
    if (s->d_totals.reserve(sizeof(Totals)) != cudaSuccess || s->h_totals.reserve(sizeof(Totals)) != cudaSuccess) {
        error = "scratch allocation failed"; delete s; return nullptr;
    }
    s->in_use = true;
    return s;
}

void engine_release_slot(ScanSlot* slot) {
    if (!slot) return;
    slot->in_use = false;
    std::lock_guard<std::mutex> lk(g_mu);
    g_free_slots.push_back(slot);
}

void slot_set_want_records(ScanSlot* slot, bool want) { slot->want_records = want; }
void slot_set_invert(ScanSlot* slot, bool invert) { slot->invert = invert; }
void slot_set_spans(ScanSlot* slot, const PikeProgram* program) { slot->pike = program; }
void slot_set_literals(ScanSlot* slot, bool literal) { slot->literal = literal; }
void slot_set_context(ScanSlot* slot, uint32_t before, uint32_t after) {
    slot->ctx_before = before;
    slot->ctx_after = after;
}

uint8_t* slot_host_buffer(ScanSlot* slot, size_t capacity, std::string& error) {
    if (slot->h_stage.reserve(capacity + 64) != cudaSuccess) { error = "cudaHostAlloc failed for the staging buffer"; return nullptr; }
    return slot->h_stage.as<uint8_t>();
}

// Grid of a persistent (grid-stride) kernel: exactly as many blocks as can be resident at once.  A larger grid runs a
// second, partly empty wave in which the late blocks repeat the full per-block share of the work.
template <class Kernel>
static unsigned blocks_per_sm(Kernel kernel, int block, size_t smem = 0) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem) != cudaSuccess || per_sm < 1) {
        (void)cudaGetLastError();
        per_sm = 1;
    }
    return (unsigned)per_sm;
}

template <class Load>
static void launch_scan(cudaStream_t st, Load load, size_t n, unsigned long long* out, unsigned long long* sums, unsigned long long* total,
                        SegmentStats& stats, const unsigned long long* limit = nullptr, int limit_shift = 32) {
    size_t nb = (n + kScanTile - 1) / kScanTile;
    if (nb == 0) nb = 1;
    // persistent grid: with a device-side `limit` most tiles are empty, and empty blocks are not free to schedule
    static const unsigned per_sm = blocks_per_sm(k_scan_sums<Load>, kScanThreads);
    unsigned grid = (unsigned)std::min<size_t>(nb, (size_t)per_sm * device_sms());
    k_scan_sums<Load><<<grid, kScanThreads, 0, st>>>(load, n, sums, nb, limit, limit_shift);
    k_scan_top<<<1, 1024, 0, st>>>(sums, nb, total);
    k_scan_write<Load><<<grid, kScanThreads, 0, st>>>(load, n, sums, out, nb, limit, limit_shift);
    stats.launches += 3;
}

template <int STRIDE, bool FOLD, int MODE, int NODD, bool NUL>
static cudaError_t launch_stream_t(cudaStream_t st, int grid, int block, size_t smem, const uint8_t* data, size_t n, unsigned long long* meta,
                                   uint32_t* nlmask, unsigned long long* gsum, const DevicePrefilter* pf,
                                   unsigned int* flags) {
    if (smem > 48 * 1024) {
        static SmemLimit limit;
        cudaError_t e = raise_smem_limit(limit, k_stream<STRIDE, FOLD, MODE, NODD, NUL>, smem);
        if (e != cudaSuccess) return e;
    }
    k_stream<STRIDE, FOLD, MODE, NODD, NUL><<<grid, block, smem, st>>>(data, n, meta, nlmask, gsum, pf ? pf->d_table : nullptr, pf ? pf->table_words : 0,
                                                            pf ? pf->pp : ProbeParams{}, flags);
    return cudaGetLastError();
}

template <int MODE, bool NUL>
static cudaError_t launch_stream_m(cudaStream_t st, int grid, int block, size_t smem, const uint8_t* data, size_t n, unsigned long long* meta,
                                   uint32_t* nlmask, unsigned long long* gsum, const DevicePrefilter* pf,
                                   unsigned int* flags) {
    int key = pf->stride * 2 + (pf->fold ? 1 : 0);
    if (MODE == 2 && pf->stride == 4 && pf->nodd > 0)
        return pf->fold ? launch_stream_t<4, true, MODE, 2, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags)
                        : launch_stream_t<4, false, MODE, 2, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
    switch (key) {
        case 8: return launch_stream_t<4, false, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
        case 9: return launch_stream_t<4, true, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
        case 4: return launch_stream_t<2, false, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
        case 5: return launch_stream_t<2, true, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
        case 2: return launch_stream_t<1, false, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
        default: return launch_stream_t<1, true, MODE, 0, NUL>(st, grid, block, smem, data, n, meta, nlmask, gsum, pf, flags);
    }
}

int slot_submit(ScanSlot* s, const DeviceDb& ddb, const DevicePrefilter* pf, const uint8_t* host_data, const uint8_t* dev_data, size_t n,
                int buffer_size, void* user_stream, std::string& error) {
    if (n >= ((size_t)1 << 32) - 1024) { error = "segment too large"; return 7; }
    if (s->literal != ddb.literal) { error = "fixed-string scan of a database that is not a fixed-string set, or the reverse"; return 7; }
    s->stream = user_stream ? (cudaStream_t)user_stream : s->own_stream;
    cudaStream_t st = s->stream;
    s->ddb = &ddb;
    s->n = n;
    s->buffer_size = buffer_size;
    s->stats = SegmentStats();
    s->nblk = (n + 511) / 512;
    // fast path: simple mode + prefilter + buffer large enough that "a super-block without newline" is a cheap
    // sufficient test for "no line needs gzgets splitting"
    size_t super_bytes = 0;
    if (buffer_size >= 4096) {
        super_bytes = 2048;
        while (super_bytes * 4 <= (size_t)buffer_size && super_bytes < 65536) super_bytes *= 2;   // 2*super-1 <= buffer_size-1
    }
    // (NFA-fallback patterns ride the fast path when the exact gram table is there: it tells which candidates they own)
    // (fixed strings need the literal index, and the confirm table it hangs off; mode 2 is the bloom table k_confirm reads)
    s->fast = s->pike == nullptr && ddb.simple && pf != nullptr && super_bytes >= 2048 && std::getenv("GPUGREP_FORCE_GENERAL") == nullptr &&
              (ddb.nnfa == 0 || (pf->mode == 2 && pf->d_confirm != nullptr && std::getenv("GPUGREP_NFA_GENERAL") == nullptr)) &&
              (!ddb.literal || (pf->mode == 2 && pf->lit_index.begin != nullptr));

    if (host_data) {
        if (s->d_input.reserve(n + 1024) != cudaSuccess) { error = "cudaMalloc failed for the input segment"; return 3; }
        CUDA_TRY(cudaMemcpyAsync(s->d_input.p, host_data, n, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemsetAsync(s->d_input.as<uint8_t>() + n, 0, 1024, st));
        s->data = s->d_input.as<uint8_t>();
        s->stats.h2d_bytes += n;
    } else {
        if (((uintptr_t)dev_data & 15) != 0) {
            // unaligned device segment (no aligned line end was available for the cut): stage it once, device to device
            if (s->d_input.reserve(n + 1024) != cudaSuccess) { error = "cudaMalloc failed for the input segment"; return 3; }
            CUDA_TRY(cudaMemcpyAsync(s->d_input.p, dev_data, n, cudaMemcpyDeviceToDevice, st));
            CUDA_TRY(cudaMemsetAsync(s->d_input.as<uint8_t>() + n, 0, 1024, st));
            s->data = s->d_input.as<uint8_t>();
        } else {
            s->data = dev_data;
        }
    }
    s->cand_cap = n / 32 + 4096;   // half of all 16-byte chunks; beyond that the segment falls back to the general path
    s->rec_cap = n / 48 + 4096;
    size_t nb_scan = (std::max(s->nblk, s->cand_cap) + kScanTile - 1) / kScanTile + 1;
    if (s->d_meta.reserve((s->nblk + 8) * 8) != cudaSuccess || s->d_nlmask.reserve((s->nblk + 8) * 4) != cudaSuccess ||
        s->d_gsum.reserve((s->nblk / kGroupBlocks + 4) * 8) != cudaSuccess ||
        s->d_prefix.reserve((s->nblk + 8) * 8) != cudaSuccess ||
        s->d_sums.reserve(nb_scan * 8) != cudaSuccess) { error = "cudaMalloc failed for scan scratch"; return 3; }
    if (s->fast) {
        if (s->d_cand.reserve(s->cand_cap * 4) != cudaSuccess || s->d_res.reserve(s->cand_cap * sizeof(uint32_t)) != cudaSuccess ||
            s->d_recoff.reserve((s->cand_cap / kEmitTile + 2) * sizeof(uint32_t)) != cudaSuccess || s->d_recs.reserve(s->rec_cap * sizeof(LineRec)) != cudaSuccess) {
            error = "cudaMalloc failed for candidate scratch"; return 3;
        }
        // (confirmation scratch too, although only multi-group / large sets use it: an allocation in the middle of the launch
        //  sequence would stall the stream)
        if ((ddb.ngroups >= 2 || ddb.nnfa > 0 || pf->bloom_false_rate > 0.005 || ddb.literal) &&
            (s->d_hitinfo.reserve(s->cand_cap * 8) != cudaSuccess || s->d_survivors.reserve(s->cand_cap * 4) != cudaSuccess)) {
            error = "cudaMalloc failed for candidate scratch"; return 3;
        }
    }
    Totals* dT = s->d_totals.as<Totals>();
    CUDA_TRY(cudaMemsetAsync(dT, 0, sizeof(Totals), st));
    CUDA_TRY(cudaEventRecord(s->ev[0], st));
    if (n == 0) {
        CUDA_TRY(cudaEventRecord(s->ev[1], st));
        CUDA_TRY(cudaEventRecord(s->done, st));
        return 0;
    }
    ReprobeParams rp{};
    if (s->fast) {
        // Finding the hits again costs two loads per sampled gram and candidate.  It pays when bloom collisions flag a
        // noticeable share of chunks (large gram sets: those candidates are dropped without a walk) and when several DFA
        // groups would each walk the whole chunk (measured with 32 patterns / 1 group / 415 grams: no gain, so not there).
        const bool want_reprobe = ddb.ngroups >= 2 || pf->bloom_false_rate > 0.005 || ddb.nnfa > 0;
        // (fixed strings: always, the literal index is found through the confirm slot of each hit)
        if (pf->mode >= 2 && pf->d_confirm && ((want_reprobe && (ddb.nnfa > 0 || std::getenv("GPUGREP_NO_REPROBE") == nullptr)) || ddb.literal)) {
            rp.keys = pf->d_confirm;
            rp.groups = pf->d_confirm_groups;
            rp.mul = pf->confirm_mul; rp.mul2 = pf->confirm_mul2; rp.shift = 32 - pf->confirm_log2; rp.half = 1u << pf->confirm_log2;
            rp.stride = pf->stride; rp.fold = pf->fold ? 1 : 0;
            rp.nodd = pf->nodd;
            for (int k = 0; k < 2; k++) { rp.odd_mul[k] = pf->pp.odd_mul[k]; rp.odd_add[k] = pf->pp.odd_add[k]; }
            if (pf->d_confirm_ext && pf->d_ext_keys) {
                rp.ext_info = pf->d_confirm_ext;
                rp.ext_keys = pf->d_ext_keys;
                rp.ext_mul = pf->ext_mul; rp.ext_mul2 = pf->ext_mul2; rp.ext_shift = 64 - pf->ext_log2; rp.ext_half = 1u << pf->ext_log2;
            }
        }
    }
    // ---- K1 ----
    // persistent grid: enough CTAs to fill every SM, each warp strides over groups of kStreamU blocks
    size_t smem = 0;
    if (s->fast) smem = (size_t)pf->table_words * 4 + (pf->mode == 1 ? pf->pp.half_bytes : 0);
    int block = smem > 32 * 1024 ? 1024 : 256;
    int ctas_per_sm = smem > 100 * 1024 ? 1 : (smem > 32 * 1024 ? 2 : 6);
    int grid = device_sms() * ctas_per_sm;
    size_t groups = (s->nblk + kStreamU - 1) / kStreamU;
    size_t max_grid = (groups + (block / 32) - 1) / (block / 32);
    if ((size_t)grid > max_grid) grid = (int)std::max<size_t>(1, max_grid);
    unsigned long long* meta = s->d_meta.as<unsigned long long>();
    uint32_t* nlmask = s->d_nlmask.as<uint32_t>();
    // totals per group of four blocks, written by the streaming kernel and read by the scan; the blocks of the last,
    // partial group add theirs with atomics into a zeroed slot
    unsigned long long* gsum = s->d_gsum.as<unsigned long long>();
    const size_t ngroups = (s->nblk + kGroupBlocks - 1) / kGroupBlocks;
    CUDA_TRY(cudaMemsetAsync(gsum + (ngroups ? ngroups - 1 : 0), 0, 16, st));
    CUDA_TRY(cudaEventRecord(s->ev[2], st));
    cudaError_t le;
    // the NUL test (Totals::flags bit 3) only serves count-only scans (k_emit_nlm<*, true>)
    const bool nul_test = !s->want_records;
    if (!s->fast) le = nul_test ? launch_stream_t<4, false, 0, 0, true>(st, grid, block, 0, s->data, n, meta, nlmask, gsum, nullptr, &dT->flags)
                                : launch_stream_t<4, false, 0, 0, false>(st, grid, block, 0, s->data, n, meta, nlmask, gsum, nullptr, &dT->flags);
    else if (pf->mode == 1) le = nul_test ? launch_stream_m<1, true>(st, grid, block, smem, s->data, n, meta, nlmask, gsum, pf, &dT->flags)
                                          : launch_stream_m<1, false>(st, grid, block, smem, s->data, n, meta, nlmask, gsum, pf, &dT->flags);
    else le = nul_test ? launch_stream_m<2, true>(st, grid, block, smem, s->data, n, meta, nlmask, gsum, pf, &dT->flags)
                       : launch_stream_m<2, false>(st, grid, block, smem, s->data, n, meta, nlmask, gsum, pf, &dT->flags);
    if (le != cudaSuccess) { error = std::string("k_stream launch: ") + cudaGetErrorString(le); return 7; }
    CUDA_TRY(cudaEventRecord(s->ev[3], st));
    s->stats.launches++;
    s->stats.stream_launches++;
    // ---- scan of (candidates, newlines) ----
    unsigned long long* prefix = s->d_prefix.as<unsigned long long>();
    launch_scan(st, LoadU64{gsum}, ngroups, prefix, s->d_sums.as<unsigned long long>(), &dT->meta_total, s->stats);
    if (s->fast) {
        const unsigned sms = (unsigned)device_sms();
        const size_t bps = super_bytes / 512;
        static const unsigned list_per_sm = blocks_per_sm(k_list_candidates, 256);
        k_list_candidates<<<(unsigned)std::min<size_t>((s->nblk + 255) / 256, (size_t)list_per_sm * sms), 256, 0, st>>>(meta, prefix, s->nblk, bps, &dT->meta_total,
                                                                                                                    s->d_cand.as<uint32_t>(), s->cand_cap, dT);
        DbView view{ddb.d_groups, ddb.ngroups, ddb.d_nfas, ddb.nnfa};
        // record offsets per emit tile of kEmitTile candidates: counted by the verification kernel, scanned by one block
        uint32_t* tile_records = s->d_recoff.as<uint32_t>();
        CUDA_TRY(cudaMemsetAsync(tile_records, 0, (s->cand_cap / kEmitTile + 2) * sizeof(uint32_t), st));
        // the last sampled gram of a chunk starts at offset 16 - stride (14 with the compares of mixed sampling) and is 4 bytes long
        const uint32_t idle_span = pf->nodd ? 18u : 20u - (uint32_t)pf->stride;
        // Verification.  Single-group databases whose class-compressed table fits shared memory, with a look-back that the
        // staged text window covers, take k_verify_smem; everything else the global-table kernel.
        // Confirmation of the candidates (which grams really hit, which DFA groups they lead to) in a kernel of its own:
        // the bloom table again from shared memory, exact tables only for what passes it.
        const unsigned long long* hitinfo = nullptr;
        const uint32_t* survivors = nullptr;
        if (rp.keys) {
            if (s->d_hitinfo.reserve(s->cand_cap * 8) != cudaSuccess || s->d_survivors.reserve(s->cand_cap * 4) != cudaSuccess) {
                error = "cudaMalloc failed for candidate scratch"; return 3;
            }
            const size_t csmem = (size_t)pf->table_words * 4;
            static SmemLimit confirm_limit;
            CUDA_TRY(raise_smem_limit(confirm_limit, k_confirm, csmem));
            const unsigned cgrid = (unsigned)std::min<size_t>((s->cand_cap + kConfirmThreads - 1) / kConfirmThreads, sms);
            k_confirm<<<cgrid, kConfirmThreads, csmem, st>>>(s->data, n, s->d_cand.as<uint32_t>(), &dT->meta_total, s->cand_cap, pf->d_table, pf->table_words,
                                                             pf->pp, rp, s->d_hitinfo.as<unsigned long long>(), s->d_res.as<uint32_t>(),
                                                             s->d_survivors.as<uint32_t>(), dT);
            // (checked before anything that reads its output is queued)
            le = cudaGetLastError();
            if (le != cudaSuccess) { error = std::string("k_confirm launch: ") + cudaGetErrorString(le); return 7; }
            hitinfo = s->d_hitinfo.as<unsigned long long>();
            survivors = s->d_survivors.as<uint32_t>();
            s->stats.launches++;
        }
        const char* vsel = std::getenv("GPUGREP_VERIFY");
        const bool v1 = vsel && std::strcmp(vsel, "v1") == 0;
        if (ddb.literal) {
            const unsigned per_sm = blocks_per_sm(k_verify_literals, 128);
            const unsigned vgrid = (unsigned)std::min<size_t>((s->cand_cap + 127) / 128, (size_t)per_sm * sms);
            k_verify_literals<<<vgrid, 128, 0, st>>>(ddb.lits, pf->lit_index, rp, s->data, n, s->d_cand.as<uint32_t>(), hitinfo, survivors, dT,
                                                     s->d_res.as<uint32_t>(), tile_records);
        } else if (!v1 && ddb.smem_table_bytes && hitinfo == nullptr && pf->lookback <= 64u) {
            const size_t vsmem = 256 + ddb.smem_table_bytes;
            static SmemLimit verify_limit;
            CUDA_TRY(raise_smem_limit(verify_limit, k_verify_smem, vsmem));
            const unsigned per_sm = blocks_per_sm(k_verify_smem, kVerifySmemThreads, vsmem);
            unsigned vgrid = (unsigned)std::min<size_t>((s->cand_cap + kVerifySmemThreads - 1) / kVerifySmemThreads, (size_t)per_sm * sms);
            k_verify_smem<<<vgrid, kVerifySmemThreads, vsmem, st>>>(view, s->data, n, s->d_cand.as<uint32_t>(), &dT->meta_total, s->cand_cap, pf->lookback,
                                                                    idle_span, s->d_res.as<uint32_t>(), tile_records);
        } else {
            auto kernel = ddb.nnfa > 0 ? k_verify_local<true> : k_verify_local<false>;
            const unsigned verify_per_sm = blocks_per_sm(kernel, 128);
            unsigned vgrid = (unsigned)std::min<size_t>((s->cand_cap + 127) / 128, (size_t)verify_per_sm * sms);
            kernel<<<vgrid, 128, 0, st>>>(view, s->data, n, s->d_cand.as<uint32_t>(), &dT->meta_total, s->cand_cap, pf->lookback, idle_span, hitinfo,
                                          survivors, dT, s->d_res.as<uint32_t>(), tile_records);
        }
        le = cudaGetLastError();
        if (le != cudaSuccess) { error = std::string("verification kernel launch: ") + cudaGetErrorString(le); return 7; }
        k_tile_offsets<<<1, 1024, 0, st>>>(tile_records, &dT->meta_total, s->cand_cap, &dT->rec_total);
        // Without records (count-only scans) the emit kernel writes one 4-byte key per record into the record buffer, and
        // k_count_keys counts the distinct lines.  Either way a segment with more records than fit falls back to the general
        // path (flags bit 2), so that the count never depends on the capacity.
        const bool count_only = !s->want_records;
        auto emit_kernel = ddb.literal ? (count_only ? k_emit_nlm<false, true, true> : k_emit_nlm<false, false, true>)
                           : ddb.nnfa > 0 ? (count_only ? k_emit_nlm<true, true> : k_emit_nlm<true, false>)
                                          : (count_only ? k_emit_nlm<false, true> : k_emit_nlm<false, false>);
        const size_t out_cap = count_only ? s->rec_cap * sizeof(LineRec) / sizeof(uint32_t) : s->rec_cap;
        const unsigned emit_per_sm = blocks_per_sm(emit_kernel, kEmitThreads);
        emit_kernel<<<(unsigned)std::min<size_t>((s->cand_cap + kEmitTile - 1) / kEmitTile, (size_t)emit_per_sm * sms), kEmitThreads, 0, st>>>(
            view, s->data, n, s->d_cand.as<uint32_t>(), s->d_res.as<uint32_t>(), tile_records, meta, prefix, nlmask, &dT->meta_total,
            s->cand_cap, s->d_recs.as<LineRec>(), s->d_recs.as<uint32_t>(), out_cap, dT, ddb.lits);
        if (count_only)
            k_count_keys<<<(unsigned)std::min<size_t>((out_cap + 255) / 256, (size_t)sms * 4), 256, 0, st>>>(s->d_recs.as<uint32_t>(), out_cap, dT);
        else
            k_dedupe_records<<<(unsigned)std::min<size_t>((s->rec_cap + 255) / 256, (size_t)sms * 4), 256, 0, st>>>(s->d_recs.as<LineRec>(), s->rec_cap, dT);
        s->stats.launches += 5;   // list, verify, tile offsets, emit, dedupe / key count
        CUDA_TRY(cudaEventRecord(s->ev[1], st));
    }
    CUDA_TRY(cudaMemcpyAsync(&dT->last_byte, s->data + n - 1, 1, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->h_totals.p, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(s->done, st));
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int ScanSlot::run_general(SegmentResult& out, std::string& error, size_t split_above) {
    cudaStream_t st = stream;
    Totals* dT = d_totals.as<Totals>();
    Totals* hT = h_totals.as<Totals>();
    stats.path |= 2;
    const size_t nl_total = (size_t)(uint32_t)hT->meta_total;
    const bool trailing = n > 0 && (hT->last_byte & 0xff) != '\n';
    const size_t nlines = nl_total + (trailing ? 1 : 0);
    unsigned long long* prefix = d_prefix.as<unsigned long long>();
    if (d_nlpos.reserve((nl_total + 1) * 4) != cudaSuccess) { error = "cudaMalloc failed for newline index"; return 3; }
    if (nblk) {
        k_newline_positions<<<(unsigned)((nblk * 32 + 255) / 256), 256, 0, st>>>(data, n, nblk, d_meta.as<unsigned long long>(), prefix, d_nlpos.as<uint32_t>());
        stats.launches++;
    }
    const uint32_t limit = (uint32_t)std::min<long long>(std::max(1, buffer_size - 1), 1ll << 29);   // the host cuts with the same clamp (capi.cpp clamp_limit)
    size_t npl_total = nlines;
    bool split = false;
    if (nlines) {
        if (d_npl.reserve(nlines * 4) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
        k_count_pseudo_lines<<<(unsigned)((nlines + 255) / 256), 256, 0, st>>>(d_nlpos.as<uint32_t>(), nl_total, n, nlines, limit, d_npl.as<uint32_t>(), dT);
        stats.launches++;
        CUDA_TRY(cudaMemcpyAsync(hT, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        split = hT->max_line > limit;
        if (split) {
            size_t nb_scan = (nlines + kScanTile - 1) / kScanTile + 1;
            if (d_ploff.reserve(nlines * 8) != cudaSuccess || d_sums.reserve(nb_scan * 8) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
            launch_scan(st, LoadU32{d_npl.as<uint32_t>()}, nlines, d_ploff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->aux_total, stats);
            CUDA_TRY(cudaMemcpyAsync(hT, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            npl_total = (size_t)hT->aux_total;
        }
        if (d_plstart.reserve(npl_total * 4) != cudaSuccess || d_pllen.reserve(npl_total * 4) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
        k_build_pseudo_lines<<<(unsigned)((nlines + 255) / 256), 256, 0, st>>>(d_nlpos.as<uint32_t>(), nl_total, n, nlines, limit,
                                                                                 split ? d_ploff.as<unsigned long long>() : nullptr,
                                                                                 d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>());
        stats.launches++;
    }
    out.num_lines = npl_total;
    out.lines = nullptr; out.num_line_recs = 0; out.events = nullptr; out.num_events = 0;
    if (npl_total == 0) {
        CUDA_TRY(cudaEventRecord(ev[1], st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return 0;
    }
    DbView view{ddb->d_groups, ddb->ngroups, ddb->d_nfas, ddb->nnfa};
    size_t nb_scan = (npl_total + kScanTile - 1) / kScanTile + 1;
    if (d_sums.reserve(nb_scan * 8) != cudaSuccess || d_recoff.reserve(npl_total * 8) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
    if (pike) return run_spans(out, npl_total, error, split_above);
    unsigned mgrid = (unsigned)((npl_total + 127) / 128);
    if (ddb->simple) {
        if (d_flags.reserve(npl_total) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
        if (ddb->literal)
            k_match_pl_literals<<<mgrid, 128, 0, st>>>(ddb->lits, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total, d_flags.as<uint8_t>(), invert);
        else
            k_match_pl_simple<<<mgrid, 128, 0, st>>>(view, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total, d_flags.as<uint8_t>(), invert);
        stats.launches++;
        launch_scan(st, LoadU8{d_flags.as<uint8_t>()}, npl_total, d_recoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->rec_total, stats);
        // context lines: the output flags from the window test over the prefix of the selected flags, and their prefix
        const bool ctx = context();
        if (ctx) {
            if (d_outbits.reserve(npl_total) != cudaSuccess || d_outoff.reserve(npl_total * 8) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
            k_context_flags<<<(unsigned)((npl_total + 255) / 256), 256, 0, st>>>(d_recoff.as<unsigned long long>(), &dT->rec_total, npl_total, ctx_before,
                                                                                   ctx_after, d_outbits.as<uint8_t>());
            stats.launches++;
            launch_scan(st, LoadU8{d_outbits.as<uint8_t>()}, npl_total, d_outoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->aux_total, stats);
        }
        CUDA_TRY(cudaMemcpyAsync(hT, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        size_t nrec = (size_t)(ctx ? hT->aux_total : hT->rec_total);
        if (nrec) {
            if (d_recs.reserve(nrec * sizeof(LineRec)) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
            if (h_recs.reserve(nrec * sizeof(LineRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
            if (ctx)
                k_emit_pl_context<<<(unsigned)((npl_total + 255) / 256), 256, 0, st>>>(d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total,
                                                                                         d_flags.as<uint8_t>(), d_outbits.as<uint8_t>(),
                                                                                         d_outoff.as<unsigned long long>(), d_recs.as<LineRec>());
            else
                k_emit_pl_simple<<<(unsigned)((npl_total + 255) / 256), 256, 0, st>>>(d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total,
                                                                                        d_flags.as<uint8_t>(), d_recoff.as<unsigned long long>(), d_recs.as<LineRec>());
            stats.launches++;
            CUDA_TRY(cudaEventRecord(ev[1], st));
            CUDA_TRY(cudaMemcpyAsync(h_recs.p, d_recs.p, nrec * sizeof(LineRec), cudaMemcpyDeviceToHost, st));
            stats.d2h_bytes += nrec * sizeof(LineRec);
        } else {
            CUDA_TRY(cudaEventRecord(ev[1], st));
        }
        CUDA_TRY(cudaStreamSynchronize(st));
        out.lines = h_recs.as<LineRec>();
        out.num_line_recs = nrec;
    } else {
        if (d_counts.reserve(npl_total * 4) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
        k_match_pl_events<<<mgrid, 128, 0, st>>>(view, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total, d_counts.as<uint32_t>(), nullptr, nullptr);
        stats.launches++;
        launch_scan(st, LoadU32{d_counts.as<uint32_t>()}, npl_total, d_recoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->rec_total, stats);
        CUDA_TRY(cudaMemcpyAsync(hT, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        size_t nev = (size_t)hT->rec_total;
        if (nev > ((size_t)1 << 27)) {
            // a large segment is scanned again in smaller pieces, each under the bound unless its own text is that dense
            if (split_above && n > split_above) return kSplitSegment;
            error = "too many match events in one segment (non-SINGLEMATCH pattern matching nearly every byte?)";
            return 7;
        }
        if (nev) {
            if (d_events.reserve(nev * sizeof(EventRec)) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
            if (h_recs.reserve(nev * sizeof(EventRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
            k_match_pl_events<<<mgrid, 128, 0, st>>>(view, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total, d_counts.as<uint32_t>(),
                                                     d_recoff.as<unsigned long long>(), d_events.as<EventRec>());
            stats.launches++;
            CUDA_TRY(cudaEventRecord(ev[1], st));
            CUDA_TRY(cudaMemcpyAsync(h_recs.p, d_events.p, nev * sizeof(EventRec), cudaMemcpyDeviceToHost, st));
            stats.d2h_bytes += nev * sizeof(EventRec);
        } else {
            CUDA_TRY(cudaEventRecord(ev[1], st));
        }
        CUDA_TRY(cudaStreamSynchronize(st));
        out.events = h_recs.as<EventRec>();
        out.num_events = nev;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Span stage: the spans of every pseudo-line of the table (d_plstart / d_pllen), in line order, copied to h_recs.
int ScanSlot::run_spans(SegmentResult& out, size_t npl_total, std::string& error, size_t split_above) {
    cudaStream_t st = stream;
    Totals* dT = d_totals.as<Totals>();
    Totals* hT = h_totals.as<Totals>();
    const int ninst = (int)pike->insts.size(), nsets = (int)(pike->sets.size() / 8);
    const size_t words = pike->insts.size() + pike->sets.size();
    if (d_pike.reserve(words * 4) != cudaSuccess || d_counts.reserve(npl_total * 4) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
    uint32_t* prog = d_pike.as<uint32_t>();
    CUDA_TRY(cudaMemcpyAsync(prog, pike->insts.data(), pike->insts.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(prog + ninst, pike->sets.data(), pike->sets.size() * 4, cudaMemcpyHostToDevice, st));
    stats.h2d_bytes += words * 4;
    const size_t smem = words * 4;   // at most 128 instructions and 256 sets: 8.5 KiB
    const unsigned grid = (unsigned)((npl_total + 127) / 128);
    k_spans<<<grid, 128, smem, st>>>(prog, ninst, nsets, pike->start, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total,
                                     d_counts.as<uint32_t>(), nullptr, nullptr);
    stats.launches++;
    launch_scan(st, LoadU32{d_counts.as<uint32_t>()}, npl_total, d_recoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->rec_total, stats);
    CUDA_TRY(cudaMemcpyAsync(hT, dT, sizeof(Totals), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const size_t nspan = (size_t)hT->rec_total;
    if (nspan > ((size_t)1 << 27)) {
        if (split_above && n > split_above) return kSplitSegment;
        error = "too many match spans in one segment";
        return 7;
    }
    if (nspan) {
        if (d_events.reserve(nspan * sizeof(SpanRec)) != cudaSuccess) { error = "cudaMalloc failed"; return 3; }
        if (h_recs.reserve(nspan * sizeof(SpanRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
        k_spans<<<grid, 128, smem, st>>>(prog, ninst, nsets, pike->start, data, d_plstart.as<uint32_t>(), d_pllen.as<uint32_t>(), npl_total,
                                         d_counts.as<uint32_t>(), d_recoff.as<unsigned long long>(), d_events.as<SpanRec>());
        stats.launches++;
        CUDA_TRY(cudaEventRecord(ev[1], st));
        CUDA_TRY(cudaMemcpyAsync(h_recs.p, d_events.p, nspan * sizeof(SpanRec), cudaMemcpyDeviceToHost, st));
        stats.d2h_bytes += nspan * sizeof(SpanRec);
    } else {
        CUDA_TRY(cudaEventRecord(ev[1], st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    out.spans = h_recs.as<SpanRec>();
    out.num_spans = nspan;
    return 0;
}

// Inverted fast path: records of the `selected` lines of the segment without a valid record among the first `nrec` of
// d_recs, in line order, copied to h_recs.  One synchronisation (like run_general).
int ScanSlot::run_complement(size_t nrec, size_t nlines, size_t selected, std::string& error) {
    cudaStream_t st = stream;
    Totals* dT = d_totals.as<Totals>();
    const size_t nl_total = (size_t)(uint32_t)h_totals.as<Totals>()->meta_total;
    const size_t nwords = (nlines + 31) / 32;
    const size_t nb_scan = (nwords + kScanTile - 1) / kScanTile + 1;
    // sized from the selected count, not from rec_cap: a text of very short lines selects up to one record per byte
    if (d_linebits.reserve(nwords * 4) != cudaSuccess || d_recoff.reserve(nwords * 8) != cudaSuccess || d_sums.reserve(nb_scan * 8) != cudaSuccess ||
        d_nlpos.reserve((nl_total + 1) * 4) != cudaSuccess || d_invrecs.reserve(selected * sizeof(LineRec)) != cudaSuccess) {
        error = "cudaMalloc failed for the complement of an inverted scan"; return 3;
    }
    if (h_recs.reserve(selected * sizeof(LineRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
    uint32_t* bits = d_linebits.as<uint32_t>();
    CUDA_TRY(cudaMemsetAsync(bits, 0, nwords * 4, st));
    const unsigned sms = (unsigned)device_sms();
    if (nrec) {
        k_mark_lines<<<(unsigned)std::min<size_t>((nrec + 255) / 256, (size_t)sms * 8), 256, 0, st>>>(d_recs.as<LineRec>(), nrec, bits);
        stats.launches++;
    }
    launch_scan(st, LoadPopc{bits}, nwords, d_recoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->rec_total, stats);
    k_newline_positions<<<(unsigned)((nblk * 32 + 255) / 256), 256, 0, st>>>(data, n, nblk, d_meta.as<unsigned long long>(), d_prefix.as<unsigned long long>(),
                                                                           d_nlpos.as<uint32_t>(), d_nlmask.as<uint32_t>());
    k_emit_unmarked<<<(unsigned)((nlines + 255) / 256), 256, 0, st>>>(d_nlpos.as<uint32_t>(), nl_total, n, nlines, bits, d_recoff.as<unsigned long long>(),
                                                                     d_invrecs.as<LineRec>());
    stats.launches += 2;
    CUDA_TRY(cudaEventRecord(ev[1], st));
    CUDA_TRY(cudaMemcpyAsync(h_recs.p, d_invrecs.p, selected * sizeof(LineRec), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    stats.d2h_bytes += selected * sizeof(LineRec);
    return 0;
}

// Fast path with context lines: the `count` output records of the segment (k_context.cuh), in line order, copied to h_recs.
// `selected`: lines selected (valid records, or with invert the lines without one).  The output count is only known on
// the device; the buffers are sized from a bound on it (every selected line outputs at most A+B+1 lines, the edges at
// most A+B more, and no segment more than its lines), so that the stage needs one synchronisation, like run_complement.
int ScanSlot::run_context(size_t nrec, size_t nlines, size_t selected, size_t& count, std::string& error) {
    cudaStream_t st = stream;
    Totals* dT = d_totals.as<Totals>();
    Totals* hT = h_totals.as<Totals>();
    const size_t nl_total = (size_t)(uint32_t)hT->meta_total;
    const size_t nwords = (nlines + 31) / 32;
    const size_t nb_scan = (nwords + kScanTile - 1) / kScanTile + 1;
    const unsigned __int128 window = (unsigned __int128)ctx_before + ctx_after + 1;
    const unsigned __int128 edges = (unsigned __int128)std::min<size_t>(ctx_before, nlines) + std::min<size_t>(ctx_after, nlines);
    const size_t bound = (size_t)std::min<unsigned __int128>(nlines, window * selected + edges);
    if (d_linebits.reserve(nwords * 4) != cudaSuccess || d_outbits.reserve(nwords * 4) != cudaSuccess || d_recoff.reserve(nwords * 8) != cudaSuccess ||
        d_outoff.reserve(nwords * 8) != cudaSuccess || d_sums.reserve(nb_scan * 8) != cudaSuccess || d_nlpos.reserve((nl_total + 1) * 4) != cudaSuccess ||
        d_invrecs.reserve(bound * sizeof(LineRec)) != cudaSuccess) {
        error = "cudaMalloc failed for the context lines of a scan"; return 3;
    }
    if (h_recs.reserve(bound * sizeof(LineRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
    uint32_t* bits = d_linebits.as<uint32_t>();
    uint32_t* out_bits = d_outbits.as<uint32_t>();
    CUDA_TRY(cudaMemsetAsync(bits, 0, nwords * 4, st));
    const unsigned sms = (unsigned)device_sms();
    if (nrec) {
        k_mark_lines<<<(unsigned)std::min<size_t>((nrec + 255) / 256, (size_t)sms * 8), 256, 0, st>>>(d_recs.as<LineRec>(), nrec, bits);
        stats.launches++;
    }
    launch_scan(st, LoadSelectedPopc{bits, nlines, invert}, nwords, d_recoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->rec_total, stats);
    const unsigned line_grid = (unsigned)((nwords * 32 + 255) / 256);
    k_context_bits<<<line_grid, 256, 0, st>>>(bits, nlines, invert, d_recoff.as<unsigned long long>(), &dT->rec_total, ctx_before, ctx_after, out_bits);
    launch_scan(st, LoadPopc{out_bits}, nwords, d_outoff.as<unsigned long long>(), d_sums.as<unsigned long long>(), &dT->aux_total, stats);
    k_newline_positions<<<(unsigned)((nblk * 32 + 255) / 256), 256, 0, st>>>(data, n, nblk, d_meta.as<unsigned long long>(), d_prefix.as<unsigned long long>(),
                                                                           d_nlpos.as<uint32_t>(), d_nlmask.as<uint32_t>());
    k_emit_context<<<line_grid, 256, 0, st>>>(d_nlpos.as<uint32_t>(), nl_total, n, nlines, bits, invert, out_bits, d_outoff.as<unsigned long long>(),
                                              d_invrecs.as<LineRec>());
    stats.launches += 3;
    CUDA_TRY(cudaEventRecord(ev[1], st));
    CUDA_TRY(cudaMemcpyAsync(&hT->aux_total, &dT->aux_total, sizeof(hT->aux_total), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(h_recs.p, d_invrecs.p, bound * sizeof(LineRec), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    count = (size_t)hT->aux_total;
    if (count > bound) { error = "context lines: more output lines than the bound allows"; return 7; }
    stats.d2h_bytes += bound * sizeof(LineRec) + sizeof(hT->aux_total);
    return 0;
}

int slot_collect(ScanSlot* s, SegmentResult& out, std::string& error, size_t split_above) {
    cudaStream_t st = s->stream;
    out = SegmentResult();
    // wait for THIS segment only: the stream may already hold the next segment's kernels
    CUDA_TRY(cudaEventSynchronize(s->done));
    s->stats.d2h_bytes += sizeof(Totals);
    if (s->n == 0) { out.stats = s->stats; return 0; }
    Totals* hT = s->h_totals.as<Totals>();
    s->stats.nul = (hT->flags & kSegmentNulFlag) != 0;
    bool done = false;
    if (s->fast) {
        s->stats.candidates = hT->meta_total >> 32;
        if ((hT->flags & kFallbackFlags) == 0) {
            s->stats.path |= 1;
            size_t nrec = (size_t)hT->rec_total;   // includes records marked kInvalidLen (repeats of a line, failed NUL re-checks)
            out.num_valid_recs = (size_t)hT->aux_total;
            const size_t nl_total = (size_t)(uint32_t)hT->meta_total;
            out.num_lines = nl_total + ((hT->last_byte & 0xff) != '\n' ? 1 : 0);
            if (s->context()) {
                const size_t selected = s->invert ? (size_t)out.num_lines - out.num_valid_recs : out.num_valid_recs;
                size_t count = 0;
                int rc = s->run_context(nrec, (size_t)out.num_lines, selected, count, error);
                if (rc) return rc;
                nrec = count;
                out.num_valid_recs = count;
            } else if (s->invert) {
                // the valid records are the matched lines, one each: the complement has lines - valid records
                const size_t selected = (size_t)out.num_lines - out.num_valid_recs;
                if (selected && s->want_records) {
                    int rc = s->run_complement(nrec, (size_t)out.num_lines, selected, error);
                    if (rc) return rc;
                }
                nrec = selected;
                out.num_valid_recs = selected;
            } else if (nrec && s->want_records) {
                if (s->h_recs.reserve(nrec * sizeof(LineRec)) != cudaSuccess) { error = "cudaHostAlloc failed"; return 3; }
                CUDA_TRY(cudaMemcpyAsync(s->h_recs.p, s->d_recs.p, nrec * sizeof(LineRec), cudaMemcpyDeviceToHost, s->copy_stream));
                CUDA_TRY(cudaStreamSynchronize(s->copy_stream));
                s->stats.d2h_bytes += nrec * sizeof(LineRec);
            }
            out.lines = s->want_records ? s->h_recs.as<LineRec>() : nullptr;
            out.num_line_recs = nrec;
            done = true;
        }
    }
    if (!done) {
        if (s->fast && split_above && s->n > split_above) { out.stats = s->stats; return kSplitSegment; }
        int rc = s->run_general(out, error, split_above);
        if (rc == kSplitSegment) out.stats = s->stats;
        if (rc) return rc;
    }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, s->ev[0], s->ev[1]) == cudaSuccess) s->stats.gpu_ms = ms;
    if (cudaEventElapsedTime(&ms, s->ev[2], s->ev[3]) == cudaSuccess) s->stats.stream_ms = ms;
    out.stats = s->stats;
    return 0;
}

int slot_probe_input(ScanSlot* s, const uint8_t* dev_data, size_t size, size_t chunk, std::vector<size_t>& cuts, uint8_t* head, size_t head_len,
                     void* user_stream, std::string& error) {
    cuts.clear();
    if (size == 0) return 0;
    const size_t ncuts = chunk && size > chunk ? (size + chunk - 1) / chunk : 0;
    head_len = std::min(head_len, size);
    if (s->h_probe.reserve(ncuts * 8 + head_len + 16) != cudaSuccess || (ncuts && s->d_sums.reserve(ncuts * 8) != cudaSuccess)) {
        error = "scratch allocation failed";
        return 3;
    }
    // on the caller's stream when there is one: whatever produces the buffer there has finished before the probe reads it
    cudaStream_t st = user_stream ? (cudaStream_t)user_stream : s->own_stream;
    unsigned long long* h_cuts = s->h_probe.as<unsigned long long>();
    uint8_t* h_head = s->h_probe.as<uint8_t>() + ncuts * 8;
    if (ncuts) {
        k_find_cuts<<<(unsigned)((ncuts + 63) / 64), 64, 0, st>>>(dev_data, size, chunk, (size_t)4 << 20, ncuts, s->d_sums.as<unsigned long long>());
        CUDA_TRY(cudaMemcpyAsync(h_cuts, s->d_sums.p, ncuts * 8, cudaMemcpyDeviceToHost, st));
    }
    if (head_len) CUDA_TRY(cudaMemcpyAsync(h_head, dev_data, head_len, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (head_len) std::memcpy(head, h_head, head_len);
    size_t prev = 0;
    for (size_t j = 0; j < ncuts; j++) {
        if (h_cuts[j] == 0 || h_cuts[j] <= prev) { cuts.clear(); break; }   // no newline near a boundary: caller falls back
        cuts.push_back((size_t)h_cuts[j]);
        prev = (size_t)h_cuts[j];
    }
    return 0;
}

int slot_gather_lines(ScanSlot* s, const uint32_t* starts, const uint32_t* lens, size_t count, uint8_t* out, std::string& error) {
    if (count == 0) return 0;
    cudaStream_t st = s->stream;
    // offsets on the host (small), then one gather kernel and one D2H
    std::vector<unsigned long long> off(count);
    unsigned long long total = 0;
    for (size_t i = 0; i < count; i++) { off[i] = total; total += (unsigned long long)lens[i] + 1; }
    if (s->d_gidx.reserve(count * 16) != cudaSuccess || s->d_gather.reserve(total) != cudaSuccess || s->h_gather.reserve(total) != cudaSuccess) {
        error = "allocation failed in gather"; return 3;
    }
    uint32_t* d_starts = s->d_gidx.as<uint32_t>();
    uint32_t* d_lens = d_starts + count;
    unsigned long long* d_off = reinterpret_cast<unsigned long long*>(d_starts + 2 * count);
    CUDA_TRY(cudaMemcpyAsync(d_starts, starts, count * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_lens, lens, count * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_off, off.data(), count * 8, cudaMemcpyHostToDevice, st));
    k_gather_lines<<<(unsigned)((count * 32 + 255) / 256), 256, 0, st>>>(s->data, d_starts, d_lens, d_off, count, s->d_gather.as<uint8_t>());
    CUDA_TRY(cudaMemcpyAsync(s->h_gather.p, s->d_gather.p, total, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    std::memcpy(out, s->h_gather.p, total);
    s->stats.launches++;
    s->stats.d2h_bytes += total;
    return 0;
}

}  // namespace gpugrep
