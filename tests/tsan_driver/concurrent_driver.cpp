// TEST-ONLY: concurrent scans through the host logic of the boundary, built with -fsanitize=thread over the CPU engine
// stand-in of tests/mock_engine_context (see the Makefile).  Run by tests/test_concurrent_scans.py.
//
//   concurrent_driver DIR
//
// DIR holds plain.log (over 8 MiB: one read of it is split over helper threads), small.log, members.gz and frames.zst (many
// members / frames: decode helpers) and big.log.  Every call of a fixed list runs once serially; its answer (return code, a
// hash of every record and batch size, stats.matches and stats.lines) is kept.  Then 8 threads run the list in rounds, each
// thread in its own order, and every answer must equal the serial one.  This is done twice: on one device, then with
// $GPUGREP_DEVICES=all over the mock devices of $GPUGREP_MOCK_DEVICES, where plain files and host buffers over 2 MiB are
// split into shards (set between the phases, while no scan runs).  Exit 0 and "concurrent driver ok" on success, 1 on a
// difference; ThreadSanitizer's own exit code on a report.
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iterator>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "gpugrep.h"

namespace {

struct Answer {
    int rc = -1;
    uint64_t hash = 0;
    unsigned long long records = 0, matches = 0, lines = 0;
    bool operator==(const Answer& o) const {
        return rc == o.rc && hash == o.hash && records == o.records && matches == o.matches && lines == o.lines;
    }
};

// the callback runs on the calling thread (sharded scans merge there too): one accumulator per thread
thread_local uint64_t t_hash = 0;
thread_local unsigned long long t_records = 0;

void mix(const void* p, size_t n) {
    const uint8_t* b = static_cast<const uint8_t*>(p);
    for (size_t i = 0; i < n; i++) t_hash = (t_hash ^ b[i]) * 1099511628211ull;
}

void on_event(hyperscanner_result_t* results, int count) {
    mix(&count, sizeof(count));
    for (int i = 0; i < count; i++) {
        mix(&results[i].id, sizeof(results[i].id));
        mix(&results[i].line_number, sizeof(results[i].line_number));
        mix(results[i].line, std::strlen(results[i].line));
        t_records++;
    }
}

enum class Entry { Hyperscan, Scan, Count, Invert, InvertCount, Context, InvertContext };
enum class Input { File, Host };

struct PatternSet {
    std::vector<const char*> patterns;
    std::vector<unsigned> flags, ids;
};

struct Call {
    Entry entry;
    Input input;
    std::string file;
    const PatternSet* set;
    std::string label;
};

std::vector<char> read_file(const std::string& path) {
    std::ifstream in(path, std::ios::binary);
    return std::vector<char>(std::istreambuf_iterator<char>(in), std::istreambuf_iterator<char>());
}

struct Texts {
    std::vector<std::vector<char>> blobs;
    std::vector<std::string> names;
    const std::vector<char>& get(const std::string& name) const {
        for (size_t k = 0; k < names.size(); k++)
            if (names[k] == name) return blobs[k];
        std::fprintf(stderr, "no text %s\n", name.c_str());
        std::exit(2);
    }
};

Answer run(const Call& c, const Texts& texts) {
    t_hash = 1469598103934665603ull;
    t_records = 0;
    gpugrep_stats st{};
    const PatternSet& p = *c.set;
    const unsigned n = (unsigned)p.patterns.size();
    const char* const* pa = p.patterns.data();
    const bool collect = c.entry != Entry::Count && c.entry != Entry::InvertCount;
    hs_event cb = collect ? on_event : nullptr;
    Answer a;
    if (c.input == Input::File) {
        const char* path = c.file.c_str();
        switch (c.entry) {
            case Entry::Hyperscan:
                a.rc = hyperscan(const_cast<char*>(path), pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7, 0);
                break;
            case Entry::Scan: case Entry::Count:
                a.rc = gpugrep_scan_file(path, pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7, 0, &st);
                break;
            case Entry::Invert: case Entry::InvertCount:
                a.rc = gpugrep_invert_scan_file(path, pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7, 0, &st);
                break;
            case Entry::Context: case Entry::InvertContext:
                a.rc = gpugrep_context_scan_file(path, pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7, 0, 2, 1, c.entry == Entry::InvertContext,
                                                 &st);
                break;
        }
    } else {
        const std::vector<char>& text = texts.get(c.file);
        switch (c.entry) {
            case Entry::Hyperscan: case Entry::Scan: case Entry::Count:
                a.rc = gpugrep_scan_buffer(text.data(), text.size(), GPUGREP_LOC_HOST, pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7, 0,
                                           nullptr, &st);
                break;
            case Entry::Invert: case Entry::InvertCount:
                a.rc = gpugrep_invert_scan_buffer(text.data(), text.size(), GPUGREP_LOC_HOST, pa, p.flags.data(), p.ids.data(), n, cb, 262140, 7,
                                                  0, nullptr, &st);
                break;
            case Entry::Context: case Entry::InvertContext:
                a.rc = gpugrep_context_scan_buffer(text.data(), text.size(), GPUGREP_LOC_HOST, pa, p.flags.data(), p.ids.data(), n, cb, 262140,
                                                   7, 0, 2, 1, c.entry == Entry::InvertContext, nullptr, &st);
                break;
        }
    }
    a.hash = t_hash;
    a.records = t_records;
    a.matches = st.matches;
    a.lines = st.lines;
    return a;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc != 2) {
        std::fprintf(stderr, "usage: %s DIR\n", argv[0]);
        return 2;
    }
    const std::string dir = argv[1];
    PatternSet one{{"ERROR"}, {14}, {0}};
    PatternSet literals{{"port 8080", "sshd", "timeout", "GET /index", "user=bob"}, {14, 14, 14, 14, 14}, {0, 0, 0, 0, 0}};
    // several ids, some patterns without SINGLEMATCH: the general host path (events, id order)
    PatternSet general{{"ERROR", "port [0-9]+", "sshd", "fail(ed|ure)", "x{2,}"}, {6, 14, 6, 14, 6}, {1, 2, 3, 4, 5}};
    PatternSet caseless{{"error", "alpha.*kilo"}, {15, 15}, {0, 0}};

    Texts texts;
    texts.names = {"big.log", "small.log"};
    for (const auto& name : texts.names) texts.blobs.push_back(read_file(dir + "/" + name));

    std::vector<Call> calls;
    auto add = [&](Entry e, Input in, const std::string& file, const PatternSet& set, const char* what) {
        calls.push_back(Call{e, in, in == Input::File ? dir + "/" + file : file, &set, std::string(what) + " " + file});
    };
    add(Entry::Hyperscan, Input::File, "plain.log", general, "hyperscan");
    for (const PatternSet* set : {&one, &literals, &general, &caseless}) {
        add(Entry::Hyperscan, Input::File, "small.log", *set, "hyperscan");
        add(Entry::Scan, Input::File, "members.gz", *set, "scan");
        add(Entry::Scan, Input::File, "frames.zst", *set, "scan");
        add(Entry::Scan, Input::Host, "big.log", *set, "scan");
        add(Entry::Count, Input::Host, "big.log", *set, "count");
        add(Entry::Scan, Input::Host, "small.log", *set, "scan");
    }
    add(Entry::Count, Input::File, "plain.log", literals, "count");
    add(Entry::Invert, Input::File, "members.gz", literals, "invert");
    add(Entry::Invert, Input::Host, "big.log", one, "invert");
    add(Entry::InvertCount, Input::Host, "big.log", literals, "invert count");
    add(Entry::InvertCount, Input::File, "frames.zst", one, "invert count");
    add(Entry::Context, Input::File, "members.gz", literals, "context");
    add(Entry::Context, Input::Host, "big.log", one, "context");
    add(Entry::InvertContext, Input::File, "frames.zst", literals, "invert context");
    add(Entry::InvertContext, Input::Host, "small.log", one, "invert context");

    std::atomic<int> failures{0};
    constexpr int kThreads = 8, kRounds = 1;
    for (int phase = 0; phase < 2; phase++) {
        if (phase == 1) {
            setenv("GPUGREP_DEVICES", "all", 1);
            setenv("GPUGREP_MIN_SHARD_BYTES", "1048576", 1);
        }
        std::vector<Answer> serial;
        for (const Call& c : calls) {
            serial.push_back(run(c, texts));
            if (serial.back().rc != 0) {
                std::fprintf(stderr, "%s: return code %d (%s)\n", c.label.c_str(), serial.back().rc, gpugrep_last_error());
                return 1;
            }
        }
        for (int round = 0; round < kRounds; round++) {
            std::vector<std::thread> threads;
            for (int t = 0; t < kThreads; t++) {
                threads.emplace_back([&, t, round] {
                    std::vector<size_t> order(calls.size());
                    for (size_t k = 0; k < order.size(); k++) order[k] = k;
                    std::mt19937 rng((unsigned)((phase * kRounds + round) * kThreads + t + 1));
                    std::shuffle(order.begin(), order.end(), rng);
                    for (size_t k : order) {
                        const Answer a = run(calls[k], texts);
                        if (!(a == serial[k])) {
                            std::fprintf(stderr, "phase %d round %d thread %d: %s differs: rc %d/%d records %llu/%llu matches %llu/%llu lines %llu/%llu\n",
                                         phase, round, t, calls[k].label.c_str(), a.rc, serial[k].rc, a.records, serial[k].records, a.matches,
                                         serial[k].matches, a.lines, serial[k].lines);
                            failures++;
                        }
                    }
                });
            }
            for (auto& th : threads) th.join();
        }
    }
    if (failures.load()) return 1;
    std::printf("concurrent driver ok: %zu calls, %d threads x %d rounds, two phases\n", calls.size(), kThreads, kRounds);
    return 0;
}
