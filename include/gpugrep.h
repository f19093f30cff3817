/*
 * libgpugrep.so — C ABI of the B200-native multi-pattern log scanner.
 *
 * Section 1 is the drop-in boundary: exactly the two symbols the reference's Python layer binds with ctypes
 * (reference hypergrep/utils.py:116-121 and :339-349), with the signatures, record layout, return codes and
 * callback discipline of the reference's C shim (reference hypergrep/lib/c/hyperscanner.c:25-56, 154-159,
 * 248-258).  Section 2 holds extensions used by this repo's bench, tests and tools; the reference has no
 * equivalent for them.
 *
 * No symbol in this header takes or returns a torch / CUDA runtime type: plain pointers, sizes and PODs only.
 */
#ifndef GPUGREP_H
#define GPUGREP_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define GPUGREP_API __attribute__((visibility("default")))
#else
#define GPUGREP_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------------------
 * 1. Drop-in boundary
 * ---------------------------------------------------------------------------------------------------------- */

/* Return codes: reference hyperscanner.c:25-33 (enum hyperscanner_ret). 0 = success. */
enum gpugrep_ret {
    GPUGREP_OK = 0,
    GPUGREP_COMPILE_MEM = 1, /* HYPERSCANNER_COMPILE_MEM: result slots could not be allocated            */
    GPUGREP_COMPILE = 2,     /* HYPERSCANNER_COMPILE                                                       */
    GPUGREP_SCRATCH = 3,     /* HYPERSCANNER_SCRATCH: device / pinned scratch could not be allocated       */
    GPUGREP_DB = 4,          /* HYPERSCANNER_DB: a pattern was rejected (unsupported construct, empty ...) */
    GPUGREP_STATE_MEM = 5,   /* HYPERSCANNER_STATE_MEM                                                     */
    GPUGREP_GZ_OPEN = 6,     /* HYPERSCANNER_GZ_OPEN: the input file could not be opened                   */
    GPUGREP_SCAN = 7         /* HYPERSCANNER_SCAN: a CUDA error during the scan (no GPU, launch failure)   */
};

/* hyperscanner_result_t, reference hyperscanner.c:42-46 == ctypes `Result`, reference utils.py:25-40.
 * sizeof == 24 on x86-64: id @0, line_number @8, line @16. */
typedef struct hyperscanner_result {
    unsigned int id;                /* the user's match id of the pattern group that matched            */
    unsigned long long line_number; /* 0-based pseudo-line index (one per gzgets() of buffer_size)      */
    char* line;                     /* NUL-terminated line bytes incl. trailing '\n'; valid during the callback only */
} hyperscanner_result_t;

/* hs_event, reference hyperscanner.c:54.  Invoked synchronously on the calling thread, in file order, with
 * 1 <= result_count <= buffer_count: full batches first, then the remainder (hyperscanner.c:94-98, 311-313). */
typedef void (*hs_event)(hyperscanner_result_t* results, int result_count);

/* Replaces reference hyperscanner.c:248-326 `hyperscan()`.
 * file_name: plain, gzip or zstd file.  patterns/pattern_flags/pattern_ids: `elements` entries; flags are
 * HS_FLAG_CASELESS=1 | DOTALL=2 | MULTILINE=4 | SINGLEMATCH=8 (other bits -> 4).  buffer_size: a pseudo-line is
 * at most buffer_size-1 bytes (the reference's gzgets buffer).  buffer_count: callback batch size (clamped to
 * max_match_count when that is smaller, hyperscanner.c:259-262).  max_match_count: stop after the line on which
 * the total reaches it; 0 = unlimited. */
GPUGREP_API int hyperscan(char* file_name, const char* const* patterns, const unsigned int* pattern_flags,
              const unsigned int* pattern_ids, const unsigned int elements, hs_event on_event,
              const int buffer_size, int buffer_count, unsigned long long max_match_count);

/* Replaces reference hyperscanner.c:154-167 `check_patterns()`: 0 if the set compiles, else 4.
 * Never touches CUDA (safe before fork(), SURVEY.md §8b). */
GPUGREP_API int check_patterns(const char* const* patterns, const unsigned int* pattern_flags,
                   const unsigned int* pattern_ids, const unsigned int elements);

/* ------------------------------------------------------------------------------------------------------------
 * 2. Extensions (bench / tests / tools)
 * ---------------------------------------------------------------------------------------------------------- */

/* Per-call statistics of the scan entry points below (all fields are outputs). */
typedef struct gpugrep_stats {
    unsigned long long bytes_scanned;  /* uncompressed bytes handed to the kernels                        */
    unsigned long long lines;          /* pseudo-lines seen                                                */
    unsigned long long matches;        /* results delivered (or counted when on_event is NULL)             */
    unsigned long long candidates;     /* 16-byte chunks flagged by the prefilter (0 when it is off)       */
    unsigned long long h2d_bytes;      /* host->device bytes copied inside the call                        */
    unsigned long long d2h_bytes;      /* device->host bytes copied inside the call                        */
    double gpu_ms;                     /* CUDA-event time of all kernels of the call, summed over segments */
    double stream_kernel_ms;           /* of which: the streaming prefilter/newline kernel                 */
    double wall_ms;                    /* host wall-clock of the call                                      */
    unsigned int launches;             /* kernels launched by this library inside the call                 */
    unsigned int stream_launches;      /* of which: launches of the streaming kernel                       */
    unsigned int segments;             /* device segments processed                                        */
    unsigned int path;                 /* bit 0: prefilter fast path used; bit 1: general line-table path used */
    unsigned int split_segments;       /* large segments that hit a fast-path bound and were scanned again in 64 MiB pieces */
    unsigned int nul_segments;         /* segments with a NUL byte (count-only scans test for them)        */
} gpugrep_stats;

#define GPUGREP_LOC_HOST 0   /* data is host memory (pinned memory is copied directly, pageable is staged) */
#define GPUGREP_LOC_DEVICE 1 /* data is a device pointer on the current device; the kernels read it in aligned 16-byte  \
                                granules, so the allocation must be readable up to the next multiple of 16 bytes behind \
                                data + size (true for any cudaMalloc / framework allocation: their granularity is >= 256  \
                                bytes); a pointer that is not 16-byte aligned is staged once, device to device          */

/* Scan a memory buffer holding the (decompressed) file contents; same pattern, batching and callback
 * semantics as hyperscan().  on_event may be NULL: matches are then only counted (no line bytes are copied).
 * `stream` is an optional cudaStream_t (as void*) to enqueue on, NULL = the library's own stream. */
GPUGREP_API int gpugrep_scan_buffer(const void* data, size_t size, int location, const char* const* patterns,
                        const unsigned int* pattern_flags, const unsigned int* pattern_ids, unsigned int elements,
                        hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                        void* stream, gpugrep_stats* stats);

/* hyperscan() plus statistics. */
GPUGREP_API int gpugrep_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags,
                      const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size,
                      int buffer_count, unsigned long long max_match_count, gpugrep_stats* stats);

/* ---- inverted matching (`grep -v`) -------------------------------------------------------------------------------
 * Same arguments, inputs (plain / gzip / zstd files, host / pinned / device buffers, $GPUGREP_DEVICES sharding) and
 * return codes as gpugrep_scan_file / gpugrep_scan_buffer, but the delivered records are the pseudo-lines in which NO
 * pattern reports: for every input, their line numbers are {0 .. lines-1} minus those of the non-inverted scan.
 * Each selected line is one record with id 0; `line` is the stripped text (leading NULs skipped, cut at the next NUL), so a
 * pseudo-line of NUL bytes only is delivered as "".  The pattern set is compile-checked as given (4 exactly when
 * hyperscan() returns 4); ids and SINGLEMATCH do not change which lines are selected.  max_match_count counts selected
 * lines (the scan stops after the line on which the count reaches it), buffer_count batches them as in hyperscan(), and
 * stats->matches is the number of selected lines.  on_event == NULL without a limit counts on the device. */
GPUGREP_API int gpugrep_invert_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags,
                             const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size,
                             int buffer_count, unsigned long long max_match_count, gpugrep_stats* stats);
GPUGREP_API int gpugrep_invert_scan_buffer(const void* data, size_t size, int location, const char* const* patterns,
                               const unsigned int* pattern_flags, const unsigned int* pattern_ids, unsigned int elements,
                               hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                               void* stream, gpugrep_stats* stats);

/* ---- context lines (`grep -A/-B/-C`) -----------------------------------------------------------------------------
 * Same inputs and return codes as gpugrep_scan_file / gpugrep_scan_buffer.  The selected lines are the matched pseudo-lines,
 * or with `invert` != 0 those in which no pattern reports (as gpugrep_invert_scan_*).  A pseudo-line is delivered if it is
 * selected, or lies within `after` lines after or `before` lines before a selected line (a context line).  Records come in
 * line order, one per delivered line: selected lines with id 0, context lines with id GPUGREP_CONTEXT_ID; `line` is the
 * stripped text (a pseudo-line of NUL bytes only is ""), and a caller sees a new group wherever line_number jumps.
 * The pattern set is compile-checked as given, then scanned as "every pattern SINGLEMATCH, one id".  max_match_count counts
 * selected lines; after the line that reaches it, the next `after` lines are still delivered, all as context (even lines
 * that would match), then the scan stops.  Batches are full batches of buffer_count records, context lines included
 * (clamped to max_match_count when that is smaller), then the remainder.  stats->matches counts selected lines.
 * With before == after == 0 the records equal those of gpugrep_scan_* with every id 0 (or gpugrep_invert_scan_*).
 * on_event == NULL counts selected lines and ignores context.  A build of the engine without context lines returns 7. */
#define GPUGREP_CONTEXT_ID 0xFFFFFFFFu
GPUGREP_API int gpugrep_context_scan_file(const char* file_name, const char* const* patterns, const unsigned int* pattern_flags,
                              const unsigned int* pattern_ids, unsigned int elements, hs_event on_event, int buffer_size,
                              int buffer_count, unsigned long long max_match_count, unsigned int before, unsigned int after,
                              int invert, gpugrep_stats* stats);
GPUGREP_API int gpugrep_context_scan_buffer(const void* data, size_t size, int location, const char* const* patterns,
                                const unsigned int* pattern_flags, const unsigned int* pattern_ids, unsigned int elements,
                                hs_event on_event, int buffer_size, int buffer_count, unsigned long long max_match_count,
                                unsigned int before, unsigned int after, int invert, void* stream, gpugrep_stats* stats);

/* ---- fixed strings (`grep -F`) ------------------------------------------------------------------------------------
 * `elements` >= 1 NUL-terminated, non-empty literals (byte strings, not patterns) with per-literal flags (NULL: all 0):
 * HS_FLAG_CASELESS (1) is honoured, 2, 4 and 8 are accepted and change nothing, any other bit, an empty literal or
 * elements == 0 return 4.  A pseudo-line is split as hyperscan() splits it and is SELECTED when its scanned block (leading
 * NULs skipped, cut at the next NUL, the trailing '\n' included) contains some literal as a contiguous substring.  Caseless
 * literals compare with ASCII folding of A-Z / a-z only: other bytes, >= 0x80 included, compare exactly ('@' is not '`').
 * So a literal ending in '\n' matches only at a line end, and one with a '\n' before its last byte never matches.
 * Records, batches, max_match_count, trailing context after the limit, GPUGREP_CONTEXT_ID, on_event == NULL counting and
 * every input form are those of gpugrep_context_scan_* for the same set with every byte written as \xHH, the flags as
 * given plus SINGLEMATCH and ids 0.  No automaton is built: the sample-tuned gram prefilter flags candidates, and a literal
 * index over its grams leads each gram hit to the few literals it can belong to, compared byte for byte.
 * gpugrep_check_literals checks a set on the host (0 or 4).  A build of the engine without the fixed-string stage returns 7. */
GPUGREP_API int gpugrep_literal_scan_file(const char* file_name, const char* const* literals, const unsigned int* literal_flags,
                              unsigned int elements, hs_event on_event, int buffer_size, int buffer_count,
                              unsigned long long max_match_count, unsigned int before, unsigned int after, int invert,
                              gpugrep_stats* stats);
GPUGREP_API int gpugrep_literal_scan_buffer(const void* data, size_t size, int location, const char* const* literals,
                                const unsigned int* literal_flags, unsigned int elements, hs_event on_event, int buffer_size,
                                int buffer_count, unsigned long long max_match_count, unsigned int before, unsigned int after,
                                int invert, void* stream, gpugrep_stats* stats);
GPUGREP_API int gpugrep_check_literals(const char* const* literals, const unsigned int* literal_flags, unsigned int elements);

/* ---- match END offsets (SURVEY.md section 8f-4: spans for `grep -o`) --------------------------------------------
 * The reference gets the spans of `-o` by re-running Python's re.finditer() over every matched line (utils.py:205-212);
 * Hyperscan itself reports (id, end offset) per match and the reference drops the offset (hyperscanner.c:83-102).
 * gpugrep_match_ends() keeps it: one record per (pseudo-line, pattern id, end offset) at which a match of that pattern
 * ends, in hs_scan order (by line, then end offset, then id).  `end` counts bytes from the start of the scanned block,
 * i.e. of the text hyperscan() would deliver as `line` (leading NULs skipped).  HS_FLAG_SINGLEMATCH is ignored here
 * (every end is reported).  At most `capacity` records are stored; *count is the number found, so a caller that gets
 * *count > capacity repeats the call with a larger array.  Returns 0 or a code of hyperscan(). */
typedef struct gpugrep_match_end {
    unsigned long long line_number; /* 0-based pseudo-line index inside `data` */
    unsigned int id;                /* pattern id                              */
    unsigned int end;               /* offset just behind the match            */
} gpugrep_match_end;

GPUGREP_API int gpugrep_match_ends(const void* data, size_t size, int location, const char* const* patterns,
                       const unsigned int* pattern_flags, const unsigned int* pattern_ids, unsigned int elements,
                       int buffer_size, gpugrep_match_end* out, size_t capacity, size_t* count, gpugrep_stats* stats);

/* Width in bytes of every match of `pattern` compiled WITHOUT flags (what the reference's re.compile(pattern) does for
 * `-o`), or -1 if matches can differ in width, can be empty, or the pattern uses syntax whose meaning differs between
 * Python's re and this compiler (then the caller keeps using re.finditer()).  For a fixed width w the span of a match
 * that ends at e is [e - w, e), and finditer()'s non-overlapping left-to-right selection is a greedy pass over the
 * sorted ends.  Host only (no CUDA). */
GPUGREP_API int gpugrep_span_width(const char* pattern);

/* 1 if `pattern` (compiled WITHOUT flags) is accepted by gpugrep_match_spans(), else 0.  Accepted patterns use only syntax that
 * Python's re and this compiler read the same way (literals, classes without POSIX names, . \d \D \w \W \b \B \A ^, groups
 * and (?:...), alternation, * + ? {m} {m,} {m,n} and their lazy forms); they cannot match the empty string, no repeated item
 * can match it either, and the span program has at most 128 instructions.  Rejected, among others: {,n}, $, \s, inline flags,
 * POSIX classes, possessive quantifiers and non-ASCII bytes.  Host only (no CUDA). */
GPUGREP_API int gpugrep_span_exact(const char* pattern);

/* ---- leftmost-first match spans (`grep -o` of any pattern that passes gpugrep_span_exact) ----------------------------------
 * One record per match, in line order and then start order.  For every pseudo-line (split as hyperscan() splits them), the
 * records of its scanned block (leading NULs skipped, cut at the next NUL, the trailing '\n' included) are, on every byte
 * value, exactly [m.span() for m in re.compile(pattern.encode()).finditer(block)]: the leftmost start, then the end a
 * backtracking matcher picks (greedy and lazy quantifiers and alternation order count), each search resuming at the previous
 * end.  Python's bytes patterns are ASCII, so on ASCII blocks the spans also equal those of the str finditer.  `pattern` is
 * compiled without flags; one that fails gpugrep_span_exact returns 4.  A block whose searches need more than
 * min(128 * (length + 1), 2^25) thread steps (searches that rescan the block, such as `a.*b|a` on a long run of `a`, or
 * programs near the instruction cap on long lines) yields one record with start == end == GPUGREP_SPAN_OVER_BUDGET and no
 * other record: the caller finds its spans another way.  Capacity, retry and return codes as gpugrep_match_ends().
 * A build of the engine without the span stage returns 7. */
#define GPUGREP_SPAN_OVER_BUDGET 0xFFFFFFFFu
typedef struct gpugrep_match_span {
    unsigned long long line_number; /* 0-based pseudo-line index inside `data` */
    unsigned int start;             /* offset of the first byte of the match   */
    unsigned int end;               /* offset just behind the match            */
} gpugrep_match_span;

GPUGREP_API int gpugrep_match_spans(const void* data, size_t size, int location, const char* pattern, int buffer_size,
                        gpugrep_match_span* out, size_t capacity, size_t* count, gpugrep_stats* stats);

/* An hs_event that discards its batch (benchmarks: full delivery path without a Python frame per batch). */
GPUGREP_API void gpugrep_discard_results(hyperscanner_result_t* results, int result_count);

/* Byte-range sharding helper for multi-GPU runs (SURVEY.md §8e): rank r of `world` scans
 * [gpugrep_shard_begin(r), gpugrep_shard_begin(r+1)) where each boundary is advanced to just past the next '\n'.
 * `data` is host memory. */
GPUGREP_API size_t gpugrep_shard_begin(const void* data, size_t size, unsigned int rank, unsigned int world);

/* Select the CUDA device used by subsequent calls of this process; -1 restores the default, which is $GPUGREP_DEVICE,
 * else $LOCAL_RANK, else round-robin over the visible GPUs (successive scans - one per file in multiscanner - take
 * successive devices). */
GPUGREP_API void gpugrep_set_device(int device);

/* Path of the libzstd shared object used for .zst ingest (default "libzstd.so.1"). */
GPUGREP_API void gpugrep_set_zstd_path(const char* path);

/* The host ingest alone - no GPU work: reads `file_name` the way hyperscan() would (plain, gzip members, zstd frames;
 * several decode threads for files of many members, GPUGREP_DECODE_THREADS=n to set their number, 0/1 for one thread)
 * and returns the number of text bytes and a hash of them.  For measuring the ingest (reference: gzopen()/gzgets(),
 * hyperscanner.c:189-199) and for checking the multi-threaded decode against the one-thread decode.  Returns 0 or 6. */
GPUGREP_API int gpugrep_ingest_probe(const char* file_name, unsigned long long* text_bytes, unsigned long long* text_hash);

/* Human-readable reason of the last failure on this thread ("" if none). */
GPUGREP_API const char* gpugrep_last_error(void);
GPUGREP_API const char* gpugrep_version(void);

/* ---- compiled-database introspection (pattern compiler tests, DESIGN.md tables) ---- */
typedef struct gpugrep_db gpugrep_db;

typedef struct gpugrep_db_info {
    unsigned int patterns;
    unsigned int groups;          /* DFA groups                                                     */
    unsigned int simple;          /* 1: every pattern SINGLEMATCH with one shared id                */
    unsigned int simple_id;
    unsigned int prefilter;       /* 1: literal prefilter enabled                                   */
    unsigned int prefilter_stride;
    unsigned int prefilter_fold;
    unsigned int prefilter_log2_bits;   /* log2 of buckets (exact table) or of bits (bloom bitmap) */
    unsigned int prefilter_grams;
    unsigned int prefilter_min_factor;
    unsigned int prefilter_lookback;    /* a match with a gram hit at q starts at or after q - lookback; 0xffffffff = unbounded */
    unsigned int total_states;
    unsigned int reserved;              /* 1: exact gram table, 0: bloom bitmap */
} gpugrep_db_info;

typedef struct gpugrep_group_info {
    unsigned int states;
    unsigned int classes;        /* byte classes; column `classes` is the end-of-data symbol */
    unsigned int stride;         /* classes + 1                                              */
    unsigned int first_accept;   /* states >= first_accept report                            */
    int sink_match;              /* simple mode: absorbing "matched" state, else -1          */
    int dead;                    /* absorbing non-reporting state, else -1                   */
    unsigned int accept_sets;
    unsigned int members;
    unsigned int entry_mid_other; /* entry state of a walk that starts after a non-word byte inside a line */
    unsigned int entry_mid_word;  /* ... after a word byte                                                  */
    unsigned int idle_end;        /* states < idle_end have no partial match in progress                   */
    unsigned int reserved;
} gpugrep_group_info;

GPUGREP_API gpugrep_db* gpugrep_db_compile(const char* const* patterns, const unsigned int* pattern_flags,
                               const unsigned int* pattern_ids, unsigned int elements, int* rc);
GPUGREP_API void gpugrep_db_free(gpugrep_db* db);
GPUGREP_API int gpugrep_db_get_info(const gpugrep_db* db, gpugrep_db_info* out);
GPUGREP_API int gpugrep_db_get_group(const gpugrep_db* db, unsigned int group, gpugrep_group_info* out);
/* Copies the tables of one group: byte_class[256], trans[states*stride], accept_of[states]. */
GPUGREP_API int gpugrep_db_copy_group(const gpugrep_db* db, unsigned int group, uint8_t* byte_class, uint32_t* trans,
                          uint32_t* accept_of);
/* depth[state] of `group` (no partial match in progress in that state began more than depth bytes ago; 255 = unbounded):
 * what lets a local verification walk stop early.  Writes up to cap bytes, returns the number of states. */
GPUGREP_API size_t gpugrep_db_copy_depth(const gpugrep_db* db, unsigned int group, uint8_t* depth, size_t cap);
/* Reports of accept set `accept` of `group`: writes up to cap (id, singlematch) pairs, returns the count. */
GPUGREP_API int gpugrep_db_accept_reports(const gpugrep_db* db, unsigned int group, unsigned int accept, unsigned int* ids,
                              unsigned int* singlematch, unsigned int cap);
/* Copies up to cap_words words of the bloom bitmap that the streaming kernel probes by default (nothing if words is NULL);
 * returns min(cap_words, bitmap words), 0 if the prefilter is disabled.  The bitmap has words * 32 bits
 * (prefilter_log2_bits reports the exact table's slots instead when that table exists).  *bloom_mul receives its
 * multiplier: gram g (OR-ed with 0x20202020 when prefilter_fold) hits iff, with p = g * bloom_mul mod 2^32, bit (p & 7) of
 * byte p >> (32 - (log2(words * 32) - 3)) is set. */
GPUGREP_API size_t gpugrep_db_copy_prefilter(const gpugrep_db* db, uint32_t* words, size_t cap_words, uint32_t* bloom_mul);
/* Copies up to cap exact prefilter grams (little-endian 4-byte windows); returns the total gram count. */
GPUGREP_API size_t gpugrep_db_copy_grams(const gpugrep_db* db, uint32_t* out, size_t cap);
/* Mixed sampling (prefilter_stride == 4 only): besides the table lookups at text offsets = 0 (mod 4), the streaming kernel
 * tests gram * mul + add == 0 (mod 2^32) at offsets = 2 (mod 4) for each of these (mul, add) pairs.  Writes up to cap
 * pairs (2 words each), returns the number of pairs (0..2). */
GPUGREP_API size_t gpugrep_db_copy_odd_compares(const gpugrep_db* db, uint32_t* mul_add_pairs, size_t cap);
/* Re-chooses the prefilter windows of a handle against the 4-gram histogram of a text sample (what the scan entry
 * points do with the head of their input); 0 on success. */
GPUGREP_API int gpugrep_db_tune(gpugrep_db* db, const void* sample, size_t size);
GPUGREP_API const char* gpugrep_db_prefilter_note(const gpugrep_db* db);

#ifdef __cplusplus
}
#endif
#endif /* GPUGREP_H */
