/*
 * ORACLE — TEST INFRASTRUCTURE ONLY.  Nothing shipped by hypergrep_b200 links, loads or calls this file.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * CPU restatement of the reference's scan path (pyranha-labs/hypergrep v3.2.0):
 *   hypergrep/lib/c/hyperscanner.c:83-102   hs_callback   -> port_emit()
 *   hypergrep/lib/c/hyperscanner.c:126-167  init_hs_db / check_patterns -> port_compile() / check_patterns()
 *   hypergrep/lib/c/hyperscanner.c:179-231  hyperscan_gz  -> port_scan_file()
 *   hypergrep/lib/c/hyperscanner.c:248-326  hyperscan     -> hyperscan()
 *
 * The regex arithmetic of the reference lives in Intel Hyperscan 5.4.2 (utils/build_hyperscanner.sh:9,49),
 * which is neither vendored nor installed (the libhs.so.5.4.2 blob is missing from the reference checkout), so
 * the reference itself cannot be built or run here.  The matcher below is a stand-in with the PCRE semantics
 * Hyperscan documents for its supported subset: PCRE2 10.42 (libpcre2-8.so.0, resolved with dlopen because the
 * image ships no pcre2.h), applied per pseudo-line exactly as hyperscanner.c:217 applies hs_scan:
 *   - block = one gzgets() result, trailing '\n' included, leading NULs stripped, cut at the first NUL;
 *   - a report is a (match id, END offset) pair; start offsets are irrelevant (the shim drops from/to);
 *   - HS_FLAG_SINGLEMATCH: at most one report per match id per block (hs_compile.h: "If a group of
 *     expressions sharing a match ID specify the flag, then at most one match with the match ID will be
 *     generated per stream"; block mode = one stream per block);
 *   - reports arrive ordered by end offset; ties are ordered by id here (Hyperscan leaves them unspecified).
 * "All end offsets" are computed with pcre2_dfa_match() anchored at every start offset, which enumerates the
 * regular-language ends (laziness/greed are irrelevant, as in Hyperscan).
 * Patterns Hyperscan rejects (look-around, back-references, atomic/possessive, conditionals, recursion,
 * verbs, \C \R \K \X \G, callouts, patterns matching the empty buffer, unknown flag bits) are rejected by
 * hs_would_reject() before PCRE2 ever sees them -> return code 4 (hyperscanner.c:162-164, 296-299).
 *
 * Pinning: this oracle passes the reference's own 53 native-path tests (hypergrep/test/test_hypergrep.py)
 * when injected under the unmodified reference Python (tests/test_oracle_reference_suite.py, run in the
 * build container), and the golden vectors extracted from that suite (tests/golden/reference_cases.json).
 * Everything beyond those vectors (the five BASELINE configs) is "parity unpinned" by the reference: no
 * Hyperscan binary exists here to generate vectors from.
 */
#define _GNU_SOURCE
#include <dlfcn.h>
#include <errno.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

/* ---- reference ABI (hyperscanner.c:25-56) ---- */
enum { PORT_COMPILE_MEM = 1, PORT_COMPILE = 2, PORT_SCRATCH = 3, PORT_DB = 4, PORT_STATE_MEM = 5, PORT_GZ_OPEN = 6, PORT_SCAN = 7 };
typedef struct { unsigned int id; unsigned long long line_number; char* line; } port_result_t;
typedef void (*port_event)(port_result_t* results, int result_count);

#define HS_FLAG_CASELESS 1u
#define HS_FLAG_DOTALL 2u
#define HS_FLAG_MULTILINE 4u
#define HS_FLAG_SINGLEMATCH 8u

/* ---- PCRE2 via dlopen ---- */
#define P2_CASELESS 0x00000008u
#define P2_DOTALL 0x00000020u
#define P2_MULTILINE 0x00000400u
#define P2_NEVER_UTF 0x00001000u
#define P2_NEVER_UCP 0x00000800u
#define P2_NO_AUTO_CAPTURE 0x00002000u
/* Without this PCRE2 turns a trailing `\w+` into the possessive `\w++`, and pcre2_dfa_match() then reports only the
   longest match from a start offset; Hyperscan reports EVERY end offset of a non-SINGLEMATCH expression (pcre2api:
   "PCRE2_NO_AUTO_POSSESS ... may also be needed if you want all matches from pcre2_dfa_match()"). */
#define P2_NO_AUTO_POSSESS 0x00004000u
/* Hyperscan's multiline ^ is "start of data or after ANY newline" (a streaming-capable engine cannot know that a newline is
   the last byte; SURVEY.md Appendix A), PCRE2's default excludes a newline that ends the subject: PCRE2_ALT_CIRCUMFLEX
   selects the Hyperscan behaviour. */
#define P2_ALT_CIRCUMFLEX 0x00200000u
#define P2_ANCHORED 0x80000000u
#define P2_JIT_COMPLETE 0x00000001u
#define P2_NOTEMPTY 0x00000004u
#define P2_ERROR_NOMATCH (-1)
typedef struct pcre2_real_code_8 p2_code;
typedef struct pcre2_real_match_data_8 p2_md;
static struct {
    void* h;
    p2_code* (*compile)(const unsigned char*, size_t, uint32_t, int*, size_t*, void*);
    void (*code_free)(p2_code*);
    int (*jit_compile)(p2_code*, uint32_t);
    int (*match)(const p2_code*, const unsigned char*, size_t, size_t, uint32_t, p2_md*, void*);
    int (*dfa_match)(const p2_code*, const unsigned char*, size_t, size_t, uint32_t, p2_md*, void*, int*, size_t);
    p2_md* (*md_create)(uint32_t, void*);
    p2_md* (*md_create_from)(const p2_code*, void*);
    void (*md_free)(p2_md*);
    size_t* (*ovector)(p2_md*);
    int (*pattern_info)(const p2_code*, uint32_t, void*);
} P2;

static int p2_load(void) {
    if (P2.h) return 0;
    void* h = dlopen("libpcre2-8.so.0", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { fprintf(stderr, "oracle: cannot load libpcre2-8.so.0: %s\n", dlerror()); return -1; }
#define SYM(field, name) do { *(void**)(&P2.field) = dlsym(h, name); if (!P2.field) { fprintf(stderr, "oracle: missing %s\n", name); return -1; } } while (0)
    SYM(compile, "pcre2_compile_8"); SYM(code_free, "pcre2_code_free_8"); SYM(jit_compile, "pcre2_jit_compile_8");
    SYM(match, "pcre2_match_8"); SYM(dfa_match, "pcre2_dfa_match_8"); SYM(md_create, "pcre2_match_data_create_8");
    SYM(md_create_from, "pcre2_match_data_create_from_pattern_8"); SYM(md_free, "pcre2_match_data_free_8");
    SYM(ovector, "pcre2_get_ovector_pointer_8"); SYM(pattern_info, "pcre2_pattern_info_8");
#undef SYM
    P2.h = h;
    return 0;
}

/* ---- Hyperscan accept/reject rules (SURVEY.md Appendix A; Hyperscan "Unsupported Constructs") ---- */
static int hs_would_reject(const char* p) {
    size_t n = strlen(p);
    int in_class = 0;
    for (size_t i = 0; i < n; i++) {
        char c = p[i];
        if (c == '\\') {
            char d = (i + 1 < n) ? p[i + 1] : 0;
            if (d == 0) return 1; /* trailing backslash */
            if (d == 'Q') { /* \Q...\E literal span */
                const char* e = strstr(p + i + 2, "\\E");
                if (!e) return 0; /* rest is literal */
                i = (size_t)(e - p) + 1;
                continue;
            }
            if (!in_class) {
                if (d >= '1' && d <= '9') return 1;                /* back-reference */
                if (d == 'g' || d == 'k') return 1;                 /* named/relative back-reference, subroutine */
                if (d == 'C' || d == 'R' || d == 'K' || d == 'X' || d == 'G') return 1;
                if (d == 'p' || d == 'P') return 1;                 /* unicode properties need UTF8/UCP mode */
            }
            i++;
            continue;
        }
        if (in_class) {
            if (c == ']') in_class = 0;
            continue;
        }
        if (c == '[') {
            in_class = 1;
            if (i + 1 < n && p[i + 1] == '^') i++;
            if (i + 1 < n && p[i + 1] == ']') i++; /* leading ] is literal */
            continue;
        }
        if (c == '{') { /* Hyperscan: "Bounded repeat is too large" above 32767 */
            size_t j = i + 1; unsigned long v = 0; int digits = 0, big = 0;
            while (j < n && ((p[j] >= '0' && p[j] <= '9') || p[j] == ',')) {
                if (p[j] == ',') { v = 0; } else { v = v * 10 + (unsigned long)(p[j] - '0'); digits++; if (v > 32767) big = 1; }
                j++;
            }
            if (j < n && p[j] == '}' && digits && big) return 1;
        }
        if (c == '(' && i + 1 < n && p[i + 1] == '*') return 1;      /* (*VERB) / (*UTF) */
        if (c == '(' && i + 1 < n && p[i + 1] == '?') {
            char d = (i + 2 < n) ? p[i + 2] : 0;
            char e = (i + 3 < n) ? p[i + 3] : 0;
            if (d == '=' || d == '!') return 1;                      /* look-ahead */
            if (d == '<' && (e == '=' || e == '!')) return 1;       /* look-behind */
            if (d == '>') return 1;                                  /* atomic group */
            if (d == '(') return 1;                                  /* conditional */
            if (d == 'R' || d == '&' || d == '+' || (d >= '0' && d <= '9')) return 1; /* recursion */
            if (d == '-' && e >= '0' && e <= '9') return 1;
            if (d == 'P' && (e == '=' || e == '>')) return 1;       /* named back-ref / subroutine */
            if (d == 'C') return 1;                                  /* callout */
            if (d == '|') return 1;                                  /* branch reset */
        }
        if ((c == '+') && i > 0) {
            char b = p[i - 1]; /* possessive: X*+ X++ X?+ X{..}+ (previous char unescaped quantifier) */
            int esc = (i >= 2 && p[i - 2] == '\\');
            if (!esc && (b == '*' || b == '+' || b == '?' || b == '}')) {
                /* "a++" : second '+' follows a quantifier. "a\++" handled by esc. "}" may be literal; PCRE2
                   would treat "x}+" as literal '}' repeated - rare; accept that imprecision in the oracle. */
                if (b != '}' ) return 1;
                /* only possessive if the '}' closes a real quantifier {n}, {n,}, {n,m} */
                size_t j = i - 1;
                while (j > 0 && p[j] != '{') j--;
                if (p[j] == '{') {
                    int ok = (j + 1 < i - 1);
                    for (size_t k = j + 1; k < i - 1; k++) if (!((p[k] >= '0' && p[k] <= '9') || p[k] == ',')) ok = 0;
                    if (ok) return 1;
                }
            }
        }
    }
    return 0;
}

/* ---- compiled pattern set ---- */
typedef struct {
    unsigned n;
    p2_code** code;     /* per pattern */
    p2_md** md;
    unsigned* ids;
    unsigned* flags;
    int simple;         /* all SINGLEMATCH + all ids equal -> existence test only */
    p2_code* merged;    /* simple mode: one alternation of everything (speeds the CPU baseline up) */
    p2_md* merged_md;
} port_db_t;

static void port_db_free(port_db_t* db) {
    if (!db) return;
    for (unsigned i = 0; i < db->n; i++) {
        if (db->md && db->md[i]) P2.md_free(db->md[i]);
        if (db->code && db->code[i]) P2.code_free(db->code[i]);
    }
    if (db->merged_md) P2.md_free(db->merged_md);
    if (db->merged) P2.code_free(db->merged);
    free(db->code); free(db->md); free(db->ids); free(db->flags); free(db);
}

static uint32_t p2_options(unsigned hs_flags) {
    uint32_t o = P2_NEVER_UTF | P2_NEVER_UCP | P2_ALT_CIRCUMFLEX | P2_NO_AUTO_POSSESS;
    if (hs_flags & HS_FLAG_CASELESS) o |= P2_CASELESS;
    if (hs_flags & HS_FLAG_DOTALL) o |= P2_DOTALL;
    if (hs_flags & HS_FLAG_MULTILINE) o |= P2_MULTILINE;
    return o;
}

/* hyperscanner.c:126-142 (hs_compile_multi) */
static port_db_t* port_compile(const char* const* patterns, const unsigned* flags, const unsigned* ids, unsigned n) {
    if (p2_load() != 0) return NULL;
    if (n == 0 || !patterns) return NULL;
    port_db_t* db = (port_db_t*)calloc(1, sizeof(*db));
    db->n = n;
    db->code = (p2_code**)calloc(n, sizeof(p2_code*));
    db->md = (p2_md**)calloc(n, sizeof(p2_md*));
    db->ids = (unsigned*)calloc(n, sizeof(unsigned));
    db->flags = (unsigned*)calloc(n, sizeof(unsigned));
    db->simple = 1;
    for (unsigned i = 0; i < n; i++) {
        unsigned f = flags ? flags[i] : 0;
        db->ids[i] = ids ? ids[i] : 0;
        db->flags[i] = f;
        if (f & ~(HS_FLAG_CASELESS | HS_FLAG_DOTALL | HS_FLAG_MULTILINE | HS_FLAG_SINGLEMATCH)) goto fail;
        if (!patterns[i] || !patterns[i][0]) goto fail;
        if (hs_would_reject(patterns[i])) goto fail;
        int err = 0; size_t eoff = 0;
        db->code[i] = P2.compile((const unsigned char*)patterns[i], strlen(patterns[i]), p2_options(f), &err, &eoff, NULL);
        if (!db->code[i]) goto fail;
        db->md[i] = P2.md_create(2048, NULL);
        /* "Pattern matches empty buffer; use HS_FLAG_ALLOWEMPTY": Hyperscan tests its graph for a start->accept
           edge, i.e. whether the pattern can match without consuming a byte, assertions notwithstanding (so a bare
           \b or ^ is vacuous too).  PCRE2_INFO_MATCHEMPTY (13) answers the same structural question. */
        {
            uint32_t can_be_empty = 0;
            if (P2.pattern_info(db->code[i], 13u, &can_be_empty) != 0 || can_be_empty) goto fail;
        }
        P2.jit_compile(db->code[i], P2_JIT_COMPLETE);
        if (!(f & HS_FLAG_SINGLEMATCH) || db->ids[i] != db->ids[0]) db->simple = 0;
    }
    /* hs_compile.h: expressions sharing an id must agree on SINGLEMATCH */
    for (unsigned i = 0; i < n; i++)
        for (unsigned j = i + 1; j < n; j++)
            if (db->ids[i] == db->ids[j] && ((db->flags[i] ^ db->flags[j]) & HS_FLAG_SINGLEMATCH)) goto fail;
    if (db->simple && n > 1) {
        /* (?flags:p1)|(?flags:p2)|... : same language as "any pattern matches"; falls back to the loop on failure */
        size_t len = 1;
        for (unsigned i = 0; i < n; i++) len += strlen(patterns[i]) + 20;
        char* buf = (char*)malloc(len);
        size_t o = 0;
        for (unsigned i = 0; i < n; i++) {
            unsigned f = db->flags[i];
            char on[4] = "", off[4] = "";
            strcat((f & HS_FLAG_CASELESS) ? on : off, "i");
            strcat((f & HS_FLAG_DOTALL) ? on : off, "s");
            strcat((f & HS_FLAG_MULTILINE) ? on : off, "m");
            o += (size_t)sprintf(buf + o, "%s(?%s%s%s:%s)", i ? "|" : "", on, off[0] ? "-" : "", off, patterns[i]);
        }
        int err = 0; size_t eoff = 0;
        db->merged = P2.compile((const unsigned char*)buf, o, P2_NEVER_UTF | P2_NEVER_UCP | P2_NO_AUTO_CAPTURE | P2_ALT_CIRCUMFLEX, &err, &eoff, NULL);
        free(buf);
        if (db->merged) {
            if (P2.jit_compile(db->merged, P2_JIT_COMPLETE) != 0) { P2.code_free(db->merged); db->merged = NULL; }
            else db->merged_md = P2.md_create(4, NULL);
        }
    }
    return db;
fail:
    port_db_free(db);
    return NULL;
}

/* hyperscanner.c:154-167 */
int check_patterns(const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids, const unsigned int elements) {
    port_db_t* db = port_compile(patterns, pattern_flags, pattern_ids, elements);
    if (!db) return PORT_DB;
    port_db_free(db);
    return 0;
}

/* ---- state (hyperscanner.c:64-72) ---- */
typedef struct {
    unsigned long long match_count, line_number;
    char* line;
    port_event callback;
    unsigned max_result_index;
    int result_index;
    port_result_t* results;
} port_state_t;

/* hyperscanner.c:83-102 */
static void port_emit(port_state_t* st, unsigned id) {
    st->match_count++;
    st->result_index++;
    int ri = st->result_index;
    st->results[ri].id = id;
    st->results[ri].line_number = st->line_number;
    strcpy(st->results[ri].line, st->line);
    if ((unsigned)st->result_index == st->max_result_index) {
        st->callback(st->results, st->result_index + 1);
        st->result_index = -1;
    }
}

typedef struct { size_t end; unsigned id; } port_ev_t;
static int ev_cmp(const void* a, const void* b) {
    const port_ev_t* x = (const port_ev_t*)a; const port_ev_t* y = (const port_ev_t*)b;
    if (x->end != y->end) return x->end < y->end ? -1 : 1;
    if (x->id != y->id) return x->id < y->id ? -1 : 1;
    return 0;
}

/* Every (end, id) at which a match of a pattern of `db` ends in the block, in hs_scan order (by end, then id), each pair
   once: every start offset is tried with an anchored DFA match, whose ovector lists all match ends from that start.
   *out is malloc()ed (free() it); returns 0 or PORT_SCAN. */
static int port_block_ends(port_db_t* db, const char* line, size_t len, port_ev_t** out, size_t* out_n) {
    size_t cap = 64, nev = 0;
    port_ev_t* ev = (port_ev_t*)malloc(cap * sizeof(*ev));
    uint32_t ovn = (uint32_t)(len + 2);
    p2_md* md = P2.md_create(ovn, NULL);
    size_t wsn = 4096 + 64 * len;
    int* ws = (int*)malloc(wsn * sizeof(int));
    unsigned char* seen = (unsigned char*)malloc(len + 1);
    for (unsigned i = 0; i < db->n; i++) {
        memset(seen, 0, len + 1);
        for (size_t s = 0; s < len; s++) {
            int rc = P2.dfa_match(db->code[i], (const unsigned char*)line, len, s, P2_ANCHORED, md, NULL, ws, wsn);
            if (rc == P2_ERROR_NOMATCH) continue;
            if (rc < 0) { fprintf(stderr, "oracle: pcre2_dfa_match error %d\n", rc); free(ev); free(ws); free(seen); P2.md_free(md); return PORT_SCAN; }
            size_t* ov = P2.ovector(md);
            int cnt = rc == 0 ? (int)ovn : rc;
            for (int k = 0; k < cnt; k++) {
                size_t e = ov[2 * k + 1];
                if (e == s) continue; /* zero-width matches are not reports (the simple path passes PCRE2_NOTEMPTY) */
                seen[e] = 1;
            }
        }
        for (size_t e = 1; e <= len; e++) if (seen[e]) {
            if (nev == cap) { cap *= 2; ev = (port_ev_t*)realloc(ev, cap * sizeof(*ev)); }
            ev[nev].end = e; ev[nev].id = db->ids[i]; nev++;
        }
    }
    free(ws); free(seen); P2.md_free(md);
    qsort(ev, nev, sizeof(*ev), ev_cmp);
    size_t u = 0;   /* one report per (id, end) */
    for (size_t k = 0; k < nev; k++)
        if (!u || ev[k].end != ev[u - 1].end || ev[k].id != ev[u - 1].id) ev[u++] = ev[k];
    *out = ev;
    *out_n = u;
    return 0;
}

/* stand-in for hs_scan(db, line, strlen(line), ...) at hyperscanner.c:217 */
static int port_scan_block(port_db_t* db, port_state_t* st, const char* line, size_t len) {
    if (len == 0) return 0;
    if (db->simple) {
        int hit = 0, rc = P2_ERROR_NOMATCH;
        if (db->merged) {
            rc = P2.match(db->merged, (const unsigned char*)line, len, 0, P2_NOTEMPTY, db->merged_md, NULL);
            hit = rc >= 0;
        }
        if (!db->merged || (rc < 0 && rc != P2_ERROR_NOMATCH)) {
            /* per-pattern loop; a backtracking-limit error (nested quantifiers) falls back to PCRE2's DFA matcher,
               which decides the same regular-language question without backtracking */
            for (unsigned i = 0; i < db->n && !hit; i++) {
                rc = P2.match(db->code[i], (const unsigned char*)line, len, 0, P2_NOTEMPTY, db->md[i], NULL);
                if (rc < 0 && rc != P2_ERROR_NOMATCH) {
                    size_t wsn = 4096 + 64 * len;
                    int* ws = (int*)malloc(wsn * sizeof(int));
                    rc = P2.dfa_match(db->code[i], (const unsigned char*)line, len, 0, P2_NOTEMPTY, db->md[i], NULL, ws, wsn);
                    free(ws);
                    if (rc < 0 && rc != P2_ERROR_NOMATCH) { fprintf(stderr, "oracle: pcre2 error %d\n", rc); return PORT_SCAN; }
                }
                hit = rc >= 0;
            }
        }
        if (hit) port_emit(st, db->ids[0]);
        return 0;
    }
    /* general mode: all (id, end) reports */
    port_ev_t* ev = NULL;
    size_t nev = 0;
    if (port_block_ends(db, line, len, &ev, &nev) != 0) return PORT_SCAN;
    /* SINGLEMATCH ids fire once per block */
    for (size_t k = 0; k < nev; k++) {
        int sm = 0;
        for (unsigned i = 0; i < db->n; i++) if (db->ids[i] == ev[k].id) { sm = (db->flags[i] & HS_FLAG_SINGLEMATCH) != 0; break; }
        if (sm) {
            int dup = 0;
            for (size_t j = 0; j < k && !dup; j++) dup = (ev[j].id == ev[k].id);
            if (dup) continue;
        }
        port_emit(st, ev[k].id);
    }
    free(ev);
    return 0;
}

/* ---- zstd via dlopen (the reference links zstd 1.5.5's zlibWrapper, build_hyperscanner.sh:76-89) ---- */
typedef struct { const void* src; size_t size; size_t pos; } zs_in;
typedef struct { void* dst; size_t size; size_t pos; } zs_out;
static unsigned char* zstd_slurp(const unsigned char* src, size_t n, size_t* out_n) {
    void* h = dlopen("libzstd.so.1", RTLD_NOW);
    if (!h) return NULL;
    void* (*create)(void) = (void* (*)(void))dlsym(h, "ZSTD_createDStream");
    size_t (*dec)(void*, zs_out*, zs_in*) = (size_t (*)(void*, zs_out*, zs_in*))dlsym(h, "ZSTD_decompressStream");
    size_t (*freeds)(void*) = (size_t (*)(void*))dlsym(h, "ZSTD_freeDStream");
    unsigned (*is_err)(size_t) = (unsigned (*)(size_t))dlsym(h, "ZSTD_isError");
    if (!create || !dec || !freeds || !is_err) return NULL;
    void* ds = create();
    size_t cap = n * 4 + 65536, o = 0;
    unsigned char* dst = (unsigned char*)malloc(cap);
    zs_in in = { src, n, 0 };
    while (in.pos < in.size) {
        if (cap - o < 65536) { cap *= 2; dst = (unsigned char*)realloc(dst, cap); }
        zs_out out = { dst + o, cap - o, 0 };
        size_t r = dec(ds, &out, &in);
        o += out.pos;
        if (is_err(r)) break; /* zlibWrapper: gzgets returns NULL on error -> loop ends */
        if (r == 0 && in.pos < in.size) {
            /* frame finished: zlibWrapper's gz_look() (gzread.c) continues only on another gzip / zstd header; anything else -
               a skippable frame included - is trailing garbage and ends the data */
            if (in.size - in.pos < 4 || memcmp((const unsigned char*)in.src + in.pos, "\x28\xb5\x2f\xfd", 4) != 0) break;
        }
    }
    freeds(ds);
    *out_n = o;
    return dst;
}

/* NUL handling of hyperscanner.c:205-214 then strlen at :217 */
static char* port_strip(char* buf, int buffer_size) {
    char* line = buf;
    if (buf[0] == 0) {
        for (int s = 1; s < buffer_size; s++) {
            if (buf[s] != 0) { line = buf + s; break; }
        }
    }
    return line;
}

/* hyperscanner.c:179-231 */
static int port_scan_file(const char* file_name, port_state_t* st, port_db_t* db, int buffer_size, unsigned long long max_match_count) {
    int ret = 0;
    char* buf = (char*)calloc((size_t)buffer_size + 1, 1);
    /* sniff for zstd: zstd's zlibWrapper routes by magic, everything else goes to zlib (gzip or transparent) */
    unsigned char magic[4] = { 0, 0, 0, 0 };
    FILE* f = fopen(file_name, "rb");
    size_t got = f ? fread(magic, 1, 4, f) : 0;
    if (f && got == 4 && memcmp(magic, "\x28\xb5\x2f\xfd", 4) == 0) {
        fseek(f, 0, SEEK_END); long sz = ftell(f); fseek(f, 0, SEEK_SET);
        unsigned char* raw = (unsigned char*)malloc((size_t)sz);
        if (fread(raw, 1, (size_t)sz, f) != (size_t)sz) { sz = 0; }
        fclose(f);
        size_t n = 0;
        unsigned char* text = zstd_slurp(raw, (size_t)sz, &n);
        free(raw);
        if (!text) { free(buf); return PORT_GZ_OPEN; }
        size_t pos = 0;
        while (pos < n) {
            /* gzgets(): up to buffer_size-1 bytes, stop after '\n' */
            size_t lim = (size_t)buffer_size - 1, k = 0;
            while (k < lim && pos + k < n) { buf[k] = (char)text[pos + k]; k++; if (buf[k - 1] == '\n') break; }
            buf[k] = 0; pos += k;
            st->line = port_strip(buf, buffer_size);
            if ((ret = port_scan_block(db, st, st->line, strlen(st->line))) != 0) break;
            if (max_match_count > 0 && st->match_count >= max_match_count) break;
            st->line_number++;
        }
        free(text); free(buf);
        return ret;
    }
    if (f) fclose(f);
    gzFile in = gzopen(file_name, "rb");
    if (in == Z_NULL) ret = PORT_GZ_OPEN;
    while (in != Z_NULL) {
        st->line = gzgets(in, buf, buffer_size);
        if (st->line == Z_NULL) break;
        st->line = port_strip(buf, buffer_size);
        if (port_scan_block(db, st, st->line, strlen(st->line)) != 0) { ret = PORT_SCAN; break; }
        if (max_match_count > 0 && st->match_count >= max_match_count) break;
        st->line_number++;
    }
    if (in != Z_NULL) gzclose(in);
    free(buf);
    return ret;
}

/* hyperscanner.c:248-326 */
int hyperscan(char* file_name, const char* const* patterns, const unsigned int* pattern_flags, const unsigned int* pattern_ids,
              const unsigned int elements, port_event on_event, const int buffer_size, int buffer_count, unsigned long long max_match_count) {
    if (max_match_count > 0 && max_match_count < (unsigned long long)buffer_count) buffer_count = (int)max_match_count;
    int ret = 0;
    port_db_t* db = NULL;
    int allocated = 0;
    port_state_t* st = (port_state_t*)calloc(1, sizeof(*st));
    if (!st) return PORT_STATE_MEM;
    st->callback = on_event;
    st->result_index = -1;
    st->max_result_index = (unsigned)(buffer_count - 1);
    int max_results = (int)st->max_result_index + 1;
    st->results = (port_result_t*)calloc((size_t)max_results, sizeof(port_result_t));
    if (!st->results) { ret = PORT_COMPILE_MEM; goto cleanup; }
    for (int i = 0; i < max_results; i++) {
        st->results[i].line = (char*)malloc((size_t)buffer_size);
        if (!st->results[i].line) { ret = PORT_COMPILE_MEM; goto cleanup; }
        allocated++;
    }
    db = port_compile(patterns, pattern_flags, pattern_ids, elements);
    if (!db) { fprintf(stderr, "ERROR: Unable to create database. Exiting.\n"); ret = PORT_DB; goto cleanup; }
    ret = port_scan_file(file_name, st, db, buffer_size, max_match_count);
    if (st->result_index != -1) st->callback(st->results, st->result_index + 1);
cleanup:
    for (int i = 0; i < allocated; i++) free(st->results[i].line);
    free(st->results);
    free(st);
    port_db_free(db);
    return ret;
}

/* ---- extra entry for tests/bench: scan a memory buffer as if it were the (decompressed) file, count only.
 * Same loop as port_scan_file; used by bench.py's cpu_baseline leg so that page-cache reads are not timed. ---- */
typedef struct { unsigned long long matches; unsigned long long lines; } port_count_t;
static void count_cb(port_result_t* r, int n) { (void)r; (void)n; }
int oracle_count_buffer(const char* text, size_t n, const char* const* patterns, const unsigned int* flags, const unsigned int* ids,
                        unsigned elements, int buffer_size, unsigned long long* out_matches, unsigned long long* out_lines) {
    port_db_t* db = port_compile(patterns, flags, ids, elements);
    if (!db) return PORT_DB;
    port_state_t st; memset(&st, 0, sizeof(st));
    port_result_t slot; slot.line = (char*)malloc((size_t)buffer_size);
    st.callback = count_cb; st.result_index = -1; st.max_result_index = 0; st.results = &slot;
    char* buf = (char*)calloc((size_t)buffer_size + 1, 1);
    size_t pos = 0; int ret = 0;
    while (pos < n) {
        size_t lim = (size_t)buffer_size - 1;
        size_t avail = n - pos < lim ? n - pos : lim;
        const char* nl = (const char*)memchr(text + pos, '\n', avail);
        size_t k = nl ? (size_t)(nl - (text + pos)) + 1 : avail;
        memcpy(buf, text + pos, k); buf[k] = 0; pos += k;
        st.line = port_strip(buf, buffer_size);
        if ((ret = port_scan_block(db, &st, st.line, strlen(st.line))) != 0) break;
        st.line_number++;
    }
    *out_matches = st.match_count; *out_lines = st.line_number;
    free(buf); free(slot.line); port_db_free(db);
    return ret;
}

/* ---- test/bench extension: like oracle_count_buffer, and the line number of every delivered result is written to
 * out_line_numbers[0, cap) in delivery order (bench.py compares them with the GPU's on the text it times). ---- */
static __thread unsigned long long* g_sink = NULL;
static __thread unsigned long long g_sink_cap = 0, g_sink_len = 0;
static void sink_cb(port_result_t* r, int n) {
    for (int i = 0; i < n; i++) {
        if (g_sink_len < g_sink_cap) g_sink[g_sink_len] = r[i].line_number;
        g_sink_len++;
    }
}
int oracle_lines_buffer(const char* text, size_t n, const char* const* patterns, const unsigned int* flags, const unsigned int* ids,
                        unsigned elements, int buffer_size, unsigned long long* out_line_numbers, unsigned long long cap,
                        unsigned long long* out_matches, unsigned long long* out_lines) {
    port_db_t* db = port_compile(patterns, flags, ids, elements);
    if (!db) return PORT_DB;
    port_state_t st; memset(&st, 0, sizeof(st));
    port_result_t slot; slot.line = (char*)malloc((size_t)buffer_size);
    g_sink = out_line_numbers; g_sink_cap = cap; g_sink_len = 0;
    st.callback = sink_cb; st.result_index = -1; st.max_result_index = 0; st.results = &slot;
    char* buf = (char*)calloc((size_t)buffer_size + 1, 1);
    size_t pos = 0; int ret = 0;
    while (pos < n) {
        size_t lim = (size_t)buffer_size - 1;
        size_t avail = n - pos < lim ? n - pos : lim;
        const char* nl = (const char*)memchr(text + pos, '\n', avail);
        size_t k = nl ? (size_t)(nl - (text + pos)) + 1 : avail;
        memcpy(buf, text + pos, k); buf[k] = 0; pos += k;
        st.line = port_strip(buf, buffer_size);
        if ((ret = port_scan_block(db, &st, st.line, strlen(st.line))) != 0) break;
        st.line_number++;
    }
    *out_matches = st.match_count; *out_lines = st.line_number;
    g_sink = NULL;
    free(buf); free(slot.line); port_db_free(db);
    return ret;
}

/* ---- test extension: what gpugrep_match_ends() promises (include/gpugrep.h), from the same pseudo-lines, strip rule and
 * hs_scan order as the scans above: one (line, id, end) per match end, SINGLEMATCH cleared, `end` counted from the start
 * of the scanned block.  At most `capacity` records are written to `out`; *count is the number found. ---- */
typedef struct { unsigned long long line_number; unsigned int id; unsigned int end; } port_match_end_t;
int oracle_ends_buffer(const char* text, size_t n, const char* const* patterns, const unsigned int* flags, const unsigned int* ids,
                       unsigned elements, int buffer_size, port_match_end_t* out, unsigned long long capacity, unsigned long long* count) {
    unsigned* cleared = (unsigned*)malloc((elements ? elements : 1) * sizeof(unsigned));
    for (unsigned i = 0; i < elements; i++) cleared[i] = (flags ? flags[i] : 0u) & ~HS_FLAG_SINGLEMATCH;
    port_db_t* db = port_compile(patterns, cleared, ids, elements);
    free(cleared);
    if (!db) return PORT_DB;
    char* buf = (char*)calloc((size_t)buffer_size + 1, 1);
    unsigned long long line_number = 0, found = 0;
    size_t pos = 0; int ret = 0;
    while (pos < n) {
        size_t lim = (size_t)buffer_size - 1;
        size_t avail = n - pos < lim ? n - pos : lim;
        const char* nl = (const char*)memchr(text + pos, '\n', avail);
        size_t k = nl ? (size_t)(nl - (text + pos)) + 1 : avail;
        memcpy(buf, text + pos, k); buf[k] = 0; pos += k;
        const char* line = port_strip(buf, buffer_size);
        size_t len = strlen(line);
        if (len) {
            port_ev_t* ev = NULL;
            size_t nev = 0;
            if ((ret = port_block_ends(db, line, len, &ev, &nev)) != 0) break;
            for (size_t e = 0; e < nev; e++, found++)
                if (found < capacity) { out[found].line_number = line_number; out[found].id = ev[e].id; out[found].end = (unsigned)ev[e].end; }
            free(ev);
        }
        line_number++;
    }
    *count = found;
    free(buf); port_db_free(db);
    return ret;
}
