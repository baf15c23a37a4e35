/*
 * ugrep_b200.h — C ABI of the B200-native buffer-scan path for ugrep.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no C plugin
 * ABI; its boundary is the C++ pair reflex::Pattern / reflex::Matcher.  The
 * functions below are what a patched reflex::Matcher binds (see
 * INTEGRATION.md): the compiled pattern tables go in once, a buffer goes in per
 * file, and counts / (line, offset, length, accept) records come back.
 *
 * Everything is plain pointers and sizes.  There is NO CPU fallback: every scan
 * entry point runs sm_100a CUDA kernels or returns a non-zero status.
 *
 * Reference interfaces replaced (all paths into /root/reference):
 *   ugx_pattern_create    reflex::Pattern tables as consumed by reflex::Matcher
 *                         (include/reflex/pattern.h:1288-1334; the (code, pred)
 *                         constructor pattern.h:151-159, loader lib/pattern.cpp:199-274)
 *   ugx_count_lines       `ugrep -c`    loop, src/ugrep.cpp:10567-10586  (find + skip('\n'))
 *   ugx_count_matches     `ugrep -c -o` loop, src/ugrep.cpp:10536-10566  (find)
 *   ugx_find_all          `ugrep -o [-n -b]` loop, src/ugrep.cpp:10857-11047 and the
 *                         state Output::header reads (lineno(), first(), begin(), size();
 *                         include/reflex/absmatcher.h:695-766, :901-905)
 *   ugx_count_newlines    reflex::nlcount, lib/simd.cpp:62-166
 * each of which is a loop over reflex::Matcher::match(FIND), lib/matcher.cpp:42-750,
 * with the prefilters of lib/matcher.cpp:797-3549 / lib/matcher_avx2.cpp.
 */
#ifndef UGREP_B200_H
#define UGREP_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UGX_ABI_VERSION 2

/* status codes (0 = ok; nothing ever falls back to the CPU) */
enum {
  UGX_OK            = 0,
  UGX_E_INVALID     = 1, /* bad argument / malformed pattern tables */
  UGX_E_UNSUPPORTED = 2, /* pattern uses a feature outside the path's scope (HEAD/TAIL lookahead, REDO, '\n' transitions, ...) */
  UGX_E_CUDA        = 3, /* CUDA runtime error, see ugx_last_error() */
  UGX_E_NOMEM       = 4, /* host or device allocation failed */
  UGX_E_OVERFLOW    = 5, /* caller's record buffer too small: *n_out holds the required count */
  UGX_E_IO          = 6  /* pattern file unreadable */
};

/* reflex::Matcher option letters (include/reflex/absmatcher.h:354-388) */
#define UGX_OPT_N 0x01u /* "N": accept empty matches (ugrep -Y) */
#define UGX_OPT_W 0x02u /* "W": whole-word matching (ugrep -w) */

#define UGX_BTAP 2048 /* reflex::Pattern::Const::BTAP */
#define UGX_HASH 4096 /* reflex::Pattern::Const::HASH */

/*
 * The prefilter block of a compiled reflex::Pattern: a field-for-field image of
 * the members reflex::Matcher reads (include/reflex/pattern.h:1305-1334).
 * bit/tap/pma/pmh hold the in-memory values (a 0 bit = "may match").
 */
typedef struct ugx_prefilter {
  uint32_t len;  /* len_: length of the literal prefix in chr[] (0 = none) */
  uint32_t min;  /* min_: minimum length of what follows the prefix, 0..8 */
  uint32_t pin;  /* pin_: number of needle bytes per needle position, 0..16 */
  uint32_t lcp;  /* lcp_: primary needle position */
  uint32_t lcs;  /* lcs_: secondary needle position */
  uint32_t bmd;  /* bmd_: Boyer-Moore distance (>0 selects the B-M routines) */
  uint32_t npy;  /* npy_: bitap entropy */
  uint32_t one;  /* one_: pattern is the single literal chr[0..len) */
  uint32_t bol;  /* bol_: every alternative is anchored with ^ */
  uint32_t lbk;  /* lbk_: look-back distance, 0xffff = unbounded, 0 = none */
  uint32_t lbm;  /* lbm_: minimum look-back distance */
  uint32_t cut;  /* cut_: DFA s-t cut depth (informational) */
  uint8_t  chr[256];      /* chr_: literal prefix, or 2*pin needle bytes */
  uint8_t  bit[256];      /* bit_ */
  uint8_t  tap[UGX_BTAP]; /* tap_: bitap hashed byte pairs */
  uint8_t  pma[UGX_HASH]; /* pma_: PM4 predictor (min < 4) */
  uint8_t  pmh[UGX_HASH]; /* pmh_: hashed Bloom predictor (min >= 4) */
  uint8_t  cbk[32];       /* cbk_ as a 256-bit little-endian bitset */
  uint8_t  fst[32];       /* fst_ as a 256-bit little-endian bitset */
  uint8_t  bms[256];      /* bms_: Boyer-Moore shifts */
} ugx_prefilter;

/* UGXP container: header, ugx_prefilter, nop opcode words, regex text (informational) */
#define UGX_FILE_MAGIC "UGXP\1\0\0\0"
typedef struct ugx_file_header {
  char     magic[8];
  uint32_t nop;            /* number of 32-bit opcode words */
  uint32_t regex_len;      /* bytes of regex text after the opcode words */
  uint32_t prefilter_size; /* sizeof(ugx_prefilter) at write time */
  uint32_t matcher_flags;  /* UGX_OPT_* the pattern was meant to be used with */
} ugx_file_header;

/* one match, in input order: what lineno()/first()/size()/accept() return for it */
typedef struct ugx_match {
  uint64_t line;   /* 1-based line number of the match start (+ base_line) */
  uint64_t offset; /* 0-based byte offset of the match start (+ base_offset) */
  uint32_t len;    /* length in bytes */
  uint32_t cap;    /* accept index: 1-based alternative number */
} ugx_match;

/* one line, in input order: what lineno()/bol()/eol() return for it, and the first match on it (the match the `ugrep -c`
 * loop finds before it skips to the next line) */
typedef struct ugx_line {
  uint64_t line;   /* 1-based line number (+ base_line) */
  uint64_t bol;    /* offset of the line's first byte (+ base_offset) */
  uint64_t eol;    /* offset of its '\n', or the buffer end for an unterminated last line (+ base_offset) */
  uint64_t offset; /* first match on the line (first()); = bol for UGX_LINES_INVERT records */
  uint32_t len;    /* its size(); 0 for UGX_LINES_INVERT records */
  uint32_t cap;    /* its accept(); 0 = the line has no match */
} ugx_line;        /* 40 bytes */

#define UGX_LINES_INVERT 1u /* ugx_find_lines*: the lines WITHOUT a match (`ugrep -v`) */

/* facts about an uploaded pattern */
typedef struct ugx_pattern_info {
  uint32_t nop;          /* opcode words */
  uint32_t states;       /* reachable DFA states after flattening */
  uint32_t classes;      /* byte equivalence classes */
  uint32_t table_bytes;  /* dense transition table size */
  uint32_t table_in_smem;/* 1 if the scan kernels stage the table in shared memory */
  uint32_t advance;      /* UGX_ADV_* prefilter routine selected (init_advance, lib/matcher.cpp:797-954) */
  uint32_t has_meta;     /* DFA has META (anchor / word boundary) edges */
  uint32_t lookback;     /* lbk != 0 */
} ugx_pattern_info;

/* prefilter routine families of Matcher::init_advance (lib/matcher.cpp:797-954) */
enum {
  UGX_ADV_NONE = 0,
  UGX_ADV_PIN1_ONE, UGX_ADV_PIN1_PMA, UGX_ADV_PIN1_PMH,
  UGX_ADV_PIN_ONE,  UGX_ADV_PIN_PMA,  UGX_ADV_PIN_PMH,
  UGX_ADV_MIN1, UGX_ADV_MIN2, UGX_ADV_MIN3, UGX_ADV_MIN4, UGX_ADV_PMA,
  UGX_ADV_CHAR, UGX_ADV_CHAR_PMA, UGX_ADV_CHAR_PMH,
  UGX_ADV_STRING, UGX_ADV_STRING_PMA, UGX_ADV_STRING_PMH
};

/* what the host-side export derives from a compiled pattern, without touching a device: the dense DFA's shape and the
 * first-stage filter the position-parallel kernels use (csrc/filter_plan.hpp).  For tests and diagnostics. */
typedef struct ugx_plan_info {
  uint32_t states, classes, table_bytes;
  uint32_t first_acc, first_leaf; /* state numbering: [1, first_acc) plain, [first_acc, first_leaf) accepting, rest leaves */
  uint32_t max_match_len;         /* longest match in bytes, 0xffffffff = unbounded (cyclic DFA) */
  uint32_t advance;               /* UGX_ADV_* */
  uint32_t has_meta, newline_live;
  uint32_t kind;                  /* 0 all survive, 2 two literal anchors, 3 byte-set terms */
  uint32_t nterms, t_off[3];      /* byte-set terms: byte (k + t_off[t]) must not have bit 8*t set in lut[] */
  uint32_t a_off[2], a_chr[2];    /* literal anchors: offsets and bytes */
  uint32_t h4_terms, h4_shift;    /* hashed-predictor terms (steps 3.. of predict_match PMH) */
  uint32_t pm2, pm2_shift;        /* PM4 two-byte term */
  uint32_t lut[256];
  uint32_t covers;                /* proven by enumeration: every position that starts a non-empty match passes the
                                     routine's candidate test (so `-c` may skip the test); 0 = not proven or not so */
} ugx_plan_info;

enum { UGX_MODE_LINES = 0, UGX_MODE_MATCHES = 1, UGX_MODE_RECORDS = 2 }; /* ugrep -c | -c -o | -o -n -b */

typedef struct ugx_pattern ugx_pattern; /* immutable once created; shareable between host threads */
typedef struct ugx_scanner ugx_scanner; /* per host thread / per stream scratch (counters, record arena) */

/* totals every scan reports */
typedef struct ugx_totals {
  uint64_t matches;        /* count-lines: matching lines; otherwise: matches */
  uint64_t newlines;       /* '\n' bytes in the buffer (line-number base for the next shard); valid when flags has
                              UGX_TOT_NEWLINES: every call except ugx_count_lines on its streaming kernels, which
                              count newlines only with the scanner option "count_newlines" */
  uint64_t flags;          /* UGX_TOT_* */
  float    kernel_ms;      /* device time of the scan kernels (CUDA events on the scan stream) */
  uint32_t launches;       /* kernels launched by this call */
  uint32_t kernel;         /* UGX_K_*: the scan kernel that did the work (ugx_kernel_name) */
} ugx_totals;

#define UGX_TOT_NEWLINES      1u /* `newlines` was counted by this call */
#define UGX_TOT_SPAN_HANDOVER 2u /* the span kernels could not vouch for this buffer (a match longer than a window across
                                    a region start in a line without newlines, a look-back run or match beyond their
                                    bounds, a failed attempt at the very end): the line-at-a-time kernels did the scan */

/* scan kernels (reported in ugx_totals.kernel; DESIGN.md section 4) */
enum { UGX_K_NONE = 0, UGX_K_STREAM_LITERAL = 1, UGX_K_STREAM_DFA = 2, UGX_K_TILE_ANY = 3, UGX_K_LINE_SCAN = 4,
       UGX_K_RECORDS = 5, UGX_K_NEWLINES = 6, UGX_K_MATCH_LINES = 7, UGX_K_SPAN = 8, UGX_K_BATCH = 9,
       UGX_K_SPAN_LINES = 10, UGX_K_STREAM_SEARCH = 11, UGX_K_BOOL_LINES = 12 };

const char *ugx_last_error(void);
const char *ugx_kernel_name(uint32_t id);
int  ugx_abi_version(void);

/* pattern: flatten the opcode table to a dense class-compressed DFA and upload it with the prefilter tables */
int  ugx_pattern_create(const uint32_t *opc, uint32_t nop, const ugx_prefilter *pf,
                        uint32_t matcher_flags, int device, ugx_pattern **out);
int  ugx_pattern_load(const char *path, int device, ugx_pattern **out);
/* host only: the compiled form of ONE fixed string (`ugrep -F 'literal'`): the opcode words and prefilter fields the
 * reference's pattern compiler produces for it (lib/pattern.cpp:2823-3063, 4286-4340, 510-598), byte for byte, so that
 * a literal search needs no reference binary.  *nop receives the word count (UGX_E_OVERFLOW when cap is too small);
 * UGX_E_UNSUPPORTED for an empty literal, 255 bytes or more, or one that holds NUL / CR / LF.  The general regex and
 * word-list compiler is not part of this library. */
int  ugx_compile_literal(const uint8_t *literal, uint32_t len, uint32_t *opc, uint32_t cap, uint32_t *nop,
                         ugx_prefilter *pf);
/* host only: the same for a LIST of fixed strings (`ugrep -F -f words.txt`, `-F -e A -e B`; accept index = 1-based
 * position in the list): the tree DFA's opcode words and the needle / bitap / hashed-predictor tables, byte for byte
 * what the reference compiles (lib/pattern.cpp:798-866, 3812-4639, 331-598, 2764-3063).  UGX_E_UNSUPPORTED: an empty
 * string, NUL / CR / LF in a string, or a list for which the reference's DFA analysis makes a cut (look-back search:
 * that part of the analysis is not restated). */
int  ugx_compile_words(const uint8_t *const *words, const uint32_t *lens, uint32_t nwords, uint32_t *opc, uint32_t cap,
                       uint32_t *nop, ugx_prefilter *pf);
/* the same with options: UGX_COMPILE_ICASE = `ugrep -F -i -f words.txt` (the strings are lowered as they enter the tree
 * and every edge on a lowercase ASCII letter gets an uppercase twin, lib/pattern.cpp:286-311, 834) */
enum { UGX_COMPILE_ICASE = 1 };
int  ugx_compile_words_ex(const uint8_t *const *words, const uint32_t *lens, uint32_t nwords, uint32_t options,
                          uint32_t *opc, uint32_t cap, uint32_t *nop, ugx_prefilter *pf);
/* host only: a REGEX that is an alternation of plain strings — `ugrep [-i] -e 'foo\.bar|baz'` without -F.  The
 * reference's parser puts such a regex into the same tree DFA as a -F list (lib/pattern.cpp:286-311, 798-866), so this
 * is ugx_compile_words_ex on the alternatives.  Accepted: bytes other than the operators \ . [ ] ( ) { } * + ? | ^ $,
 * top-level `|`, a backslash before an operator or one of ! " # % & ' , - / : ; @ ` (that character), \t \f \v \a,
 * \Q...\E, a leading (?i) (= UGX_COMPILE_ICASE); with UGX_COMPILE_ICASE no byte >= 0x80 outside \Q...\E.  Anything else (classes, groups, repeats, anchors,
 * \d \w \b \xHH ...) returns UGX_E_UNSUPPORTED: the regex compiler proper is not part of this library.  Alternative i (1-based) is accept index i. */
int  ugx_compile_plain_regex(const uint8_t *regex, uint32_t len, uint32_t options, uint32_t *opc, uint32_t cap,
                             uint32_t *nop, ugx_prefilter *pf);
/* host only (no device needed): DFA export + filter plan of a compiled pattern */
int  ugx_plan_describe(const uint32_t *opc, uint32_t nop, const ugx_prefilter *pf, uint32_t matcher_flags,
                       ugx_plan_info *out);
/* host only: the k-gram viability tables of the scan kernels (csrc/pattern_host.hpp).  *k = bytes looked at (0 = no
 * table), *stride = bits per state code, t01[256] / t23[256] = the pre-multiplied byte ids, pair[cap_pair] = the
 * two-byte state codes, bits[cap_words] = the bit table; *npair / *words = their sizes */
int  ugx_viability_describe(const uint32_t *opc, uint32_t nop, uint32_t *k, uint32_t *stride, uint32_t *t01, uint32_t *t23,
                            uint8_t *pair, uint32_t cap_pair, uint32_t *npair,
                            uint32_t *bits, uint32_t cap_words, uint32_t *words);
/* host only: the line-resetting search automaton that `-c` runs in count_lines_search_kernel (csrc/pattern_host.hpp
 * SearchDfa, DESIGN.md 4.3a).  A state is MATCHED or the set of anchored DFA states of the line's still undecided
 * attempts; per byte: state = table[state + cls[byte]], success = (state == 0); the empty set is state offset `classes`.
 * out->eligible = 1 when `-c` takes the kernel (scanner option "no_search" aside); else out->refusal says why
 * (UGX_SEARCH_*).  cls[256] and table[cap] (u16 pre-multiplied row offsets, states * classes entries) are filled
 * when the automaton was built (refusal UGX_SEARCH_OK or UGX_SEARCH_ROUTE) and the pointers are not NULL;
 * UGX_E_OVERFLOW when cap is too small. */
enum { UGX_SEARCH_OK = 0, UGX_SEARCH_META = 1, UGX_SEARCH_ACC0 = 2, UGX_SEARCH_CYCLE = 3, UGX_SEARCH_DEPTH = 4,
       UGX_SEARCH_NEWLINE = 5, UGX_SEARCH_SIZE = 6, UGX_SEARCH_ROUTE = 7 };
typedef struct ugx_search_info {
  uint32_t eligible;
  uint32_t refusal;      /* UGX_SEARCH_*: META edges, accepting start state, cyclic or too deep undecided graph,
                            a live '\n' edge, table over 128 KiB, or not on the streaming `-c` DFA route (look-back,
                            option W, no prefilter, a literal's `one`, a candidate test not proven implied) */
  uint32_t depth;        /* decision depth D: an attempt has decided after at most D bytes (0 = not bounded) */
  uint32_t states;       /* minimised, MATCHED and the empty set included */
  uint32_t classes;
  uint32_t table_bytes;
} ugx_search_info;
int  ugx_search_describe(const uint32_t *opc, uint32_t nop, const ugx_prefilter *pf, uint32_t matcher_flags,
                         ugx_search_info *out, uint8_t *cls, uint16_t *table, uint32_t cap);
int  ugx_pattern_info_get(const ugx_pattern *p, ugx_pattern_info *info);
void ugx_pattern_destroy(ugx_pattern *p);

/* scanner: owns a stream-ordered scratch arena on `device`; `stream` is a cudaStream_t (NULL = default stream) */
int  ugx_scanner_create(int device, void *stream, ugx_scanner **out);
void ugx_scanner_destroy(ugx_scanner *s);
/* options (tests and A/B timing; defaults 0):
 *   "force_generic"   every scan takes the generic line-scan kernel
 *   "legacy_any"      `-c` takes the tile-synchronous kernel instead of the streaming one
 *   "stream_dfa"      `-c` of every eligible DFA pattern takes the streaming kernel
 *   "count_newlines"  the streaming `-c` kernels also count newlines (totals.newlines)
 *   "match_lines"     counting takes the position-parallel-attempt kernel (match_lines.cu) instead of the line scan
 *   "two_pass_records" records by a count pass + an emit pass instead of the single-pass staging form
 *   "no_pipeline"     host buffers: one copy, then the scan (default: chunked copy overlapped with the scan)
 *   "no_feeder"       pageable host buffers take one plain cudaMemcpyAsync instead of the feeder threads
 *   "no_span"         counting matches / records take the line-at-a-time kernels instead of the span kernels
 *   "no_search"       `-c` keeps count_lines_stream_kernel where the search automaton (count_lines_search_kernel,
 *                     ugx_search_describe) applies
 *   "grid_sms"        k > 0: every launch sizes its grid as if the device had min(k, SMs) SMs, so that each warp takes
 *                     many regions of a small buffer, as it does of a multi-GiB one (tests); 0 restores the device's
 *                     count, k < 0 is UGX_E_INVALID.  Results do not depend on it. */
int  ugx_scanner_set_option(ugx_scanner *s, const char *name, int value);

/*
 * Scans.  `buf` is nbytes of text; it may be a device pointer (scanned in place)
 * or a host pointer (staged to the device inside the call, chunked and
 * overlapped with the scan).  The buffer is one file or one line-aligned shard.
 */
int  ugx_count_lines(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                     ugx_totals *totals);
int  ugx_count_matches(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                       ugx_totals *totals);
/* records are written to the host array `out` (capacity `cap`), in input order */
int  ugx_find_all(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                  uint64_t base_offset, uint64_t base_line,
                  ugx_match *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
/* records stay on the device: *dev_out is owned by the scanner and valid until its next call */
int  ugx_find_all_device(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                         uint64_t base_offset, uint64_t base_line,
                         const ugx_match **dev_out, uint64_t *n_out, ugx_totals *totals);
/* copy `count` records of the last ugx_find_all_device result, starting at record `first`, to the host */
int  ugx_scanner_fetch(ugx_scanner *s, ugx_match *out, uint64_t first, uint64_t count);
/*
 * Line records (`ugrep [-n] [-b]` and `ugrep -v`, src/ugrep.cpp:10567-10586 and the output loops that read lineno(),
 * bol(), eol()): one ugx_line per line that matches, or with flags UGX_LINES_INVERT per line that does not, in input
 * order.  A line is buf[bol, eol); a buffer that ends in '\n' has no empty line after it.  The matching records are the
 * lines the `ugrep -c` loop counts (ugx_count_lines), each with that loop's match.  totals->matches = records,
 * totals->newlines is always counted.  Line records live in their own scanner arena: a ugx_find_lines* call leaves the
 * last ugx_find_all_device result valid, and the reverse.  Any other flags bit: UGX_E_INVALID.
 */
int  ugx_find_lines_device(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                           uint64_t base_offset, uint64_t base_line, uint32_t flags,
                           const ugx_line **dev_out, uint64_t *n_out, ugx_totals *totals);
int  ugx_find_lines(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                    uint64_t base_offset, uint64_t base_line, uint32_t flags,
                    ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
/* copy `count` line records of the last ugx_find_lines* / ugx_find_context* result, starting at record `first`, to
 * the host */
int  ugx_scanner_fetch_lines(ugx_scanner *s, ugx_line *out, uint64_t first, uint64_t count);
/*
 * Context lines (`ugrep -n -A NUM -B NUM -C NUM`, with UGX_LINES_INVERT `ugrep -v -n -C NUM`).  The selected lines are
 * the records ugx_find_lines returns with the same flags.  A line is printed when some selected line s has
 * s - before <= line <= s + after; windows stop at the buffer's first and last line (GNU grep's context rule, which
 * ugrep follows).  One ugx_line per printed line, in input order, none twice; every record is exactly the record
 * ugx_find_lines gives that line in its own polarity (a matching line carries its first match, a line without one has
 * offset = bol, len = 0, cap = 0).  So a line is selected iff (cap != 0) != invert, every other record is a context
 * line (`-` instead of `:`), and a group separator (`--`) goes wherever consecutive records' line numbers are not
 * consecutive.  before = after = 0 gives ugx_find_lines' result.  *n_out = printed lines, totals->matches = selected
 * lines; totals->kernel names the route that selected them.  The records live in the line arena
 * (ugx_scanner_fetch_lines); arguments, errors and paging are those of ugx_find_lines.
 */
int  ugx_find_context_device(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                             uint64_t base_offset, uint64_t base_line, uint32_t flags, uint32_t before, uint32_t after,
                             const ugx_line **dev_out, uint64_t *n_out, ugx_totals *totals);
int  ugx_find_context(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                      uint64_t base_offset, uint64_t base_line, uint32_t flags, uint32_t before, uint32_t after,
                      ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
int  ugx_count_newlines(ugx_scanner *s, const void *buf, uint64_t nbytes, ugx_totals *totals);

/*
 * Boolean line queries (`ugrep -e A --and -e B`, `A --andnot B`, `--not A`, `--bool 'A|B -C'`; the CNF sub-matchers of
 * cnf_matching, src/ugrep.cpp:3298-3366).  A query is K compiled patterns, patterns[0..K) with 1 <= K <= 32, plus a
 * conjunction of clauses.  Each clause is a pair of bit masks:
 *   pos: bit j: the clause holds on a line on which patterns[j] has a match
 *   neg: bit j: the clause holds on a line on which patterns[j] has none
 * M(L), the term mask of a line L: bit j of M(L) is set iff L is one of the matching records that
 * ugx_find_lines(patterns[j]) returns for the same buffer (equivalently, the `ugrep -c` loop of pattern j counts L).
 * A line satisfies clause c iff (M(L) & pos) != 0 || (~M(L) & neg) != 0.  A line satisfies the query iff it satisfies
 * every clause; with nclauses == 0 every line satisfies it.  The selected lines are the lines that satisfy the query;
 * with UGX_LINES_INVERT they are the lines that do not (`ugrep -v`).  Lines are those of ugx_find_lines: a line is
 * buf[bol, eol), a buffer that ends in '\n' has no empty line after it, an empty buffer has no lines.
 *
 *   ugrep                   clauses
 *   -e A --and -e B         {pos=A}, {pos=B}
 *   A --andnot B            {pos=A}, {neg=B}
 *   --bool 'A|B -C'         {pos=A|B}, {neg=C}
 *   --not A                 {neg=A}
 *   -v                      UGX_LINES_INVERT
 * Turning a query string into clauses (src/cnf.cpp) stays with the caller.
 *
 * Records: one ugx_line per selected line, in input order: line 1-based (+ base_line), bol and eol as in ugx_find_lines
 * (+ base_offset), offset = bol, len = 0, cap = M(L) over all K patterns, including patterns no clause names.  Under
 * UGX_LINES_INVERT cap is M(L) too and may be 0.  These are NOT ugx_find_lines records: cap is a term mask, not an
 * accept index.
 *
 * Errors, all checked before any device work.  UGX_E_INVALID: a null scanner, pattern array or pattern; a null buf
 * with nbytes > 0; a null clauses with nclauses > 0; npatterns == 0; a pattern on a different device from the scanner;
 * a clause with pos == neg == 0 (always false); a mask bit at or above npatterns; any flags bit other than
 * UGX_LINES_INVERT.  UGX_E_UNSUPPORTED: more than UGX_BOOL_MAX_PATTERNS patterns or more than UGX_BOOL_MAX_CLAUSES
 * clauses.  UGX_E_OVERFLOW, cap and paging: as in ugx_find_lines (*n_out is set, the records stay fetchable with
 * ugx_scanner_fetch_lines).
 *
 * Totals: matches = selected lines; newlines always counted; UGX_TOT_SPAN_HANDOVER when any term's selection handed
 * over; launches = every kernel of the call; kernel_ms = the whole call on the device (every term's selection and the
 * Boolean stage); kernel = UGX_K_BOOL_LINES.
 *
 * The records live in the line arena; the last ugx_find_all_device result stays valid.  ugx_count_lines_bool leaves
 * the line arena with zero records.
 */
#define UGX_BOOL_MAX_PATTERNS 32
#define UGX_BOOL_MAX_CLAUSES  64
typedef struct ugx_bool_clause {
  uint32_t pos; /* bit j: the clause holds on a line on which patterns[j] has a match */
  uint32_t neg; /* bit j: the clause holds on a line on which patterns[j] has none   */
} ugx_bool_clause;
int  ugx_count_lines_bool(ugx_scanner *s, const ugx_pattern *const *patterns, uint32_t npatterns,
                          const ugx_bool_clause *clauses, uint32_t nclauses,
                          const void *buf, uint64_t nbytes, uint32_t flags, ugx_totals *totals);
int  ugx_find_lines_bool_device(ugx_scanner *s, const ugx_pattern *const *patterns, uint32_t npatterns,
                                const ugx_bool_clause *clauses, uint32_t nclauses,
                                const void *buf, uint64_t nbytes, uint64_t base_offset, uint64_t base_line,
                                uint32_t flags, const ugx_line **dev_out, uint64_t *n_out, ugx_totals *totals);
int  ugx_find_lines_bool(ugx_scanner *s, const ugx_pattern *const *patterns, uint32_t npatterns,
                         const ugx_bool_clause *clauses, uint32_t nclauses,
                         const void *buf, uint64_t nbytes, uint64_t base_offset, uint64_t base_line,
                         uint32_t flags, ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);

/*
 * Many files in one launch: what the reference's per-file job queue feeds its workers (GrepMaster::submit /
 * GrepWorker::execute, src/ugrep.cpp:4295-4432).  The files lie in one buffer (host or device), file i at
 * buf[begins[i], begins[i] + lens[i]) with every begins[i] a multiple of 16 (the bytes between files are never read as
 * text); counts[i] receives what `ugrep -c` (UGX_MODE_LINES) or `ugrep -c -o` (UGX_MODE_MATCHES) prints for file i
 * scanned on its own: each file keeps its own end of buffer.  totals->matches is the sum.
 */
int  ugx_count_batch(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                     const uint64_t *begins, const uint64_t *lens, uint64_t nfiles, int mode,
                     uint64_t *counts, ugx_totals *totals);
/*
 * Records of many files in one launch sequence (`ugrep -rn`, `ugrep -r -o -n -b`, `ugrep -rv` over a source tree).  The
 * file layout is that of ugx_count_batch.  File i's records are exactly what ugx_find_all / ugx_find_lines (same flags)
 * return for that file ALONE with base_offset = base_line = 0: offsets are relative to the file's start and line
 * numbers start at 1 in every file.  The records are grouped by file in file order; first[nfiles + 1] (host) receives
 * the ranges, file i owning records [first[i], first[i + 1]).  They stay in the scanner's match arena
 * (ugx_find_all_batch) or line arena (ugx_find_lines_batch), so ugx_scanner_fetch / ugx_scanner_fetch_lines page
 * through them, and the other arena's last result stays valid.  totals->matches = records, totals->newlines = the
 * files' '\n' bytes, totals->kernel = UGX_K_BATCH.  out == NULL with cap == 0: the records stay on the device, UGX_OK.
 * Otherwise n > cap returns UGX_E_OVERFLOW with *n_out and first[] filled, and the records remain fetchable.
 * nfiles == 0: UGX_OK, first[0] = 0.  A bad file table or any flags bit other than UGX_LINES_INVERT: UGX_E_INVALID.
 */
int  ugx_find_all_batch(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                        const uint64_t *begins, const uint64_t *lens, uint64_t nfiles, uint64_t *first,
                        ugx_match *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
int  ugx_find_lines_batch(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                          const uint64_t *begins, const uint64_t *lens, uint64_t nfiles, uint32_t flags,
                          uint64_t *first, ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
/* context lines of many files (`ugrep -rn -C NUM PATTERN tree/`): file i's records are exactly what ugx_find_context
 * returns for that file alone with base_offset = base_line = 0, and context never crosses a file boundary; first[]
 * gives every file's range of printed lines.  Otherwise as ugx_find_lines_batch. */
int  ugx_find_context_batch(ugx_scanner *s, const ugx_pattern *p, const void *buf, uint64_t nbytes,
                            const uint64_t *begins, const uint64_t *lens, uint64_t nfiles, uint32_t flags,
                            uint32_t before, uint32_t after, uint64_t *first,
                            ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);
/*
 * Boolean line queries over many files (`ugrep -rn -e A --and -e B tree/`, `ugrep -rc A --andnot B`, `ugrep -rl --bool
 * 'A|B -C'`, `-v` with UGX_LINES_INVERT).  The query, its clauses, flags and errors are those of ugx_find_lines_bool;
 * the file layout is that of ugx_count_batch (host or device buffer, every begins[i] a multiple of 16; the bytes
 * between files are never text).  File i's records are byte for byte what ugx_find_lines_bool returns for that file
 * ALONE with the same patterns, clauses and flags and base_offset = base_line = 0: line numbers start at 1 in every
 * file, offsets count from the file's start, offset = bol, len = 0, cap = M(L) over all K patterns.  counts[i] is what
 * ugx_count_lines_bool gives for file i alone (`ugrep -rc --and ...`; `-l` is counts[i] != 0, `-L` counts[i] == 0).  An
 * empty file has no lines and selects nothing, UGX_LINES_INVERT included.
 *
 * Records are grouped by file in file order; first[nfiles + 1] (host) receives the ranges, file i owning
 * [first[i], first[i + 1]).  They live in the line arena (ugx_scanner_fetch_lines pages through them) and the last
 * ugx_find_all_device result stays valid.  out == NULL with cap == 0: the records stay on the device, UGX_OK.
 * Otherwise n > cap returns UGX_E_OVERFLOW with *n_out and first[] filled, and the records remain fetchable.
 * ugx_count_lines_bool_batch leaves the line arena with zero records.
 *
 * Errors, all checked before any device work: those of ugx_find_lines_bool, a file that is not a 16-byte aligned range
 * of the buffer (UGX_E_INVALID), and a null begins, lens, counts or first with nfiles > 0 (UGX_E_INVALID).
 * nfiles == 0: UGX_OK with first[0] = 0.  A batch of only empty files: zeros, no launch.
 *
 * Totals: matches = selected lines over all files; newlines = the files' '\n' bytes (padding is not counted);
 * UGX_TOT_NEWLINES; launches = every kernel of the call; kernel_ms = the whole call on the device; kernel =
 * UGX_K_BOOL_LINES.
 */
int  ugx_count_lines_bool_batch(ugx_scanner *s, const ugx_pattern *const *patterns, uint32_t npatterns,
                                const ugx_bool_clause *clauses, uint32_t nclauses,
                                const void *buf, uint64_t nbytes, const uint64_t *begins, const uint64_t *lens,
                                uint64_t nfiles, uint32_t flags, uint64_t *counts, ugx_totals *totals);
int  ugx_find_lines_bool_batch(ugx_scanner *s, const ugx_pattern *const *patterns, uint32_t npatterns,
                               const ugx_bool_clause *clauses, uint32_t nclauses,
                               const void *buf, uint64_t nbytes, const uint64_t *begins, const uint64_t *lens,
                               uint64_t nfiles, uint32_t flags, uint64_t *first,
                               ugx_line *out, uint64_t cap, uint64_t *n_out, ugx_totals *totals);

/* what ugrep asks about a file before it prints from it (Grep::init_is_binary, src/ugrep.cpp:3998-4017):
 * is_utf8 = reflex::isutf8 (lib/simd.cpp:169-421: valid UTF-8 structure, no NUL), has_nul = memchr(buf, 0, n) != NULL;
 * is_binary() is !is_utf8 by default and has_nul with -U (src/ugrep.cpp:699-711) */
typedef struct ugx_text_info {
  uint32_t is_utf8;
  uint32_t has_nul;
  float    kernel_ms;
  uint32_t launches;
} ugx_text_info;
int  ugx_check_text(ugx_scanner *s, const void *buf, uint64_t nbytes, ugx_text_info *out);

/*
 * One process, several GPUs (SURVEY.md 8e): the buffer is cut into one line-aligned shard per device (forward from
 * n*r/N to the next newline), every device scans its shard, and the per-shard {matches, newlines} give the totals and
 * the record / line-number bases.  Replaces the reference's per-file worker pool (GrepMaster / GrepWorker,
 * src/ugrep.cpp:4118-4432) for one large input.  `devices` may name a device more than once.
 */
typedef struct ugx_sharded ugx_sharded;
typedef struct ugx_shard {
  int32_t  device;
  uint32_t reserved;
  uint64_t begin, end;       /* the shard is buf[begin, end) */
  uint64_t matches, newlines;
  uint64_t line_base;        /* newlines before the shard */
  uint64_t record_base;      /* matches before the shard */
  float    kernel_ms;
  uint32_t reserved2;
} ugx_shard;
int  ugx_sharded_create(const uint32_t *opc, uint32_t nop, const ugx_prefilter *pf, uint32_t matcher_flags,
                        const int *devices, int ndev, ugx_sharded **out);
void ugx_sharded_destroy(ugx_sharded *s);
/* "pin": page-lock the caller's buffer during a scan (pays when the same buffer is scanned repeatedly);
 * every other name is passed to each device's scanner (ugx_scanner_set_option) */
int  ugx_sharded_set_option(ugx_sharded *s, const char *name, int value);
/* host_buf: host memory.  mode UGX_MODE_RECORDS writes the records of all shards to out[cap] in input order, offsets
 * and line numbers global; shards[ndev] (optional) receives what every device did */
int  ugx_sharded_scan(ugx_sharded *s, const void *host_buf, uint64_t nbytes, int mode, ugx_match *out, uint64_t cap,
                      uint64_t *n_out, ugx_totals *totals, ugx_shard *shards);
/* line records of all shards (ugx_find_lines) to out[cap] in input order, line numbers and offsets global;
 * shards[r].record_base = line records before shard r */
int  ugx_sharded_find_lines(ugx_sharded *s, const void *host_buf, uint64_t nbytes, uint32_t flags, ugx_line *out,
                            uint64_t cap, uint64_t *n_out, ugx_totals *totals, ugx_shard *shards);
const char *ugx_sharded_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* UGREP_B200_H */
