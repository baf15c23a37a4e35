// scan_kernels.hpp — launch interface of the scan kernels (host side, CUDA runtime types only)
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/ugrep_b200.h"

namespace ugx {

struct DevPattern;

constexpr int SCAN_THREADS = 256;                      // threads per CTA (512 for big staged tables: scan_threads())
// Dynamic shared memory every kernel opts in to (the 227 KiB per-CTA limit minus room for static shared memory).  The
// attribute is set to this one value for every pattern: it is process-global per kernel, and scanners on different
// host threads may launch the same kernel with different tables.
constexpr int UGX_MAX_DYN_SMEM = 227 * 1024 - 4096;
constexpr int SCAN_STRIP = 64;                         // bytes per thread per tile
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_STRIP;   // bytes per CTA iteration (16 KiB)
constexpr uint32_t SCAN_LINE_CAP = 1024;                // line starts per tile the dense line list holds
constexpr uint32_t SCAN_MAX_SMEM_TABLE = 198 * 1024;   // largest transition table staged in shared memory
constexpr uint32_t ANY_TILE = 32768;                   // bytes per CTA iteration of count_lines_any_kernel

// The slots of a scanner's device array `totals` (and of its pinned host copy).  The kernels that take `totals` write
// the result slots at [0] and [1]; the span kernels and the UTF-8 check use the others at these fixed offsets.
enum TotalsSlot : int {
  SLOT_MATCHES = 0,     // result: matches, matching lines, records or selected lines
  SLOT_NEWLINES = 1,    // result: newlines
  SLOT_HANDOVER = 2,    // span count pass: 1 = the spans' result is not valid; single-pass records: the staging cursor
  SLOT_TAIL_MATCHES = 3, // span_final_kernel: matches before the last line
  SLOT_TAIL_NEWLINES = 4, // span_final_kernel: newlines before the last line
  SLOT_LAST_LINE = 5,   // launch_last_line: start of the buffer's last line
  SLOT_SPAN_FLAGS = 6,  // SpanArgs::flags
  SLOT_UTF8 = 7,        // launch_utf8_check's flags
  SLOT_BATCH_LINES = 8, // ugx_*_lines_bool_batch: the prefix over the file line table: lines of the batch
  SLOT_BATCH_NEWLINES = 9, //   ... and its newlines
  SLOT_COUNT = 10
};

struct ScanArgs {
  const uint8_t* buf;
  uint64_t n;
  uint64_t ntiles;
  uint64_t* tile_matches;   // [ntiles]
  uint64_t* tile_newlines;  // [ntiles]
  uint32_t* strip_counts;   // [ceil(n / SCAN_STRIP)] or nullptr
  ugx_match* out;
  uint64_t out_cap;
  uint64_t base_offset;
  uint64_t base_line;
};

// CTA size / tile size of the line-scan and records kernels for this pattern (ntiles = ceil(n / scan_tile_bytes))
int scan_threads(const DevPattern& P);
uint32_t scan_tile_bytes(const DevPattern& P);
cudaError_t launch_scan_lines(const DevPattern& P, const ScanArgs& a, int mode, bool emit, int sm_count, cudaStream_t st);
// line records (`ugrep -c` loop per line, ugx_find_lines): the count pass writes a.strip_counts and the tile sums, the
// emit pass (after launch_tile_prefix) writes out[]; lflags = UGX_LINES_INVERT | SCAN_LINES_NEVER
constexpr uint32_t SCAN_LINES_NEVER = 2u;
cudaError_t launch_scan_line_records(const DevPattern& P, const ScanArgs& a, ugx_line* out, uint32_t lflags, bool emit,
                                     int sm_count, cudaStream_t st);
// `ugrep -c` for patterns without look-back: one position-parallel kernel, totals[0] = matching lines, [1] = newlines
bool count_lines_any_eligible(const DevPattern& P);
cudaError_t launch_count_lines_any(const DevPattern& P, const uint8_t* buf, uint64_t n, unsigned long long* totals,
                                   int sm_count, cudaStream_t st);
// ---- streaming `ugrep -c` (stream_count.cu) ----
#ifndef UGX_STREAM_THREADS
#define UGX_STREAM_THREADS 256
#endif
#ifndef UGX_SC_REGION
#define UGX_SC_REGION 16384
#endif
constexpr int STREAM_THREADS = UGX_STREAM_THREADS;     // threads per CTA
constexpr uint32_t SC_REGION = UGX_SC_REGION;                  // bytes per region (unit of the ticket counter and of the summaries)
constexpr uint32_t STREAM_MAX_GRID = 4096;             // capacity of the per-CTA partials

struct StreamArgs {
  uint8_t* region_sum;            // [regions(buffer) + 16] one summary byte per region of the buffer
  uint64_t region_begin;          // this launch scans the regions [region_begin, region_end) of the buffer;
  uint64_t region_end;            //   the kernel's n = the bytes of the buffer that are valid (copied) so far
  unsigned long long* partials;   // [2 * STREAM_MAX_GRID] per-CTA {lines, newlines}
  unsigned long long* ticket;     // region ticket counter (zero between launches)
  unsigned int* done;             // finished-CTA counter (zero between launches)
  unsigned long long* totals;     // [2] {matching lines, newlines}
  uint32_t finalize;              // last launch of a buffer: chain the regions' head lines
  uint32_t accumulate;            // add to totals instead of overwriting them
  uint32_t stage_table;           // set by the launcher
  uint32_t use_h4;                // set by the launcher: stage the hashed-predictor term table
  uint32_t use_via;               // set by the launcher: stage the k-gram viability tables (viability.cuh)
  uint32_t no_cover;              // evaluate the candidate predicate even when DevPattern::covers allows skipping it (A/B)
};

bool count_lines_stream_eligible(const DevPattern& P);
uint64_t stream_regions(uint64_t n);
int stream_grid(uint64_t n, int sm_count, int per_sm, int threads);
cudaError_t launch_count_lines_stream(const DevPattern& P, const uint8_t* buf, uint64_t n, StreamArgs a, bool want_nl,
                                      int sm_count, cudaStream_t st);
// the search-automaton form (stream_search.cu) for DevPattern::search_ok: the same regions, summaries and totals
cudaError_t launch_count_lines_search(const DevPattern& P, const uint8_t* buf, uint64_t n, const StreamArgs& a, bool want_nl,
                                      int sm_count, cudaStream_t st);
// the literal specialisation (stream_literal.cu), taken by launch_count_lines_stream when eligible
bool count_lines_literal_eligible(const DevPattern& P);
cudaError_t launch_count_lines_literal(const DevPattern& P, const uint8_t* buf, uint64_t n, const StreamArgs& a, bool want_nl,
                                       int sm_count, cudaStream_t st);

// find loop with position-parallel attempts (match_lines.cu): counting for patterns without META / W / start-loop skip
bool match_lines_eligible(const DevPattern& P);
uint32_t match_lines_tile_bytes(const DevPattern& P);
cudaError_t launch_match_lines(const DevPattern& P, const ScanArgs& a, int mode, int sm_count, cudaStream_t st);

// single-pass records (records_kernel.cu): staging pass + reorder into input order
cudaError_t launch_scan_records(const DevPattern& P, const ScanArgs& a, uint64_t* tile_base, ugx_match* stage_out,
                                uint64_t stage_cap, unsigned long long* cursor, int sm_count, cudaStream_t st);
cudaError_t launch_reorder_records(const ugx_match* stage, ugx_match* out, const uint64_t* pm, const uint64_t* pn,
                                   const uint64_t* tile_base, uint64_t ntiles, const unsigned long long* totals,
                                   uint64_t base_line, int sm_count, cudaStream_t st);

// ---- span scan (span_scan.cu): `ugrep -c -o` / `ugrep -o -n -b` with every DFA attempt taken out of the find loop ----
constexpr uint64_t SPAN_TAIL_MAX = 65536;   // a last line up to this long is left to the final kernel's line-at-a-time form

struct SpanArgs {
  uint64_t* reg_matches;   // [regions] count pass: matches that start in the region; after the final kernel: exclusive prefix
  uint64_t* reg_newlines;  // [regions] likewise, newlines
  uint64_t* reg_emain;     // [regions] farthest end of a success that starts in spans 0..30 of the region
  uint64_t* reg_elast;     // [regions] ... in its last span (the next region's window)
  uint64_t* reg_v;         // [regions] validation point of the region's chain start (~0 = none needed)
  uint16_t* sel_bits;      // [ceil(n / 16) + 32] or nullptr: the selected match starts of every 16-byte chunk (records)
  ugx_match* out;          // emit pass: records in input order
  uint64_t out_cap;
  uint64_t base_offset, base_line;
  const uint64_t* tail;    // device: [0] = start of the last line (the spans scan [0, tail[0]))
  unsigned int* flags;     // device: bit 0 an attempt failed at the end of the buffer, bit 1 a match too long for the span tables
  uint32_t stage_table;    // set by the launcher
  uint32_t use_via;        // set by the launcher: the viability tables are staged in shared memory
  uint32_t no_cover;       // decide membership in the attempt set even when DevPattern::covers makes it moot (A/B)
};

bool span_scan_eligible(const DevPattern& P);
cudaError_t launch_last_line(const uint8_t* buf, uint64_t n, uint64_t* tail, cudaStream_t st);
cudaError_t launch_span_scan(const DevPattern& P, const uint8_t* buf, uint64_t n, SpanArgs a, bool emit, int sm_count,
                             cudaStream_t st);
cudaError_t launch_span_final(const DevPattern& P, const uint8_t* buf, uint64_t n, const SpanArgs& a, bool emit,
                              unsigned long long* totals, cudaStream_t st);

// ---- line records from the span kernels' selected match starts (span_scan.cu, ugx_find_lines) ----
// A line belongs to the region that holds its '\n'; a line that began in an earlier region gets its start and its first
// match from carries over the regions before (span_lines_final_kernel).  The region values, [regions] each:
struct SpanLinesArgs {
  uint64_t* reg_nl;        // count pass: newlines in the region;            after the final kernel: newlines before it
  uint64_t* reg_m;         //   owned lines after the first with a selected start;           records before the region
  uint64_t* reg_bol;       //   last newline + 1 (0 = none);                 start of the line that runs into the region
  uint64_t* reg_fb;        //   first selected start before the first newline (~0 = none)   (unused afterwards)
  uint64_t* reg_fa;        //   first selected start after the last newline;  first selected start since reg_bol, before the region
  uint64_t* tail;          // [8] the line after the last region's last newline: {line, bol, eol, offset, len | cap << 32
                           //     (~0 = longest_at still to run), record index, present}
  const uint16_t* sel_bits;// span_scan_kernel's selected match starts
  const uint64_t* limit;   // device: where the spans stop (SpanArgs::tail)
  ugx_line* out;           // emit pass: records in input order
  uint64_t out_cap;
  uint64_t base_offset, base_line;
  uint32_t invert;         // UGX_LINES_INVERT: the records are the lines without a selected start
  uint32_t stage_table;    // set by the launcher
};
cudaError_t launch_span_lines(const DevPattern& P, const uint8_t* buf, uint64_t n, SpanLinesArgs a, bool emit, int sm_count,
                              cudaStream_t st);
// one CTA: record / line bases and carries of the regions, the last line; totals[0] = records, [1] = newlines
cudaError_t launch_span_lines_final(const DevPattern& P, const uint8_t* buf, uint64_t n, const SpanLinesArgs& a,
                                    unsigned long long* totals, cudaStream_t st);

// reflex::nlcount (newline_count.cu)
cudaError_t launch_count_newlines(const uint8_t* buf, uint64_t n, unsigned long long* total, int sm_count, cudaStream_t st);

// ---- many files in one launch (batch_kernel.cu) ----
struct BatchArgs {
  const uint64_t* begins;        // [nfiles] device: offset of every file in the batch buffer (multiples of 16)
  const uint64_t* lens;          // [nfiles] device: its length
  const uint32_t* tile_file;     // [ntiles] device: the file a tile belongs to
  const uint32_t* tile_index;    // [ntiles] device: its index within that file
  uint64_t ntiles;
  unsigned long long* counts;    // [nfiles] device, zeroed by the caller
  uint32_t stage_table;          // set by the launcher
};
cudaError_t launch_scan_batch(const DevPattern& P, const uint8_t* buf, BatchArgs a, int mode, int sm_count, cudaStream_t st);
// records of a batch (batch_records.cu, ugx_find_all_batch / ugx_find_lines_batch): a count pass, launch_tile_prefix over
// the batch tiles, an emit pass.  a.counts receives the records of every file (count pass).
struct BatchRecordArgs {
  uint64_t* tile_matches;   // [ntiles] count pass: records of the tile; after launch_tile_prefix: records before it
  uint64_t* tile_newlines;  // [ntiles] likewise, newlines
  uint32_t* strip_counts;   // [ntiles * SCAN_THREADS] records owned by every 64-byte strip of every tile
  ugx_match* out;           // emit pass: match records (lines == false)
  ugx_line* lout;           // emit pass: line records (lines == true)
  uint64_t out_cap;         // emit pass: the total number of records
  uint32_t lflags;          // UGX_LINES_INVERT | SCAN_LINES_NEVER
};
cudaError_t launch_scan_batch_records(const DevPattern& P, const uint8_t* buf, BatchArgs a, const BatchRecordArgs& r,
                                      bool lines, bool emit, int sm_count, cudaStream_t st);

// ---- context lines (context_lines.cu, ugx_find_context / ugx_find_context_batch: `-A` / `-B` / `-C`) ----
// The selected line records of ugx_find_lines[_batch] in, one record per printed line out: a count pass (printed lines
// every selected record owns), launch_tile_prefix over the count pass's block sums, an emit pass, and under
// UGX_LINES_INVERT a pass that gives every context line its first match.
constexpr uint32_t CTX_PER_BLOCK = 4096; // selected records per block of the count pass
struct ContextArgs {
  const ugx_line* sel;      // [nsel] selected records, grouped by file, in input order
  uint64_t nsel;
  const uint8_t* buf;       // the buffer (one buffer) or the batch buffer
  uint64_t n;               // one buffer: its size
  uint64_t nl_total;        // newlines of the buffer / of all files of the batch
  uint64_t base_offset, base_line; // one buffer; 0 for a batch
  // a batch (fsel == nullptr: one buffer): the file table of BatchArgs, every file's selected records
  // [fsel[f], fsel[f + 1]) and first batch tile ftile[f], and the exclusive newline prefix of the batch tiles
  uint64_t nfiles;
  const uint64_t* begins;
  const uint64_t* lens;
  const uint64_t* fsel;     // [nfiles + 1]
  const uint64_t* ftile;    // [nfiles + 1]
  const uint64_t* tile_nl;  // [ntiles]
  uint64_t ntiles;
  uint32_t before, after;
  uint32_t invert;          // UGX_LINES_INVERT: context lines are matching lines and carry their first match
  uint64_t* pos;            // [nsel] count pass: printed lines before record i within its block
  uint64_t* blk;            // [2 * blocks] count pass: printed lines of every block (then zeros); after the prefix: before it
  ugx_line* out;            // emit pass: [nout] records in input order
  uint64_t nout;
  uint64_t* fout;           // emit pass, a batch: [nfiles + 1] every file's first printed line, or nullptr
};
uint64_t context_blocks(uint64_t nsel);
cudaError_t launch_context_count(const ContextArgs& a, cudaStream_t st);
cudaError_t launch_context_emit(const ContextArgs& a, int sm_count, cudaStream_t st);
// under UGX_LINES_INVERT, after the emit pass: the first match of every context line
cudaError_t launch_context_match(const DevPattern& P, const ContextArgs& a, int sm_count, cudaStream_t st);

// ---- Boolean line queries (bool_lines.cu, ugx_*_lines_bool and ugx_*_lines_bool_batch: `--and`, `--andnot`, `--bool`) ----
// One buffer: after every term's selection launch_bool_mark ORs its bit into the term mask of each record's line; then
// a count pass (selected lines per line block, newlines per byte region), launch_tile_prefix over both, and for records
// an index pass (every line's end) and the emit pass.
// Many files: the batch's lines are numbered across the files, file f owning [lb[f], lb[f + 1]).  After the first term's
// count pass (launch_scan_batch_records) and its tile prefix, launch_bool_batch_lines writes every file's lines and
// newlines, and launch_tile_prefix over those columns ([nfiles + 1] each, zeroed by the caller) gives lb[] with
// lb[nfiles] = the lines.  After every term's selection launch_bool_batch_mark ORs its bit into the mask of each
// record's line (the batch tiles' record prefix locates the records of a file).  Then the batch count pass,
// launch_tile_prefix over its block values, and for records the batch index pass and the emit pass.
// The emit pass serves both: one buffer is one file, lines [0, nlines), with the call's bases.
constexpr uint32_t BOOL_LINES_PER_BLOCK = 8192; // lines per block of the count and emit passes
constexpr uint32_t BOOL_REGION = 65536;         // bytes per block of the newline count and the index pass (one buffer)
struct BoolQuery {                              // the clauses, passed by value in the kernel parameters
  uint32_t pos[UGX_BOOL_MAX_CLAUSES];
  uint32_t neg[UGX_BOOL_MAX_CLAUSES];
  uint32_t nclauses;
  uint32_t invert;                              // UGX_LINES_INVERT: the lines that do not satisfy the query
};
struct BoolArgs {
  const uint8_t* buf;            // the buffer, or the batch buffer
  uint64_t n;                    // one buffer: its size
  BatchArgs files;               // a batch: its file and tile tables
  uint64_t nfiles;               // 1 for one buffer
  uint64_t* lb;                  // [nfiles + 1] every file's first line; lb[nfiles] = nlines.  One buffer: {0, nlines},
                                 //   written by the count pass with want_index
  uint64_t nlines;               // one buffer: newlines + (last byte != '\n')
  const uint32_t* mask;          // [nlines] term mask of every line
  unsigned long long* fsel;      // a batch, count pass: selected lines of every file (zeroed by the caller)
  uint64_t* blk;                 // [2 * nblocks] count pass: selected lines of line block b | newlines of region b (a
                                 //   batch: 0); after the prefix: the same before b
  uint64_t nblocks;              // grid of the count pass: line blocks, or for one buffer with want_index the larger of
                                 //   them and the regions
  uint32_t want_index;           // one buffer: the count pass also counts newlines per region (records follow)
  const uint64_t* tile_nl;       // a batch, index pass: the exclusive newline prefix of the batch tiles
  uint64_t* eol;                 // [nlines] index pass: offset within its buffer or file of every line's '\n' (or its end)
  ugx_line* out;                 // emit pass: [selected lines] grouped by file, in input order
  uint64_t base_offset, base_line; // one buffer; 0 for a batch
};
uint64_t bool_line_blocks(uint64_t nlines);
uint64_t bool_regions(uint64_t n);
cudaError_t launch_bool_mark(const ugx_line* rec, uint64_t nrec, uint32_t* mask, uint32_t bit, int sm_count,
                             cudaStream_t st);
cudaError_t launch_bool_count(const BoolArgs& a, const BoolQuery& q, cudaStream_t st);
cudaError_t launch_bool_index(const BoolArgs& a, cudaStream_t st);
cudaError_t launch_bool_batch_lines(const uint8_t* buf, const BatchArgs& b, const uint64_t* tile_nl,
                                    const unsigned long long* nl_total, uint64_t* flines, uint64_t* fnl, cudaStream_t st);
cudaError_t launch_bool_batch_mark(const ugx_line* rec, uint64_t nrec, const uint64_t* tile_rec, const BatchArgs& b,
                                   const uint64_t* lb, uint32_t* mask, uint32_t bit, int sm_count, cudaStream_t st);
cudaError_t launch_bool_batch_count(const BoolArgs& a, const BoolQuery& q, cudaStream_t st);
cudaError_t launch_bool_batch_index(const BoolArgs& a, cudaStream_t st);
cudaError_t launch_bool_batch_emit(const BoolArgs& a, const BoolQuery& q, cudaStream_t st);

// reflex::isutf8 / NUL test (utf8_check.cu): flags bit 0 = not UTF-8 by the reference's rule, bit 1 = has a NUL
cudaError_t launch_utf8_check(const uint8_t* buf, uint64_t n, unsigned int* flags, int sm_count, cudaStream_t st);

cudaError_t launch_tile_prefix(uint64_t* tile_matches, uint64_t* tile_newlines, uint64_t ntiles,
                               unsigned long long* totals, cudaStream_t st);

} // namespace ugx
