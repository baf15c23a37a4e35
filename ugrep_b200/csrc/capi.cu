// capi.cu — the C ABI declared in include/ugrep_b200.h: pattern upload, scanner scratch,
// and the scan entry points.  Host C++ only calls CUDA through this file and scan_kernels.cu.
// There is no CPU scan path: without a usable CUDA device every entry point fails.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/ugrep_b200.h"
#include "device_pattern.cuh"
#include "pattern_host.hpp"
#include "scan_kernels.hpp"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg)
{
  g_err = msg;
  return code;
}

int cuda_fail(cudaError_t e, const char* what)
{
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return UGX_E_CUDA;
}

#define CU(call)                         \
  do                                     \
  {                                      \
    cudaError_t e_ = (call);             \
    if (e_ != cudaSuccess)               \
      return cuda_fail(e_, #call);       \
  } while (0)

// a status code other than UGX_OK ends the calling function with it
#define TRY(call)                        \
  do                                     \
  {                                      \
    const int rc_ = (call);              \
    if (rc_ != UGX_OK)                   \
      return rc_;                        \
  } while (0)

const int k_word_ranges[] = {
#include "word_ranges.inc"
};

// a device copy of host[bytes] in `dev`, owned by the pattern's `allocs`
template <typename T>
int upload(std::vector<void*>& allocs, const T*& dev, const void* host, size_t bytes)
{
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
  if (e != cudaSuccess)
    return cuda_fail(e, "cudaMalloc");
  if (bytes)
  {
    e = cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
    {
      cudaFree(p);
      return cuda_fail(e, "cudaMemcpy");
    }
  }
  allocs.push_back(p);
  dev = static_cast<const T*>(p);
  return UGX_OK;
}

void set256(uint32_t* set, const uint8_t* bytes32)
{
  for (int i = 0; i < 8; ++i)
    set[i] = static_cast<uint32_t>(bytes32[4 * i]) | (static_cast<uint32_t>(bytes32[4 * i + 1]) << 8) |
             (static_cast<uint32_t>(bytes32[4 * i + 2]) << 16) | (static_cast<uint32_t>(bytes32[4 * i + 3]) << 24);
}

// device scratch of a scanner: grown on demand (by an eighth and 64 elements over the need), freed with the scanner
template <typename T>
struct DevBuf {
  T* p = nullptr;
  uint64_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { cudaFree(p); }
  int ensure(uint64_t need)
  {
    if (need <= cap)
      return UGX_OK;
    if (p != nullptr)
      cudaFree(p);
    p = nullptr;
    cap = 0;
    uint64_t want = need + need / 8 + 64;
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, want * sizeof(T));
    if (e != cudaSuccess)
    {
      g_err = std::string("cudaMalloc scratch: ") + cudaGetErrorString(e);
      return e == cudaErrorMemoryAllocation ? UGX_E_NOMEM : UGX_E_CUDA;
    }
    p = static_cast<T*>(q);
    cap = want;
    return UGX_OK;
  }
  void swap(DevBuf& o)
  {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }
};

// no C++ exception may cross the C ABI: an allocation failure becomes UGX_E_NOMEM "out of host memory", and any other
// exception becomes `code` with the exception's text after `who` (who == nullptr: "out of host memory")
template <typename F>
int guarded(int code, const char* who, F&& body)
{
  try
  {
    return body();
  }
  catch (const std::bad_alloc&)
  {
    return fail(UGX_E_NOMEM, "out of host memory");
  }
  catch (const std::exception& ex)
  {
    return fail(code, who ? std::string(who) + ": " + ex.what() : std::string("out of host memory"));
  }
}

} // namespace

struct ugx_pattern {
  ugx::HostDfa dfa;
  ugx_prefilter pf;
  uint32_t flags = 0;
  int adv = 0;
  bool never = false; // the prefilter tables admit no candidate at all (config 3, SURVEY.md Q1): every scan finds nothing
  int device = 0;
  uint32_t nop = 0;
  ugx::DevPattern dev;
  std::vector<void*> allocs;
  ~ugx_pattern()
  {
    for (void* p : allocs)
      cudaFree(p);
  }
};

struct ugx_scanner {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 0;    // the SM count every launch sizes its grid by: device_sms, or fewer under the "grid_sms" option
  int device_sms = 0;  // the device's own SM count
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // scratch
  DevBuf<uint64_t> tile_matches;
  DevBuf<uint64_t> tile_newlines;
  DevBuf<uint32_t> strip_counts;
  unsigned long long* totals = nullptr; // device [ugx::SLOT_COUNT]
  unsigned long long* h_totals = nullptr; // pinned [ugx::SLOT_COUNT]
  DevBuf<ugx_match> records;
  uint64_t records_n = 0;
  DevBuf<uint8_t> stage; // device copy of a host buffer
  bool force_generic = false; // tests: always take the generic line-scan kernel
  bool legacy_any = false;    // tests / A-B timing: the tile-synchronous count_lines_any kernel instead of the streaming one
  bool count_newlines = false; // the streaming count also counts newlines
  bool match_lines = false;      // counting takes match_lines_kernel (position-parallel attempts) instead of scan_lines_kernel
  bool two_pass_records = false; // records by count pass + emit pass (A/B against the single-pass staging form)
  DevBuf<uint64_t> tile_base;    // staging base of every tile's records
  DevBuf<ugx_match> rec_stage;   // records in tile completion order
  bool no_pipeline = false;    // host buffers: one copy, then the scan (A/B timing of the overlapped path)
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copy = nullptr;
  bool stream_dfa = false;     // DFA patterns take the streaming count too (default: the tile-synchronous kernel)
  // streaming count scratch
  DevBuf<uint8_t> region_sum;
  unsigned long long* partials = nullptr; // [2 * STREAM_MAX_GRID]
  unsigned long long* ticket = nullptr;   // {ticket (u64), done (u32)}
  // span scan scratch
  DevBuf<uint64_t> span_regions; // [5 * regions]
  // pageable host buffers: feeder threads copy chunks into pinned slots, each slot goes to the device on its thread's stream
  std::vector<uint8_t*> feed_slots;      // [2 * feed_threads] pinned, FEED_CHUNK bytes each
  std::vector<cudaStream_t> feed_streams; // [feed_threads]
  std::vector<cudaEvent_t> feed_events;   // [2 * feed_threads] slot free again
  bool no_feeder = false;         // pageable buffers take one plain cudaMemcpyAsync (A/B timing)
  DevBuf<uint16_t> span_sel;      // records: selected match starts per 16-byte chunk
  DevBuf<uint64_t> batch;         // ugx_count_batch: file table, counters, tile table
  bool no_span = false;           // counting matches / records take the line-at-a-time kernels (A/B timing, tests)
  bool no_cover = false;          // the streaming count evaluates the candidate predicate even where it is proven implied
  bool no_search = false;         // `-c` keeps count_lines_stream_kernel where the search automaton applies (A/B, tests)
  // line records (ugx_find_lines*): an arena of their own, so that they and the match records stay valid side by side
  DevBuf<ugx_line> lines;
  uint64_t lines_n = 0;
  DevBuf<uint64_t> lines_regions; // [5 * regions + 8] span route: SpanLinesArgs region values and the last line
  // context lines (ugx_find_context*): the selected records, swapped out of the line arena, and the count pass scratch
  DevBuf<ugx_line> ctx_sel;
  DevBuf<uint64_t> ctx_pos;      // [nsel] | [2 * blocks] | a batch: fsel, ftile, fout [nfiles + 1] each
  // Boolean line queries (ugx_*_lines_bool): the term mask of every line, and the count pass's block values + line ends
  DevBuf<uint32_t> bool_mask;
  DevBuf<uint64_t> bool_pos;     // [2 * blocks] | [lines]
  DevBuf<uint64_t> bool_files;   // a batch: every file's lines | newlines [nfiles + 1] each, selected lines [nfiles]
};

extern "C" {

const char* ugx_last_error(void) { return g_err.c_str(); }
int ugx_abi_version(void) { return UGX_ABI_VERSION; }

static int pattern_create_impl(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, int device,
                               ugx_pattern** out);

// the search automaton of `-c` (stream_search.cu), built when the attempt semantics allow it and then kept only on the
// streaming `-c` DFA route where DevPattern::covers makes "a line counts iff some position in it starts a match" exact
static void plan_search(const ugx::HostDfa& dfa, const ugx_prefilter& pf, uint32_t matcher_flags, int adv, bool covers,
                        ugx::SearchDfa& sd)
{
  ugx::build_search_dfa(dfa, sd);
  if (sd.refusal == UGX_SEARCH_OK &&
      (pf.lbk != 0 || (matcher_flags & UGX_OPT_W) != 0 || adv == UGX_ADV_NONE || pf.one != 0 || !covers))
    sd.refusal = UGX_SEARCH_ROUTE;
}

int ugx_pattern_create(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, int device,
                       ugx_pattern** out)
{
  return guarded(UGX_E_INVALID, "ugx_pattern_create", [&] { return pattern_create_impl(opc, nop, pf, matcher_flags, device, out); });
}

static int pattern_create_impl(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, int device,
                               ugx_pattern** out)
{
  if (opc == nullptr || nop == 0 || pf == nullptr || out == nullptr)
    return fail(UGX_E_INVALID, "ugx_pattern_create: null argument");
  std::unique_ptr<ugx_pattern> holder(new (std::nothrow) ugx_pattern()); // freed on every early return and on a throw
  ugx_pattern* p = holder.get();
  if (p == nullptr)
    return fail(UGX_E_NOMEM, "out of host memory");
  std::string err;
  int rc = ugx::flatten_dfa(opc, nop, p->dfa, err);
  if (rc == UGX_OK)
    rc = ugx::check_scope(p->dfa, *pf, matcher_flags, err);
  if (rc != UGX_OK)
  {
    return fail(rc, err);
  }
  p->pf = *pf;
  p->flags = matcher_flags;
  p->adv = ugx::select_advance(*pf, matcher_flags);
  p->never = ugx::prefilter_never_fires(*pf, p->adv);
  p->device = device;
  p->nop = nop;
  cudaError_t ce = cudaSetDevice(device);
  if (ce != cudaSuccess)
  {
    return cuda_fail(ce, "cudaSetDevice (the scan path needs a CUDA device; there is no CPU fallback)");
  }
  ugx::DevPattern& d = p->dev;
  memset(&d, 0, sizeof(d));
  d.adv = p->adv;
  d.len = pf->len;
  d.min = pf->min;
  d.pin = pf->pin;
  d.lcp = pf->lcp;
  d.lcs = pf->lcs;
  d.one = pf->one;
  d.bol = pf->bol;
  d.lbk = pf->lbk;
  d.lbm = pf->lbm;
  d.flags = matcher_flags;
  d.nstates = p->dfa.nstates;
  d.ncls = p->dfa.ncls;
  d.has_meta = p->dfa.has_meta;
  d.to_start = p->dfa.to_start;
  d.nop = nop;
  d.table_bytes = p->dfa.table_bytes();
  d.first_acc = p->dfa.first_acc;
  d.first_leaf = p->dfa.first_leaf;
  d.acc0 = p->dfa.accept[0] != 0;
  ugx::plan_filter(*pf, p->adv, d.plan);
  d.covers = ugx::prefilter_covers_matches(p->dfa, *pf, p->adv, matcher_flags) ? 1u : 0u;
  ugx::SearchDfa sd;
  plan_search(p->dfa, *pf, matcher_flags, p->adv, d.covers != 0, sd);
  d.n_word_ranges = sizeof(k_word_ranges) / sizeof(int) / 2;
  memcpy(d.chr, pf->chr, 256);
  set256(d.cbk, pf->cbk);
  set256(d.fst, pf->fst);
  if (pf->len == 0 && pf->pin >= 1 && pf->pin <= 16)
  {
    for (uint32_t i = 0; i < pf->pin; ++i)
    {
      uint32_t a = pf->chr[i], b = pf->chr[pf->pin + i];
      d.pin_a[a >> 5] |= 1u << (a & 31);
      d.pin_b[b >> 5] |= 1u << (b & 31);
    }
  }
  // accept words: bit 31 marks a state without outgoing byte edges (the interpreter halts there before reading)
  std::vector<uint32_t> acc(p->dfa.nstates);
  for (uint32_t s = 0; s < p->dfa.nstates; ++s)
  {
    bool any = false;
    for (uint32_t c = 0; c < p->dfa.ncls && !any; ++c)
      any = p->dfa.next[static_cast<size_t>(s) * p->dfa.ncls + c] != ugx::DEAD;
    acc[s] = (p->dfa.accept[s] & 0x7fffffffu) | (any ? 0u : 0x80000000u);
  }
  std::vector<uint32_t> opcp(opc, opc + nop);
  opcp.push_back(ugx::OP_HALT);
  opcp.push_back(ugx::OP_HALT);
  std::vector<uint16_t> next = p->dfa.next;
  next.resize((next.size() + 7) / 8 * 8, ugx::DEAD); // whole uint4s for the staging loop
  ugx::Viability via;
  ugx::build_viability(p->dfa, via);
  d.via_k = via.k;
  d.via_stride = via.stride;
  std::vector<uint32_t> via_t(512);
  for (int b = 0; b < 256; ++b)
  {
    via_t[2 * b] = via.t01[b];
    via_t[2 * b + 1] = via.t23[b];
  }
  if (via.k != 0 && via.bits.size() * 32 <= 8192)
  {
    // a small table is stored one byte per entry: the device then needs one load per position instead of load, shift, mask
    std::vector<uint32_t> bytes(via.bits.size() * 8, 0);
    for (size_t i = 0; i < via.bits.size() * 32; ++i)
      if ((via.bits[i >> 5] >> (i & 31)) & 1u)
        bytes[i >> 2] |= 1u << (8 * (i & 3));
    via.bits.swap(bytes);
    d.via_bytes = 1;
  }
  via.bits.resize((via.bits.size() + 3) / 4 * 4 + 4, 0); // whole uint4s for the staging copy
  via.pair.resize((via.pair.size() + 15) / 16 * 16 + 16, 0);
  d.via_words = static_cast<uint32_t>(via.bits.size());
  d.via_pair_bytes = static_cast<uint32_t>(via.pair.size());
  TRY(upload(p->allocs, d.cls, p->dfa.cls, 256));
  TRY(upload(p->allocs, d.next, next.data(), next.size() * 2));
  TRY(upload(p->allocs, d.accept, acc.data(), acc.size() * 4));
  TRY(upload(p->allocs, d.opc, opcp.data(), opcp.size() * 4));
  TRY(upload(p->allocs, d.pred, pf->min < 4 ? pf->pma : pf->pmh, UGX_HASH));
  TRY(upload(p->allocs, d.tap, pf->tap, UGX_BTAP));
  TRY(upload(p->allocs, d.word_ranges, k_word_ranges, sizeof(k_word_ranges)));
  TRY(upload(p->allocs, d.via_ids, via_t.data(), via_t.size() * 4));
  TRY(upload(p->allocs, d.via_bits, via.bits.data(), via.bits.size() * 4));
  TRY(upload(p->allocs, d.via_pair, via.pair.data(), via.pair.size()));
  if (sd.refusal == UGX_SEARCH_OK)
  {
    sd.next.resize((sd.next.size() + 7) / 8 * 8, 0); // whole 16-byte units for the bulk copy into shared memory
    TRY(upload(p->allocs, d.search_cls, sd.cls, 256));
    TRY(upload(p->allocs, d.search_next, sd.next.data(), sd.next.size() * 2));
    d.search_ok = 1;
    d.search_depth = sd.depth;
    d.search_ncls = sd.ncls;
    d.search_bytes = static_cast<uint32_t>(sd.next.size() * 2);
  }
  *out = holder.release();
  return UGX_OK;
}

static int plan_describe_impl(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, ugx_plan_info* out);

int ugx_plan_describe(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, ugx_plan_info* out)
{
  return guarded(UGX_E_INVALID, "ugx_plan_describe", [&] { return plan_describe_impl(opc, nop, pf, matcher_flags, out); });
}

static int plan_describe_impl(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, ugx_plan_info* out)
{
  if (opc == nullptr || nop == 0 || pf == nullptr || out == nullptr)
    return fail(UGX_E_INVALID, "ugx_plan_describe: null argument");
  ugx::HostDfa dfa;
  std::string err;
  int rc = ugx::flatten_dfa(opc, nop, dfa, err);
  if (rc != UGX_OK)
    return fail(rc, err);
  memset(out, 0, sizeof(*out));
  out->states = dfa.nstates;
  out->classes = dfa.ncls;
  out->table_bytes = dfa.table_bytes();
  out->first_acc = dfa.first_acc;
  out->first_leaf = dfa.first_leaf;
  out->max_match_len = dfa.max_match_len;
  out->has_meta = dfa.has_meta;
  out->newline_live = dfa.newline_live;
  const int adv = ugx::select_advance(*pf, matcher_flags);
  out->advance = adv;
  out->covers = ugx::prefilter_covers_matches(dfa, *pf, adv, matcher_flags) ? 1u : 0u;
  ugx::FilterPlan plan;
  ugx::plan_filter(*pf, adv, plan);
  out->kind = plan.kind;
  out->nterms = plan.nterms;
  for (int i = 0; i < 3; ++i)
    out->t_off[i] = plan.t_off[i];
  for (int i = 0; i < 2; ++i)
  {
    out->a_off[i] = plan.a_off[i];
    out->a_chr[i] = plan.a_chr[i] & 0xffu;
  }
  out->h4_terms = plan.h4_terms;
  out->h4_shift = plan.h4_shift;
  out->pm2 = plan.pm2;
  out->pm2_shift = plan.pm2_shift;
  memcpy(out->lut, plan.lut, sizeof(out->lut));
  rc = ugx::check_scope(dfa, *pf, matcher_flags, err);
  if (rc != UGX_OK)
    return fail(rc, err);
  return UGX_OK;
}

int ugx_viability_describe(const uint32_t* opc, uint32_t nop, uint32_t* k, uint32_t* stride, uint32_t* t01, uint32_t* t23,
                           uint8_t* pair, uint32_t cap_pair, uint32_t* npair, uint32_t* bits, uint32_t cap_words,
                           uint32_t* words)
{
  if (opc == nullptr || nop == 0 || k == nullptr || stride == nullptr || t01 == nullptr || t23 == nullptr ||
      npair == nullptr || words == nullptr)
    return fail(UGX_E_INVALID, "ugx_viability_describe: null argument");
  return guarded(UGX_E_NOMEM, nullptr, [&]() -> int {
    ugx::HostDfa dfa;
    std::string err;
    const int rc = ugx::flatten_dfa(opc, nop, dfa, err);
    if (rc != UGX_OK)
      return fail(rc, err);
    ugx::Viability v;
    ugx::build_viability(dfa, v);
    *k = v.k;
    *stride = v.stride;
    memcpy(t01, v.t01, sizeof(v.t01));
    memcpy(t23, v.t23, sizeof(v.t23));
    *npair = static_cast<uint32_t>(v.pair.size());
    *words = static_cast<uint32_t>(v.bits.size());
    if (v.bits.size() > cap_words || v.pair.size() > cap_pair)
      return fail(UGX_E_OVERFLOW, "viability table larger than the caller's buffer");
    if (!v.pair.empty() && pair != nullptr)
      memcpy(pair, v.pair.data(), v.pair.size());
    if (!v.bits.empty() && bits != nullptr)
      memcpy(bits, v.bits.data(), v.bits.size() * 4);
    return UGX_OK;
  });
}

int ugx_search_describe(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags,
                        ugx_search_info* out, uint8_t* cls, uint16_t* table, uint32_t cap)
{
  if (opc == nullptr || nop == 0 || pf == nullptr || out == nullptr)
    return fail(UGX_E_INVALID, "ugx_search_describe: null argument");
  return guarded(UGX_E_NOMEM, nullptr, [&]() -> int {
    ugx::HostDfa dfa;
    std::string err;
    int rc = ugx::flatten_dfa(opc, nop, dfa, err);
    if (rc == UGX_OK)
      rc = ugx::check_scope(dfa, *pf, matcher_flags, err);
    if (rc != UGX_OK)
      return fail(rc, err);
    const int adv = ugx::select_advance(*pf, matcher_flags);
    ugx::SearchDfa sd;
    plan_search(dfa, *pf, matcher_flags, adv, ugx::prefilter_covers_matches(dfa, *pf, adv, matcher_flags), sd);
    memset(out, 0, sizeof(*out));
    out->eligible = sd.refusal == UGX_SEARCH_OK ? 1u : 0u;
    out->refusal = sd.refusal;
    out->depth = sd.depth;
    out->states = sd.next.empty() ? 0u : sd.nstates;
    out->classes = sd.next.empty() ? 0u : sd.ncls;
    out->table_bytes = sd.next.empty() ? 0u : sd.table_bytes();
    if (sd.next.empty())
      return UGX_OK;
    if (cls != nullptr)
      memcpy(cls, sd.cls, 256);
    if (table != nullptr)
    {
      if (sd.next.size() > cap)
        return fail(UGX_E_OVERFLOW, "search table larger than the caller's buffer");
      memcpy(table, sd.next.data(), sd.next.size() * 2);
    }
    return UGX_OK;
  });
}

int ugx_pattern_load(const char* path, int device, ugx_pattern** out)
{
  FILE* f = fopen(path, "rb");
  if (f == nullptr)
    return fail(UGX_E_IO, std::string("cannot open ") + path);
  ugx_file_header h;
  ugx_prefilter pf;
  std::vector<uint32_t> opc;
  bool ok = fread(&h, sizeof(h), 1, f) == 1 && memcmp(h.magic, UGX_FILE_MAGIC, 8) == 0 &&
            h.prefilter_size == sizeof(pf) && fread(&pf, sizeof(pf), 1, f) == 1;
  if (ok)
  {
    // the opcode count comes from the file: it must fit in what is left of the file before anything is allocated
    const long here = ftell(f);
    ok = here >= 0 && fseek(f, 0, SEEK_END) == 0;
    const long size = ok ? ftell(f) : -1;
    ok = ok && size >= here && h.nop > 0 && static_cast<uint64_t>(h.nop) * 4 <= static_cast<uint64_t>(size - here) &&
         fseek(f, here, SEEK_SET) == 0;
  }
  if (ok)
  {
    try
    {
      opc.resize(h.nop);
    }
    catch (const std::exception&)
    {
      fclose(f);
      return fail(UGX_E_NOMEM, "out of host memory");
    }
    ok = fread(opc.data(), 4, h.nop, f) == h.nop;
  }
  fclose(f);
  if (!ok)
    return fail(UGX_E_IO, std::string("not a UGXP pattern file: ") + path);
  return ugx_pattern_create(opc.data(), h.nop, &pf, h.matcher_flags, device, out);
}

int ugx_pattern_info_get(const ugx_pattern* p, ugx_pattern_info* info)
{
  if (p == nullptr || info == nullptr)
    return fail(UGX_E_INVALID, "null argument");
  info->nop = p->nop;
  info->states = p->dfa.nstates;
  info->classes = p->dfa.ncls;
  info->table_bytes = p->dfa.table_bytes();
  info->table_in_smem = !p->dfa.has_meta && p->dfa.table_bytes() <= ugx::SCAN_MAX_SMEM_TABLE;
  info->advance = p->adv;
  info->has_meta = p->dfa.has_meta;
  info->lookback = p->pf.lbk != 0;
  return UGX_OK;
}

void ugx_pattern_destroy(ugx_pattern* p)
{
  if (p != nullptr)
  {
    cudaSetDevice(p->device);
    delete p;
  }
}

int ugx_scanner_create(int device, void* stream, ugx_scanner** out)
{
  if (out == nullptr)
    return fail(UGX_E_INVALID, "null argument");
  CU(cudaSetDevice(device));
  ugx_scanner* s = new (std::nothrow) ugx_scanner();
  if (s == nullptr)
    return fail(UGX_E_NOMEM, "out of host memory");
  s->device = device;
  s->stream = static_cast<cudaStream_t>(stream);
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e == cudaSuccess)
    e = cudaEventCreate(&s->ev0);
  if (e == cudaSuccess)
    e = cudaEventCreate(&s->ev1);
  if (e == cudaSuccess)
    e = cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess)
    e = cudaEventCreateWithFlags(&s->ev_copy, cudaEventDisableTiming);
  if (e == cudaSuccess)
    e = cudaMalloc(reinterpret_cast<void**>(&s->totals), ugx::SLOT_COUNT * sizeof(unsigned long long));
  if (e == cudaSuccess)
    e = cudaMallocHost(reinterpret_cast<void**>(&s->h_totals), ugx::SLOT_COUNT * sizeof(unsigned long long));
  if (e == cudaSuccess)
    e = cudaMalloc(reinterpret_cast<void**>(&s->partials), 2 * ugx::STREAM_MAX_GRID * sizeof(unsigned long long));
  if (e == cudaSuccess)
    e = cudaMalloc(reinterpret_cast<void**>(&s->ticket), 2 * sizeof(unsigned long long));
  if (e == cudaSuccess)
    e = cudaMemset(s->ticket, 0, 2 * sizeof(unsigned long long));
  if (e != cudaSuccess)
  {
    ugx_scanner_destroy(s);
    return cuda_fail(e, "ugx_scanner_create");
  }
  s->device_sms = s->sm_count = prop.multiProcessorCount;
  *out = s;
  return UGX_OK;
}

void ugx_scanner_destroy(ugx_scanner* s)
{
  if (s == nullptr)
    return;
  cudaSetDevice(s->device); // the scratch buffers are freed by their destructors in `delete s`
  cudaFree(s->totals);
  cudaFreeHost(s->h_totals);
  for (uint8_t* p : s->feed_slots)
    cudaFreeHost(p);
  for (cudaEvent_t e : s->feed_events)
    cudaEventDestroy(e);
  for (cudaStream_t st : s->feed_streams)
    cudaStreamDestroy(st);
  cudaFree(s->partials);
  cudaFree(s->ticket);
  if (s->ev0)
    cudaEventDestroy(s->ev0);
  if (s->ev1)
    cudaEventDestroy(s->ev1);
  if (s->ev_copy)
    cudaEventDestroy(s->ev_copy);
  if (s->copy_stream)
    cudaStreamDestroy(s->copy_stream);
  delete s;
}

} // extern "C"

namespace {

constexpr uint64_t FEED_CHUNK = 8ull << 20; // bytes per pinned slot of the pageable feeder
constexpr uint64_t FEED_MIN = 32ull << 20;  // smaller pageable buffers take one plain copy

// Host-to-device copy of a PAGEABLE buffer (what an mmap'ing caller such as ugrep hands over).  cudaMemcpyAsync from
// pageable memory goes through the driver's own staging at ~10 GB/s on this box; here K host threads copy 8 MiB chunks
// into pinned slots (two per thread) and send each slot on the thread's own stream, so the memcpy's of some chunks
// overlap the DMA of others.  The scan stream waits on every thread's last copy.
int feed_pageable(ugx_scanner* s, uint8_t* dst, const uint8_t* src, uint64_t n)
{
  if (s->feed_streams.empty())
  {
    // half the host threads, shared between the ranks of this box when there are several (torchrun's LOCAL_WORLD_SIZE)
    unsigned hw = std::thread::hardware_concurrency();
    unsigned ranks = 1;
    if (const char* lws = getenv("LOCAL_WORLD_SIZE"))
      ranks = static_cast<unsigned>(atoi(lws)) > 0 ? static_cast<unsigned>(atoi(lws)) : 1;
    unsigned k = hw / (2 * ranks);
    if (const char* env = getenv("UGX_FEED_THREADS"))
      k = static_cast<unsigned>(atoi(env));
    if (k < 2)
      k = 2;
    if (k > 8)
      k = 8;
    // all or nothing: a feeder that could not get its streams / pinned slots leaves no half-built state behind
    cudaError_t e = cudaSuccess;
    for (unsigned i = 0; i < k && e == cudaSuccess; ++i)
    {
      cudaStream_t st = nullptr;
      e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
      if (e != cudaSuccess)
        break;
      s->feed_streams.push_back(st);
      for (int j = 0; j < 2 && e == cudaSuccess; ++j)
      {
        void* p = nullptr;
        e = cudaHostAlloc(&p, FEED_CHUNK, cudaHostAllocDefault);
        if (e != cudaSuccess)
          break;
        s->feed_slots.push_back(static_cast<uint8_t*>(p));
        cudaEvent_t ev = nullptr;
        e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (e == cudaSuccess)
          s->feed_events.push_back(ev);
      }
    }
    if (e != cudaSuccess)
    {
      for (uint8_t* p : s->feed_slots)
        cudaFreeHost(p);
      for (cudaEvent_t ev : s->feed_events)
        cudaEventDestroy(ev);
      for (cudaStream_t st : s->feed_streams)
        cudaStreamDestroy(st);
      s->feed_slots.clear();
      s->feed_events.clear();
      s->feed_streams.clear();
      return cuda_fail(e, "pageable feeder setup");
    }
  }
  const unsigned K = static_cast<unsigned>(s->feed_streams.size());
  const uint64_t nchunks = (n + FEED_CHUNK - 1) / FEED_CHUNK;
  std::vector<cudaError_t> errs(K, cudaSuccess);
  std::vector<std::thread> workers;
  for (unsigned w = 0; w < K; ++w)
    workers.emplace_back([&, w]() {
      cudaError_t e = cudaSetDevice(s->device);
      uint64_t round = 0;
      for (uint64_t c = w; c < nchunks && e == cudaSuccess; c += K, ++round)
      {
        const unsigned slot = 2 * w + static_cast<unsigned>(round & 1);
        if (round >= 2)
          e = cudaEventSynchronize(s->feed_events[slot]); // the slot's previous copy has left it
        if (e != cudaSuccess)
          break;
        const uint64_t off = c * FEED_CHUNK;
        const uint64_t len = n - off < FEED_CHUNK ? n - off : FEED_CHUNK;
        memcpy(s->feed_slots[slot], src + off, len);
        e = cudaMemcpyAsync(dst + off, s->feed_slots[slot], len, cudaMemcpyHostToDevice, s->feed_streams[w]);
        if (e == cudaSuccess)
          e = cudaEventRecord(s->feed_events[slot], s->feed_streams[w]);
      }
      errs[w] = e;
    });
  for (auto& t : workers)
    t.join();
  for (unsigned w = 0; w < K; ++w)
    if (errs[w] != cudaSuccess)
      return cuda_fail(errs[w], "pageable feeder");
  // the scan stream continues after the last copy of every feeder stream
  for (unsigned w = 0; w < K; ++w)
  {
    CU(cudaEventRecord(s->ev_copy, s->feed_streams[w]));
    CU(cudaStreamWaitEvent(s->stream, s->ev_copy, 0));
  }
  return UGX_OK;
}

// make `buf` visible to the device: device pointers are used in place, host pointers are staged
int resolve(ugx_scanner* s, const void* buf, uint64_t n, const uint8_t** dev)
{
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, buf);
  if (e == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged))
  {
    if ((reinterpret_cast<uintptr_t>(buf) & 15) == 0)
    {
      *dev = static_cast<const uint8_t*>(buf);
      return UGX_OK;
    }
    // the kernels use 16-byte vector loads: a misaligned device buffer is copied to aligned scratch
    TRY(s->stage.ensure(n + 16));
    CU(cudaMemcpyAsync(s->stage.p, buf, n, cudaMemcpyDeviceToDevice, s->stream));
    *dev = s->stage.p;
    return UGX_OK;
  }
  if (e != cudaSuccess)
    cudaGetLastError(); // plain host memory on older drivers reports an error: clear it
  TRY(s->stage.ensure(n + 16));
  const bool pageable = e != cudaSuccess || at.type == cudaMemoryTypeUnregistered;
  if (pageable && n >= FEED_MIN && !s->no_feeder)
  {
    // earlier work on the scan stream may still read the staging buffer
    CU(cudaStreamSynchronize(s->stream));
    TRY(feed_pageable(s, s->stage.p, static_cast<const uint8_t*>(buf), n));
  }
  else
    CU(cudaMemcpyAsync(s->stage.p, buf, n, cudaMemcpyHostToDevice, s->stream));
  *dev = s->stage.p;
  return UGX_OK;
}

constexpr uint64_t PIPE_CHUNK = 32ull << 20; // bytes per host-to-device chunk of the pipelined path (region-aligned)

// a host buffer the pipelined path takes: page-locked memory (cudaHostAlloc / cudaHostRegister: DMA reads it
// directly), and with pageable_too any host memory
bool pipeline_source(const void* buf, bool pageable_too)
{
  cudaPointerAttributes at;
  const cudaError_t e = cudaPointerGetAttributes(&at, buf);
  if (e != cudaSuccess)
  {
    cudaGetLastError();
    return pageable_too;
  }
  return at.type == cudaMemoryTypeHost ||
         (pageable_too && at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged);
}

// ---- the call frame of the scan entry points ----
// An entry point checks its arguments (check_scan) and zeroes its outputs.  begin_scan answers an empty buffer with
// *totals = tt and no device work (*dbuf stays nullptr); otherwise it sets the device, makes the buffer visible to the
// device (resolve; with stage_only just the staging buffer, which the pipelined stream route fills itself), enqueues
// `setup` (what is not kernel time: uploads, flags to zero, scratch) and records ev0 before the first launch.
// end_scan records ev1 after the last launch and the copies of the results, waits for the stream, and fills
// kernel_ms, the results `read` from h_totals and *totals.

// the checks of a scan over one pattern, in the order the entry points report them; `who` names the entry point
int check_scan(const char* who, const ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t n, uint32_t flags = 0)
{
  if (s == nullptr || p == nullptr || (buf == nullptr && n != 0))
    return fail(UGX_E_INVALID, "null argument");
  if ((flags & ~UGX_LINES_INVERT) != 0)
    return fail(UGX_E_INVALID, std::string(who) + ": unknown flags");
  if (s->device != p->device)
    return fail(UGX_E_INVALID, "pattern and scanner live on different devices");
  return UGX_OK;
}

int no_setup() { return UGX_OK; }

template <typename Setup = int (&)()>
int begin_scan(ugx_scanner* s, const void* buf, uint64_t n, const ugx_totals& tt, ugx_totals* totals, const uint8_t** dbuf,
               Setup&& setup = no_setup, bool stage_only = false)
{
  *dbuf = nullptr;
  if (n == 0)
  {
    if (totals)
      *totals = tt;
    return UGX_OK;
  }
  CU(cudaSetDevice(s->device));
  TRY(stage_only ? s->stage.ensure(n + 16) : resolve(s, buf, n, dbuf));
  if (stage_only)
    *dbuf = s->stage.p;
  TRY(setup());
  CU(cudaEventRecord(s->ev0, s->stream));
  return UGX_OK;
}

enum : unsigned { READ_MATCHES = 1, READ_NEWLINES = 2 }; // results end_scan takes from h_totals

// ev1_recorded: the caller stopped the clock itself, before copies that are not kernel time
int end_scan(ugx_scanner* s, ugx_totals& tt, ugx_totals* totals, unsigned read = 0, bool ev1_recorded = false)
{
  if (!ev1_recorded)
    CU(cudaEventRecord(s->ev1, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  CU(cudaEventElapsedTime(&tt.kernel_ms, s->ev0, s->ev1));
  if (read & READ_MATCHES)
    tt.matches = s->h_totals[ugx::SLOT_MATCHES];
  if (read & READ_NEWLINES)
    tt.newlines = s->h_totals[ugx::SLOT_NEWLINES];
  if (totals)
    *totals = tt;
  return UGX_OK;
}

// the host's read of totals slots [0, k) after a count pass
int read_totals(ugx_scanner* s, int k)
{
  CU(cudaMemcpyAsync(s->h_totals, s->totals, k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  return UGX_OK;
}

// ... and the arena grown for the *nrec = h_totals[SLOT_MATCHES] records of the emit pass
template <typename T>
int read_count(ugx_scanner* s, int k, DevBuf<T>& arena, uint64_t* nrec)
{
  TRY(read_totals(s, k));
  *nrec = s->h_totals[ugx::SLOT_MATCHES];
  return arena.ensure(*nrec);
}

// the records of the last call from the device to the caller's out[cap]; *n_out is set before an overflow is reported.
// With keep_on_device (the batch calls), out == NULL with cap == 0 leaves the records on the device.
int copy_out(ugx_scanner* s, const void* dev, size_t rec_bytes, uint64_t n, void* out, uint64_t cap, uint64_t* n_out,
             bool keep_on_device, const char* overflow)
{
  if (n_out)
    *n_out = n;
  if (keep_on_device && out == nullptr && cap == 0)
    return UGX_OK;
  if (n > cap)
    return fail(UGX_E_OVERFLOW, overflow);
  if (n > 0)
  {
    if (out == nullptr)
      return fail(UGX_E_INVALID, "null record buffer");
    CU(cudaMemcpyAsync(out, dev, n * rec_bytes, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaStreamSynchronize(s->stream));
  }
  return UGX_OK;
}

// ugx_scanner_fetch / ugx_scanner_fetch_lines: records [first, first + count) of the n in `arena`
template <typename R>
int fetch(ugx_scanner* s, const DevBuf<R>& arena, uint64_t n, R* out, uint64_t first, uint64_t count, const char* range)
{
  if (first > n || count > n - first)
    return fail(UGX_E_INVALID, range);
  if (count == 0)
    return UGX_OK;
  CU(cudaSetDevice(s->device));
  CU(cudaMemcpyAsync(out, arena.p + first, count * sizeof(R), cudaMemcpyDeviceToHost, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  return UGX_OK;
}

// the record outputs of an entry point: zeroed on entry, the arena and its count once a result stands
template <typename R>
void set_records(const R** dev_out, uint64_t* n_out, const R* dev, uint64_t n)
{
  if (n_out)
    *n_out = n;
  if (dev_out)
    *dev_out = dev;
}

// the per-tile sums of the line-at-a-time and batch kernels
int ensure_tiles(ugx_scanner* s, uint64_t ntiles)
{
  TRY(s->tile_matches.ensure(ntiles));
  return s->tile_newlines.ensure(ntiles);
}

// reflex::nlcount into the newlines slot, read back by end_scan (READ_NEWLINES): ugx_count_newlines, and every scan
// with a pattern whose prefilter admits no candidate
int newline_pass(ugx_scanner* s, const uint8_t* dbuf, uint64_t n, ugx_totals& tt)
{
  CU(ugx::launch_count_newlines(dbuf, n, s->totals + ugx::SLOT_NEWLINES, s->sm_count, s->stream));
  CU(cudaMemcpyAsync(s->h_totals + ugx::SLOT_NEWLINES, s->totals + ugx::SLOT_NEWLINES, sizeof(unsigned long long),
                     cudaMemcpyDeviceToHost, s->stream));
  tt.flags |= UGX_TOT_NEWLINES;
  tt.launches = 1;
  tt.kernel = UGX_K_NEWLINES;
  return UGX_OK;
}

// the count pass of the span kernels (last line, span_scan_kernel, span_final_kernel) up to the host's read of
// s->h_totals[0..2]; with want_sel the selected match starts are left in s->span_sel
int span_count_pass(ugx_scanner* s, const ugx_pattern* p, const uint8_t* dbuf, uint64_t n, bool want_sel, uint64_t base_offset,
                    uint64_t base_line, ugx::SpanArgs& a, ugx_totals* tt)
{
  const uint64_t nreg = ugx::stream_regions(n);
  TRY(s->span_regions.ensure(5 * nreg + 8));
  if (want_sel)
    TRY(s->span_sel.ensure((n + 15) / 16 + 64));
  memset(&a, 0, sizeof(a));
  a.reg_matches = s->span_regions.p;
  a.reg_newlines = s->span_regions.p + nreg;
  a.reg_emain = s->span_regions.p + 2 * nreg;
  a.reg_elast = s->span_regions.p + 3 * nreg;
  a.reg_v = s->span_regions.p + 4 * nreg;
  a.sel_bits = want_sel ? s->span_sel.p : nullptr;
  a.base_offset = base_offset;
  a.base_line = base_line;
  a.no_cover = s->no_cover ? 1u : 0u;
  a.tail = reinterpret_cast<const uint64_t*>(s->totals + ugx::SLOT_LAST_LINE);
  a.flags = reinterpret_cast<unsigned int*>(s->totals + ugx::SLOT_SPAN_FLAGS);
  CU(cudaMemsetAsync(s->totals + ugx::SLOT_SPAN_FLAGS, 0, sizeof(unsigned long long), s->stream));
  CU(ugx::launch_last_line(dbuf, n, reinterpret_cast<uint64_t*>(s->totals + ugx::SLOT_LAST_LINE), s->stream));
  CU(ugx::launch_span_scan(p->dev, dbuf, n, a, false, s->sm_count, s->stream));
  CU(ugx::launch_span_final(p->dev, dbuf, n, a, false, s->totals, s->stream));
  TRY(read_totals(s, 3));
  tt->launches += 3;
  return UGX_OK;
}

// ScanArgs of the line-at-a-time kernels over dbuf[0, n), with the scanner's tile sums and, for the count pass of
// records, its strip counts
int line_scan_args(ugx_scanner* s, const ugx_pattern* p, const uint8_t* dbuf, uint64_t n, bool strips, uint64_t base_offset,
                   uint64_t base_line, ugx::ScanArgs& a)
{
  const uint64_t tile_bytes = ugx::scan_tile_bytes(p->dev);
  const uint64_t ntiles = (n + tile_bytes - 1) / tile_bytes;
  TRY(ensure_tiles(s, ntiles));
  if (strips)
    TRY(s->strip_counts.ensure((n + ugx::SCAN_STRIP - 1) / ugx::SCAN_STRIP));
  a.buf = dbuf;
  a.n = n;
  a.ntiles = ntiles;
  a.tile_matches = s->tile_matches.p;
  a.tile_newlines = s->tile_newlines.p;
  a.strip_counts = strips ? s->strip_counts.p : nullptr;
  a.out = nullptr;
  a.out_cap = 0;
  a.base_offset = base_offset;
  a.base_line = base_line;
  return UGX_OK;
}

// ---- ugx_count_lines / ugx_count_matches / ugx_find_all*: scan_route picks a route, and each route reports its own
// results: the totals, the results its last copy leaves in h_totals for end_scan (`read`), and the match records ----
enum class Route {
  NEVER,       // the prefilter admits no candidate: the result is empty, the pass over the text only counts newlines
  SPAN,        // the span kernels; they may hand over to RECORDS or LINE_SCAN
  STREAM,      // streaming `-c`: literal, DFA or search automaton
  TILE_ANY,    // the tile-synchronous count_lines_any_kernel
  MATCH_LINES, // counting with position-parallel attempts
  RECORDS,     // single-pass match records: staging pass, prefix, reorder
  TWO_PASS,    // match records by a count pass and an emit pass of the line scan
  LINE_SCAN,   // counting with scan_lines_kernel
};

// the span kernels take line records, and match counts and records where scan_route allows, unless an option sends
// the scan to the line-at-a-time kernels
bool span_route(const ugx_scanner* s, const ugx_pattern* p)
{
  return !p->never && !s->force_generic && !s->no_span && ugx::span_scan_eligible(p->dev);
}

Route scan_route(const ugx_scanner* s, const ugx_pattern* p, int mode, bool want_records)
{
  const ugx::DevPattern& d = p->dev;
  if (p->never)
    return Route::NEVER;
  if (mode == 1 && !s->match_lines && !s->two_pass_records && span_route(s, p))
    return Route::SPAN;
  if (mode == 0 && !want_records && !s->force_generic)
  {
    if (!s->legacy_any && ugx::count_lines_stream_eligible(d) &&
        (s->stream_dfa || ugx::count_lines_literal_eligible(d) || d.plan.h4_terms >= 1 || d.plan.pm2 != 0 ||
         (d.plan.kind == ugx::FK_LUT && d.plan.nterms >= 1 && d.one == 0)))
      return Route::STREAM;
    if (ugx::count_lines_any_eligible(d))
      return Route::TILE_ANY;
  }
  if (!want_records && !s->force_generic && s->match_lines && ugx::match_lines_eligible(d))
    return Route::MATCH_LINES;
  if (want_records)
    return s->two_pass_records ? Route::TWO_PASS : Route::RECORDS;
  return Route::LINE_SCAN;
}

// one call: its arguments, the device view of its buffer, ScanArgs of the line-at-a-time routes, and the results
struct Scan {
  ugx_scanner* s;
  const ugx_pattern* p;
  const void* buf;
  uint64_t n;
  int mode;
  bool want_records;
  uint64_t base_offset, base_line;
  const ugx_match** dev_out;
  uint64_t* n_out;
  const uint8_t* dbuf;
  ugx::ScanArgs a;
  ugx_totals tt;
  unsigned read;
};

// the end of a counting route: the two result slots to the host for end_scan
int copy_results(Scan& c, bool newlines)
{
  CU(cudaMemcpyAsync(c.s->h_totals, c.s->totals, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c.s->stream));
  c.read = READ_MATCHES | READ_NEWLINES;
  if (newlines)
    c.tt.flags |= UGX_TOT_NEWLINES;
  return UGX_OK;
}

// the end of a records route: the match arena holds nrec records, published to the caller
void publish_records(Scan& c, uint64_t nrec)
{
  c.s->records_n = nrec;
  set_records(c.dev_out, c.n_out, c.s->records.p, nrec);
}

// Route::SPAN (span_scan.cu).  *valid = false: the spans could not vouch for their result on this buffer (a match
// longer than a window across a region start in a line without newlines, an attempt that failed at the very end of
// the buffer, a match of 64 KiB or more) — the caller then takes the line-at-a-time kernels.
int scan_spans(Scan& c, bool* valid)
{
  ugx_scanner* s = c.s;
  *valid = false;
  ugx::SpanArgs a;
  TRY(span_count_pass(s, c.p, c.dbuf, c.n, c.want_records, c.base_offset, c.base_line, a, &c.tt));
  if (s->h_totals[ugx::SLOT_HANDOVER] != 0)
    return UGX_OK; // not valid: nothing of this attempt is used
  const uint64_t nrec = s->h_totals[ugx::SLOT_MATCHES];
  if (c.want_records)
  {
    TRY(s->records.ensure(nrec));
    if (nrec > 0)
    {
      a.out = s->records.p;
      a.out_cap = nrec;
      CU(ugx::launch_span_scan(c.p->dev, c.dbuf, c.n, a, true, s->sm_count, s->stream));
      CU(ugx::launch_span_final(c.p->dev, c.dbuf, c.n, a, true, s->totals, s->stream));
      c.tt.launches += 2;
    }
    publish_records(c, nrec);
  }
  c.tt.matches = nrec;
  c.tt.newlines = s->h_totals[ugx::SLOT_NEWLINES];
  c.tt.flags |= UGX_TOT_NEWLINES;
  c.tt.kernel = UGX_K_SPAN;
  *valid = true;
  return UGX_OK;
}

// Route::STREAM; a pipelined host buffer is copied into s->stage here
int stream_count(Scan& c, bool pipelined)
{
  ugx_scanner* s = c.s;
  const ugx_pattern* p = c.p;
  const uint8_t* dbuf = c.dbuf;
  const uint64_t n = c.n;
  TRY(s->region_sum.ensure(ugx::stream_regions(n) + 64));
  ugx::StreamArgs sa;
  sa.region_sum = s->region_sum.p;
  sa.partials = s->partials;
  sa.ticket = s->ticket;
  sa.done = reinterpret_cast<unsigned int*>(s->ticket + 1);
  sa.totals = s->totals;
  sa.stage_table = 0;
  sa.use_h4 = 0;
  sa.use_via = 0;
  sa.no_cover = s->no_cover ? 1u : 0u;
  const uint64_t nreg = ugx::stream_regions(n);
  const bool search = p->dev.search_ok != 0 && !s->no_search;
  if (pipelined)
  {
    // host buffer: copy in chunks on the copy stream and scan chunk i while chunk i + 1 is in flight.  A launch
    // trails the copied bytes by one region, so that every read of a scanned position (literal verify, a DFA
    // attempt of bounded length) finds its bytes; the region summaries chain the launches.
    uint64_t copied = 0, scanned = 0;
    c.tt.launches = 0;
    while (scanned < nreg)
    {
      const uint64_t take = n - copied < PIPE_CHUNK ? n - copied : PIPE_CHUNK;
      if (take > 0)
      {
        CU(cudaMemcpyAsync(s->stage.p + copied, static_cast<const uint8_t*>(c.buf) + copied, take, cudaMemcpyHostToDevice,
                           s->copy_stream));
        copied += take;
        CU(cudaEventRecord(s->ev_copy, s->copy_stream));
        CU(cudaStreamWaitEvent(s->stream, s->ev_copy, 0));
      }
      const uint64_t upto = copied == n ? nreg : copied / ugx::SC_REGION - 1;
      if (upto <= scanned)
        continue;
      sa.region_begin = scanned;
      sa.region_end = upto;
      sa.finalize = upto == nreg ? 1u : 0u;
      sa.accumulate = scanned == 0 ? 0u : 1u;
      CU(search ? ugx::launch_count_lines_search(p->dev, dbuf, copied, sa, s->count_newlines, s->sm_count, s->stream)
                : ugx::launch_count_lines_stream(p->dev, dbuf, copied, sa, s->count_newlines, s->sm_count, s->stream));
      scanned = upto;
      ++c.tt.launches;
    }
  }
  else
  {
    sa.region_begin = 0;
    sa.region_end = nreg;
    sa.finalize = 1;
    sa.accumulate = 0;
    CU(search ? ugx::launch_count_lines_search(p->dev, dbuf, n, sa, s->count_newlines, s->sm_count, s->stream)
              : ugx::launch_count_lines_stream(p->dev, dbuf, n, sa, s->count_newlines, s->sm_count, s->stream));
    c.tt.launches = 1;
  }
  c.tt.kernel = ugx::count_lines_literal_eligible(p->dev) ? UGX_K_STREAM_LITERAL
                : search                                   ? UGX_K_STREAM_SEARCH
                                                           : UGX_K_STREAM_DFA;
  return copy_results(c, s->count_newlines);
}

// Route::MATCH_LINES (match_lines.cu); its tiles are smaller than the line scan's
int match_lines_count(Scan& c)
{
  ugx_scanner* s = c.s;
  const uint64_t tb = ugx::match_lines_tile_bytes(c.p->dev);
  const uint64_t nt = (c.n + tb - 1) / tb;
  TRY(ensure_tiles(s, nt));
  c.a.ntiles = nt;
  c.a.tile_matches = s->tile_matches.p;
  c.a.tile_newlines = s->tile_newlines.p;
  CU(ugx::launch_match_lines(c.p->dev, c.a, c.mode, s->sm_count, s->stream));
  CU(ugx::launch_tile_prefix(s->tile_matches.p, s->tile_newlines.p, nt, s->totals, s->stream));
  c.tt.launches = 2;
  c.tt.kernel = UGX_K_MATCH_LINES;
  return copy_results(c, true);
}

// Route::RECORDS: staging pass (tiles in completion order) + prefix + reorder into input order.  The staging capacity
// is a guess (the last result, or one record per 96 bytes); the cursor tells the exact need, so a second staging pass
// always fits.
int staged_records(Scan& c)
{
  ugx_scanner* s = c.s;
  const ugx::ScanArgs& a = c.a;
  TRY(s->tile_base.ensure(a.ntiles));
  TRY(s->rec_stage.ensure(s->records_n + s->records_n / 4 + a.n / 96 + 1024));
  unsigned long long* cursor = s->totals + ugx::SLOT_HANDOVER;
  uint64_t nrec = 0;
  for (int attempt = 0; attempt < 2; ++attempt)
  {
    CU(ugx::launch_scan_records(c.p->dev, a, s->tile_base.p, s->rec_stage.p, s->rec_stage.cap, cursor, s->sm_count, s->stream));
    CU(ugx::launch_tile_prefix(a.tile_matches, a.tile_newlines, a.ntiles, s->totals, s->stream));
    TRY(read_totals(s, 2));
    c.tt.launches += 2;
    nrec = s->h_totals[ugx::SLOT_MATCHES];
    if (nrec <= s->rec_stage.cap)
      break;
    if (attempt == 1)
      return fail(UGX_E_CUDA, "record staging overflowed twice");
    TRY(s->rec_stage.ensure(nrec));
  }
  TRY(s->records.ensure(nrec));
  if (nrec > 0)
  {
    CU(ugx::launch_reorder_records(s->rec_stage.p, s->records.p, a.tile_matches, a.tile_newlines, s->tile_base.p, a.ntiles,
                                   s->totals, a.base_line, s->sm_count, s->stream));
    c.tt.launches += 1;
  }
  c.tt.kernel = UGX_K_RECORDS;
  c.tt.flags |= UGX_TOT_NEWLINES;
  c.read = READ_MATCHES | READ_NEWLINES; // left in h_totals by the last staging pass
  publish_records(c, nrec);
  return UGX_OK;
}

// Route::TWO_PASS: the line scan's count pass into the strip counts, the tile prefix, and its emit pass
int two_pass_records(Scan& c)
{
  ugx_scanner* s = c.s;
  CU(ugx::launch_scan_lines(c.p->dev, c.a, c.mode, false, s->sm_count, s->stream));
  CU(ugx::launch_tile_prefix(c.a.tile_matches, c.a.tile_newlines, c.a.ntiles, s->totals, s->stream));
  c.tt.launches = 2;
  c.tt.kernel = UGX_K_LINE_SCAN;
  uint64_t nrec = 0;
  TRY(read_count(s, 2, s->records, &nrec));
  if (nrec > 0)
  {
    c.a.out = s->records.p;
    c.a.out_cap = nrec;
    CU(ugx::launch_scan_lines(c.p->dev, c.a, c.mode, true, s->sm_count, s->stream));
    c.tt.launches += 1;
  }
  c.tt.flags |= UGX_TOT_NEWLINES;
  c.read = READ_MATCHES | READ_NEWLINES; // left in h_totals by the count pass
  publish_records(c, nrec);
  return UGX_OK;
}

// every route but SPAN, once ScanArgs and ev0 are in place
int run_route(Scan& c, Route r, bool pipelined)
{
  ugx_scanner* s = c.s;
  switch (r)
  {
    case Route::NEVER:
      TRY(newline_pass(s, c.dbuf, c.n, c.tt));
      c.read = READ_NEWLINES;
      s->records_n = 0;
      return UGX_OK;
    case Route::SPAN: return UGX_OK; // scan_spans has run
    case Route::STREAM: return stream_count(c, pipelined);
    case Route::TILE_ANY:
      CU(ugx::launch_count_lines_any(c.p->dev, c.dbuf, c.n, s->totals, s->sm_count, s->stream));
      c.tt.launches = 1;
      c.tt.kernel = UGX_K_TILE_ANY;
      return copy_results(c, true);
    case Route::MATCH_LINES: return match_lines_count(c);
    case Route::RECORDS: return staged_records(c);
    case Route::TWO_PASS: return two_pass_records(c);
    case Route::LINE_SCAN: break;
  }
  CU(ugx::launch_scan_lines(c.p->dev, c.a, c.mode, false, s->sm_count, s->stream));
  CU(ugx::launch_tile_prefix(c.a.tile_matches, c.a.tile_newlines, c.a.ntiles, s->totals, s->stream));
  c.tt.launches = 2;
  c.tt.kernel = UGX_K_LINE_SCAN;
  return copy_results(c, true);
}

int scan_common(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t n, int mode, bool want_records,
                uint64_t base_offset, uint64_t base_line, const ugx_match** dev_out, uint64_t* n_out, ugx_totals* totals)
{
  TRY(check_scan("scan", s, p, buf, n));
  Scan c{s, p, buf, n, mode, want_records, base_offset, base_line, dev_out, n_out};
  set_records<ugx_match>(dev_out, n_out, nullptr, 0);
  Route r = scan_route(s, p, mode, want_records);
  // a host buffer on the streaming route is copied chunk by chunk, overlapped with the scan, when every read of a
  // scanned position stays within one region of it: pure literals, and DFAs whose longest match is bounded
  const bool bounded = ugx::count_lines_literal_eligible(p->dev) || p->dfa.max_match_len < ugx::SC_REGION - 512;
  // (chunk-wise overlap of copy and scan for page-locked buffers; pageable ones go through the feeder threads of resolve())
  const bool pipelined = r == Route::STREAM && bounded && !s->no_pipeline && n >= 2 * PIPE_CHUNK &&
                         pipeline_source(buf, s->no_feeder);
  // the line-at-a-time routes size their tile sums before the clock starts
  const bool tiles = r != Route::NEVER && r != Route::SPAN;
  TRY(begin_scan(s, buf, n, c.tt, totals, &c.dbuf, [&]() -> int {
    return tiles ? line_scan_args(s, p, c.dbuf, n, r == Route::TWO_PASS, base_offset, base_line, c.a) : UGX_OK;
  }, pipelined));
  if (c.dbuf == nullptr)
    return UGX_OK;
  if (r == Route::SPAN)
  {
    bool valid = false;
    TRY(scan_spans(c, &valid));
    if (!valid)
    {
      // the line-at-a-time kernels take over (the span route excludes match_lines and two_pass_records)
      r = want_records ? Route::RECORDS : Route::LINE_SCAN;
      c.tt.launches = 0;
      c.tt.flags |= UGX_TOT_SPAN_HANDOVER;
      TRY(line_scan_args(s, p, c.dbuf, n, false, base_offset, base_line, c.a));
      CU(cudaEventRecord(s->ev0, s->stream));
    }
  }
  TRY(run_route(c, r, pipelined));
  return end_scan(s, c.tt, totals, c.read);
}

// line records through the span kernels: the selected match starts of span_scan_kernel, then span_lines_kernel's count
// pass, one CTA for the bases and carries, and the emit pass.  *valid = false as for scan_spans.
int span_lines(ugx_scanner* s, const ugx_pattern* p, const uint8_t* dbuf, uint64_t n, uint32_t flags, uint64_t base_offset,
               uint64_t base_line, ugx_totals* tt, bool* valid)
{
  *valid = false;
  ugx::SpanArgs sa;
  TRY(span_count_pass(s, p, dbuf, n, true, base_offset, base_line, sa, tt));
  if (s->h_totals[ugx::SLOT_HANDOVER] != 0)
    return UGX_OK;
  const uint64_t nreg = ugx::stream_regions(n);
  TRY(s->lines_regions.ensure(5 * nreg + 8));
  ugx::SpanLinesArgs a{};
  a.reg_nl = s->lines_regions.p;
  a.reg_m = s->lines_regions.p + nreg;
  a.reg_bol = s->lines_regions.p + 2 * nreg;
  a.reg_fb = s->lines_regions.p + 3 * nreg;
  a.reg_fa = s->lines_regions.p + 4 * nreg;
  a.tail = s->lines_regions.p + 5 * nreg;
  a.sel_bits = s->span_sel.p;
  a.limit = sa.tail;
  a.base_offset = base_offset;
  a.base_line = base_line;
  a.invert = flags & UGX_LINES_INVERT;
  CU(ugx::launch_span_lines(p->dev, dbuf, n, a, false, s->sm_count, s->stream));
  CU(ugx::launch_span_lines_final(p->dev, dbuf, n, a, s->totals, s->stream));
  uint64_t nrec = 0;
  TRY(read_count(s, 2, s->lines, &nrec));
  tt->launches += 2;
  if (nrec > 0)
  {
    a.out = s->lines.p;
    a.out_cap = nrec;
    CU(ugx::launch_span_lines(p->dev, dbuf, n, a, true, s->sm_count, s->stream));
    tt->launches += 1;
  }
  s->lines_n = nrec;
  tt->matches = nrec;
  tt->newlines = s->h_totals[ugx::SLOT_NEWLINES];
  tt->flags |= UGX_TOT_NEWLINES;
  tt->kernel = UGX_K_SPAN_LINES;
  *valid = true;
  return UGX_OK;
}

// `-A` / `-B` / `-C`: the context stage over the selected line records in the line arena (context_lines.cu).  The
// caller fills a's buffer and file fields; the selected records are swapped out of the arena into s->ctx_sel, the
// count pass and the prefix over its block sums size the arena in one synchronise, and the emit pass writes every
// printed line to its final slot.  A batch (a.fsel != nullptr on entry: the host's selected-record ranges) gets every
// file's printed-line range in first_out[nfiles + 1], valid after the caller's next synchronise.
struct Context {
  uint32_t before, after;
};

int context_stage(ugx_scanner* s, const ugx_pattern* p, const Context& ctx, uint32_t flags, ugx::ContextArgs& a,
                  const uint64_t* fsel_host, const std::vector<uint64_t>& ftile_host, uint64_t* first_out, ugx_totals* tt)
{
  a.before = ctx.before;
  a.after = ctx.after;
  a.invert = flags & UGX_LINES_INVERT;
  const uint64_t nsel = s->lines_n;
  s->lines.swap(s->ctx_sel);
  s->lines_n = 0;
  const bool batch = fsel_host != nullptr;
  const uint64_t nf = batch ? a.nfiles + 1 : 0;
  if (nsel == 0)
  {
    if (batch)
      memset(first_out, 0, nf * sizeof(uint64_t));
    return UGX_OK;
  }
  const uint64_t nblk = ugx::context_blocks(nsel);
  TRY(s->ctx_pos.ensure(nsel + 2 * nblk + 3 * nf));
  a.sel = s->ctx_sel.p;
  a.nsel = nsel;
  a.pos = s->ctx_pos.p;
  a.blk = s->ctx_pos.p + nsel;
  if (batch)
  {
    uint64_t* d_fsel = a.blk + 2 * nblk;
    CU(cudaMemcpyAsync(d_fsel, fsel_host, nf * sizeof(uint64_t), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(d_fsel + nf, ftile_host.data(), nf * sizeof(uint64_t), cudaMemcpyHostToDevice, s->stream));
    a.fsel = d_fsel;
    a.ftile = d_fsel + nf;
    a.fout = d_fsel + 2 * nf;
  }
  CU(ugx::launch_context_count(a, s->stream));
  CU(ugx::launch_tile_prefix(a.blk, a.blk + nblk, nblk, s->totals, s->stream));
  uint64_t nout = 0;
  TRY(read_count(s, 1, s->lines, &nout));
  tt->launches += 2;
  a.out = s->lines.p;
  a.nout = nout;
  CU(ugx::launch_context_emit(a, s->sm_count, s->stream));
  tt->launches += 1;
  if (a.invert)
  {
    CU(ugx::launch_context_match(p->dev, a, s->sm_count, s->stream));
    tt->launches += 1;
  }
  if (batch)
    CU(cudaMemcpyAsync(first_out, a.fout, nf * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
  s->lines_n = nout;
  return UGX_OK;
}

// the line selection of ugx_find_lines: the span route where it applies, else (or after its hand-over) the line-at-a-time
// count pass, tile prefix and emit pass.  The records land in s->lines[0, s->lines_n); *tt receives their count, the
// newlines, the launches, the kernel and the hand-over flag.
int select_lines(ugx_scanner* s, const ugx_pattern* p, const uint8_t* dbuf, uint64_t n, uint32_t flags, uint64_t base_offset,
                 uint64_t base_line, ugx_totals* tt)
{
  int rc;
  if (span_route(s, p))
  {
    bool done = false;
    rc = span_lines(s, p, dbuf, n, flags, base_offset, base_line, tt, &done);
    if (rc != UGX_OK || done)
      return rc;
    tt->launches = 0; // the line-at-a-time kernels take over
    tt->flags |= UGX_TOT_SPAN_HANDOVER;
  }
  // the line-at-a-time kernels: a count pass into strip_counts, the tile prefix, an emit pass.  A pattern whose
  // prefilter admits no candidate searches no line (all lines are records of the inverted form).
  ugx::ScanArgs a;
  TRY(line_scan_args(s, p, dbuf, n, true, base_offset, base_line, a));
  const uint32_t lflags = flags | (p->never ? ugx::SCAN_LINES_NEVER : 0u);
  CU(ugx::launch_scan_line_records(p->dev, a, nullptr, lflags, false, s->sm_count, s->stream));
  CU(ugx::launch_tile_prefix(a.tile_matches, a.tile_newlines, a.ntiles, s->totals, s->stream));
  uint64_t nrec = 0;
  TRY(read_count(s, 2, s->lines, &nrec));
  tt->launches += 2;
  if (nrec > 0)
  {
    a.out_cap = nrec;
    CU(ugx::launch_scan_line_records(p->dev, a, s->lines.p, lflags, true, s->sm_count, s->stream));
    tt->launches += 1;
  }
  s->lines_n = nrec;
  tt->matches = nrec;
  tt->newlines = s->h_totals[ugx::SLOT_NEWLINES];
  tt->kernel = UGX_K_LINE_SCAN;
  return UGX_OK;
}

int find_lines_common(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t n, uint64_t base_offset,
                      uint64_t base_line, uint32_t flags, const ugx_line** dev_out, uint64_t* n_out, ugx_totals* totals,
                      const Context* ctx = nullptr)
{
  TRY(check_scan(ctx ? "ugx_find_context" : "ugx_find_lines", s, p, buf, n, flags));
  ugx_totals tt{};
  tt.flags = UGX_TOT_NEWLINES;
  set_records<ugx_line>(dev_out, n_out, nullptr, 0);
  if (n == 0)
    s->lines_n = 0;
  const uint8_t* dbuf;
  TRY(begin_scan(s, buf, n, tt, totals, &dbuf));
  if (dbuf == nullptr)
    return UGX_OK;
  TRY(select_lines(s, p, dbuf, n, flags, base_offset, base_line, &tt));
  if (ctx != nullptr)
  {
    ugx::ContextArgs a{};
    a.buf = dbuf;
    a.n = n;
    a.nl_total = tt.newlines;
    a.base_offset = base_offset;
    a.base_line = base_line;
    a.nfiles = 1;
    TRY(context_stage(s, p, *ctx, flags, a, nullptr, {}, nullptr, &tt));
  }
  TRY(end_scan(s, tt, totals));
  set_records(dev_out, n_out, s->lines.p, s->lines_n);
  return UGX_OK;
}

// ugx_find_lines / ugx_find_context: the records copied to out[cap]
int find_lines_to_host(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                       uint64_t base_line, uint32_t flags, ugx_line* out, uint64_t cap, uint64_t* n_out,
                       ugx_totals* totals, const Context* ctx)
{
  const ugx_line* dev = nullptr;
  uint64_t n = 0;
  TRY(find_lines_common(s, p, buf, nbytes, base_offset, base_line, flags, &dev, &n, totals, ctx));
  return copy_out(s, dev, sizeof(ugx_line), n, out, cap, n_out, false, "line record buffer too small");
}

// ugx_*_lines_bool: every check before any device work
int bool_check(const ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns, const ugx_bool_clause* clauses,
               uint32_t nclauses, const void* buf, uint64_t n, uint32_t flags)
{
  if (s == nullptr || patterns == nullptr || (buf == nullptr && n != 0) || (clauses == nullptr && nclauses != 0))
    return fail(UGX_E_INVALID, "null argument");
  if (npatterns == 0)
    return fail(UGX_E_INVALID, "ugx_lines_bool: no patterns");
  if (npatterns > UGX_BOOL_MAX_PATTERNS || nclauses > UGX_BOOL_MAX_CLAUSES)
    return fail(UGX_E_UNSUPPORTED, "ugx_lines_bool: more than 32 patterns or 64 clauses");
  for (uint32_t j = 0; j < npatterns; ++j)
  {
    TRY(check_scan("ugx_lines_bool", s, patterns[j], buf, n));
  }
  const uint32_t terms = npatterns == 32 ? ~0u : (1u << npatterns) - 1u;
  for (uint32_t c = 0; c < nclauses; ++c)
  {
    if ((clauses[c].pos | clauses[c].neg) == 0)
      return fail(UGX_E_INVALID, "ugx_lines_bool: an empty clause");
    if (((clauses[c].pos | clauses[c].neg) & ~terms) != 0)
      return fail(UGX_E_INVALID, "ugx_lines_bool: a clause names a pattern at or above npatterns");
  }
  if ((flags & ~UGX_LINES_INVERT) != 0)
    return fail(UGX_E_INVALID, "ugx_lines_bool: unknown flags");
  return UGX_OK;
}

// the clauses as the Boolean kernels take them, by value
ugx::BoolQuery bool_query(const ugx_bool_clause* clauses, uint32_t nclauses, uint32_t flags)
{
  ugx::BoolQuery q{};
  for (uint32_t c = 0; c < nclauses; ++c)
  {
    q.pos[c] = clauses[c].pos;
    q.neg[c] = clauses[c].neg;
  }
  q.nclauses = nclauses;
  q.invert = flags & UGX_LINES_INVERT;
  return q;
}

// Boolean line queries: every term's matching lines (select_lines, bases 0) marked into one term mask per line, then
// the clauses (bool_lines.cu).  want_records = false stops after the count (ugx_count_lines_bool).
int bool_common(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns, const ugx_bool_clause* clauses,
                uint32_t nclauses, const void* buf, uint64_t n, uint64_t base_offset, uint64_t base_line, uint32_t flags,
                bool want_records, const ugx_line** dev_out, uint64_t* n_out, ugx_totals* totals)
{
  TRY(bool_check(s, patterns, npatterns, clauses, nclauses, buf, n, flags));
  ugx_totals tt{};
  tt.flags = UGX_TOT_NEWLINES;
  tt.kernel = UGX_K_BOOL_LINES;
  set_records<ugx_line>(dev_out, n_out, nullptr, 0);
  s->lines_n = 0;
  const uint8_t* dbuf;
  TRY(begin_scan(s, buf, n, tt, totals, &dbuf));
  if (dbuf == nullptr)
    return UGX_OK;
  uint64_t nlines = 0;
  for (uint32_t j = 0; j < npatterns; ++j)
  {
    ugx_totals t{};
    TRY(select_lines(s, patterns[j], dbuf, n, 0, 0, 0, &t));
    tt.launches += t.launches;
    tt.flags |= t.flags & UGX_TOT_SPAN_HANDOVER;
    if (j == 0)
    {
      uint8_t last = 0;
      CU(cudaMemcpyAsync(&last, dbuf + n - 1, 1, cudaMemcpyDeviceToHost, s->stream));
      CU(cudaStreamSynchronize(s->stream));
      tt.newlines = t.newlines;
      nlines = t.newlines + (last != '\n' ? 1u : 0u);
      TRY(s->bool_mask.ensure(nlines));
      CU(cudaMemsetAsync(s->bool_mask.p, 0, nlines * sizeof(uint32_t), s->stream));
    }
    if (s->lines_n > 0)
    {
      CU(ugx::launch_bool_mark(s->lines.p, s->lines_n, s->bool_mask.p, 1u << j, s->sm_count, s->stream));
      tt.launches += 1;
    }
  }
  s->lines_n = 0;
  const ugx::BoolQuery q = bool_query(clauses, nclauses, flags);
  const uint64_t nlb = ugx::bool_line_blocks(nlines), nreg = want_records ? ugx::bool_regions(n) : 0;
  const uint64_t nblk = nlb > nreg ? nlb : nreg;
  // block values | line ends | the emit pass's one-file line table
  TRY(s->bool_pos.ensure(2 * nblk + (want_records ? nlines + 2 : 0)));
  ugx::BoolArgs a{};
  a.buf = dbuf;
  a.n = n;
  a.nfiles = 1;
  a.lb = s->bool_pos.p + 2 * nblk + nlines;
  a.nlines = nlines;
  a.mask = s->bool_mask.p;
  a.blk = s->bool_pos.p;
  a.nblocks = nblk;
  a.want_index = want_records ? 1u : 0u;
  a.eol = s->bool_pos.p + 2 * nblk;
  a.base_offset = base_offset;
  a.base_line = base_line;
  CU(ugx::launch_bool_count(a, q, s->stream));
  CU(ugx::launch_tile_prefix(a.blk, a.blk + nblk, nblk, s->totals, s->stream));
  TRY(read_totals(s, 1));
  tt.launches += 2;
  const uint64_t nsel = s->h_totals[ugx::SLOT_MATCHES];
  tt.matches = nsel;
  if (want_records && nsel > 0)
  {
    TRY(s->lines.ensure(nsel));
    a.out = s->lines.p;
    CU(ugx::launch_bool_index(a, s->stream));
    CU(ugx::launch_bool_batch_emit(a, q, s->stream));
    tt.launches += 2;
    s->lines_n = nsel;
  }
  TRY(end_scan(s, tt, totals));
  set_records(dev_out, n_out, s->lines.p, s->lines_n);
  return UGX_OK;
}

} // namespace

extern "C" {

int ugx_find_lines_device(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                          uint64_t base_line, uint32_t flags, const ugx_line** dev_out, uint64_t* n_out, ugx_totals* totals)
{
  return find_lines_common(s, p, buf, nbytes, base_offset, base_line, flags, dev_out, n_out, totals);
}

int ugx_find_lines(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                   uint64_t base_line, uint32_t flags, ugx_line* out, uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  return find_lines_to_host(s, p, buf, nbytes, base_offset, base_line, flags, out, cap, n_out, totals, nullptr);
}

int ugx_find_context_device(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                            uint64_t base_line, uint32_t flags, uint32_t before, uint32_t after, const ugx_line** dev_out,
                            uint64_t* n_out, ugx_totals* totals)
{
  const Context ctx{before, after};
  return find_lines_common(s, p, buf, nbytes, base_offset, base_line, flags, dev_out, n_out, totals, &ctx);
}

int ugx_find_context(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                     uint64_t base_line, uint32_t flags, uint32_t before, uint32_t after, ugx_line* out, uint64_t cap,
                     uint64_t* n_out, ugx_totals* totals)
{
  const Context ctx{before, after};
  return find_lines_to_host(s, p, buf, nbytes, base_offset, base_line, flags, out, cap, n_out, totals, &ctx);
}

int ugx_count_lines_bool(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns,
                         const ugx_bool_clause* clauses, uint32_t nclauses, const void* buf, uint64_t nbytes, uint32_t flags,
                         ugx_totals* totals)
{
  return bool_common(s, patterns, npatterns, clauses, nclauses, buf, nbytes, 0, 0, flags, false, nullptr, nullptr, totals);
}

int ugx_find_lines_bool_device(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns,
                               const ugx_bool_clause* clauses, uint32_t nclauses, const void* buf, uint64_t nbytes,
                               uint64_t base_offset, uint64_t base_line, uint32_t flags, const ugx_line** dev_out,
                               uint64_t* n_out, ugx_totals* totals)
{
  return bool_common(s, patterns, npatterns, clauses, nclauses, buf, nbytes, base_offset, base_line, flags, true, dev_out,
                     n_out, totals);
}

int ugx_find_lines_bool(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns,
                        const ugx_bool_clause* clauses, uint32_t nclauses, const void* buf, uint64_t nbytes,
                        uint64_t base_offset, uint64_t base_line, uint32_t flags, ugx_line* out, uint64_t cap,
                        uint64_t* n_out, ugx_totals* totals)
{
  const ugx_line* dev = nullptr;
  uint64_t n = 0;
  TRY(bool_common(s, patterns, npatterns, clauses, nclauses, buf, nbytes, base_offset, base_line, flags, true, &dev,
                       &n, totals));
  return copy_out(s, dev, sizeof(ugx_line), n, out, cap, n_out, false, "line record buffer too small");
}

int ugx_scanner_fetch_lines(ugx_scanner* s, ugx_line* out, uint64_t first, uint64_t count)
{
  if (s == nullptr || (out == nullptr && count != 0))
    return fail(UGX_E_INVALID, "null argument");
  return fetch(s, s->lines, s->lines_n, out, first, count, "record range outside the last line-record result");
}

int ugx_count_lines(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, ugx_totals* totals)
{
  return scan_common(s, p, buf, nbytes, 0, false, 0, 0, nullptr, nullptr, totals);
}

int ugx_count_matches(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, ugx_totals* totals)
{
  return scan_common(s, p, buf, nbytes, 1, false, 0, 0, nullptr, nullptr, totals);
}

int ugx_find_all_device(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                        uint64_t base_line, const ugx_match** dev_out, uint64_t* n_out, ugx_totals* totals)
{
  return scan_common(s, p, buf, nbytes, 1, true, base_offset, base_line, dev_out, n_out, totals);
}

int ugx_find_all(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, uint64_t base_offset,
                 uint64_t base_line, ugx_match* out, uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  const ugx_match* dev = nullptr;
  uint64_t n = 0;
  TRY(scan_common(s, p, buf, nbytes, 1, true, base_offset, base_line, &dev, &n, totals));
  return copy_out(s, dev, sizeof(ugx_match), n, out, cap, n_out, false, "record buffer too small");
}

const char* ugx_kernel_name(uint32_t id)
{
  switch (id)
  {
    case UGX_K_STREAM_LITERAL: return "count_lines_literal_kernel";
    case UGX_K_STREAM_DFA: return "count_lines_stream_kernel";
    case UGX_K_STREAM_SEARCH: return "count_lines_search_kernel";
    case UGX_K_TILE_ANY: return "count_lines_any_kernel";
    case UGX_K_LINE_SCAN: return "scan_lines_kernel";
    case UGX_K_RECORDS: return "scan_records_kernel";
    case UGX_K_NEWLINES: return "count_newlines_kernel";
    case UGX_K_MATCH_LINES: return "match_lines_kernel";
    case UGX_K_SPAN: return "span_scan_kernel";
    case UGX_K_BATCH: return "scan_batch_kernel";
    case UGX_K_SPAN_LINES: return "span_lines_kernel";
    case UGX_K_BOOL_LINES: return "bool_count_kernel";
    default: return "none";
  }
}

int ugx_scanner_set_option(ugx_scanner* s, const char* name, int value)
{
  if (s == nullptr || name == nullptr)
    return fail(UGX_E_INVALID, "null argument");
  // grids sized as if the device had min(value, SMs) SMs (0: all of them), so that a small buffer gives every warp the
  // many regions a multi-GiB buffer gives it on the whole device.  No scratch depends on it: the stream partials hold
  // STREAM_MAX_GRID CTAs whatever the grid, and the rest is sized by the buffer, its tiles, lines or records.
  if (strcmp(name, "grid_sms") == 0)
  {
    if (value < 0)
      return fail(UGX_E_INVALID, "scanner option grid_sms must be >= 0");
    s->sm_count = value == 0 || value > s->device_sms ? s->device_sms : value;
    return UGX_OK;
  }
  using Flag = bool ugx_scanner::*;
  static const struct {
    const char* name;
    Flag flag;
  } options[] = {
      {"force_generic", &ugx_scanner::force_generic}, {"legacy_any", &ugx_scanner::legacy_any},
      {"match_lines", &ugx_scanner::match_lines},     {"two_pass_records", &ugx_scanner::two_pass_records},
      {"no_pipeline", &ugx_scanner::no_pipeline},     {"stream_dfa", &ugx_scanner::stream_dfa},
      {"no_feeder", &ugx_scanner::no_feeder},         {"no_span", &ugx_scanner::no_span},
      {"no_cover", &ugx_scanner::no_cover},           {"no_search", &ugx_scanner::no_search},
      {"count_newlines", &ugx_scanner::count_newlines},
  };
  for (const auto& o : options)
    if (strcmp(name, o.name) == 0)
    {
      s->*o.flag = value != 0;
      return UGX_OK;
    }
  return fail(UGX_E_INVALID, std::string("unknown scanner option ") + name);
}

int ugx_scanner_fetch(ugx_scanner* s, ugx_match* out, uint64_t first, uint64_t count)
{
  if (s == nullptr || (out == nullptr && count != 0))
    return fail(UGX_E_INVALID, "null argument");
  return fetch(s, s->records, s->records_n, out, first, count, "record range outside the last result");
}

} // extern "C"

namespace {

// ---- many files in one launch (ugx_count_batch, ugx_find_all_batch, ugx_find_lines_batch) ----
// The files lie in one buffer, file f at buf[begins[f], begins[f] + lens[f]); tile g of a launch is tile ti[g] of file
// tf[g], so the tiles are ordered by file and then by offset.
struct Batch {
  uint64_t nfiles = 0;
  std::vector<uint32_t> tf, ti;
  const uint8_t* dbuf = nullptr;
  ugx::BatchArgs a;
};

// the checks of the file table every batch entry point makes, and the tile table; `who` names the entry point
int batch_tiles(const char* who, uint64_t nbytes, const uint64_t* begins, const uint64_t* lens, uint64_t nfiles, Batch& b)
{
  b.nfiles = nfiles;
  for (uint64_t f = 0; f < nfiles; ++f)
  {
    if ((begins[f] & 15) != 0 || begins[f] > nbytes || lens[f] > nbytes - begins[f])
      return fail(UGX_E_INVALID, std::string(who) + ": file " + std::to_string(f) + " is not a 16-byte aligned range of the buffer");
    if (nfiles > 0xffffffffull || lens[f] / ugx::SCAN_TILE > 0xfffffffeull)
      return fail(UGX_E_INVALID, std::string(who) + ": too many files / a file too large for one batch");
    const uint64_t nt = (lens[f] + ugx::SCAN_TILE - 1) / ugx::SCAN_TILE;
    for (uint64_t j = 0; j < nt; ++j)
    {
      b.tf.push_back(static_cast<uint32_t>(f));
      b.ti.push_back(static_cast<uint32_t>(j));
    }
  }
  return UGX_OK;
}

// begin_scan's setup for a batch: the file and tile tables uploaded and the per-file counters zeroed, all on the
// scanner's stream: b.a is ready for a launch
int batch_upload(ugx_scanner* s, const uint64_t* begins, const uint64_t* lens, uint64_t nfiles, Batch& b)
{
  // one scratch block: begins | lens | counts | tile_file | tile_index
  const uint64_t words = 3 * nfiles + (b.tf.size() + 1) / 2 * 2;
  TRY(s->batch.ensure(words + 4));
  uint64_t* d_begins = s->batch.p;
  uint64_t* d_lens = d_begins + nfiles;
  unsigned long long* d_counts = reinterpret_cast<unsigned long long*>(d_lens + nfiles);
  uint32_t* d_tf = reinterpret_cast<uint32_t*>(d_counts + nfiles);
  uint32_t* d_ti = d_tf + b.tf.size();
  CU(cudaMemcpyAsync(d_begins, begins, nfiles * 8, cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemcpyAsync(d_lens, lens, nfiles * 8, cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemsetAsync(d_counts, 0, nfiles * 8, s->stream));
  CU(cudaMemcpyAsync(d_tf, b.tf.data(), b.tf.size() * 4, cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemcpyAsync(d_ti, b.ti.data(), b.ti.size() * 4, cudaMemcpyHostToDevice, s->stream));
  b.a.begins = d_begins;
  b.a.lens = d_lens;
  b.a.tile_file = d_tf;
  b.a.tile_index = d_ti;
  b.a.ntiles = b.tf.size();
  b.a.counts = d_counts;
  b.a.stage_table = 0;
  return UGX_OK;
}

// the start of a batch's records (batch_records, bool_batch), inside `guarded`: the tile table (b), the arena's last
// result dropped, per_file[nper] zeroed, and begin_scan with the file and tile tables uploaded and the tile scratch
// sized; `extra` sizes the caller's own scratch.  b.dbuf stays nullptr when every file is empty: nothing to scan.
template <typename Extra = int (&)()>
int begin_batch(ugx_scanner* s, const char* who, const void* buf, uint64_t nbytes, const uint64_t* begins,
                const uint64_t* lens, uint64_t nfiles, uint64_t& arena_n, uint64_t* per_file, uint64_t nper,
                const ugx_totals& tt, Batch& b, Extra&& extra = no_setup)
{
  TRY(batch_tiles(who, nbytes, begins, lens, nfiles, b));
  // the arena is rewritten by the caller: its last result is gone from here on
  arena_n = 0;
  memset(per_file, 0, nper * sizeof(uint64_t));
  if (b.tf.empty())
    return UGX_OK;
  const uint64_t ntiles = b.tf.size();
  return begin_scan(s, buf, nbytes, tt, nullptr, &b.dbuf, [&]() -> int {
    TRY(batch_upload(s, begins, lens, nfiles, b));
    TRY(ensure_tiles(s, ntiles));
    TRY(s->strip_counts.ensure(ntiles * ugx::SCAN_THREADS));
    return extra();
  });
}

// the selection of a batch, match records (lines == false) or line records: the count pass, the tile prefix, then the
// per-file counts and the totals to the host in the one synchronise that sizes the arena (`before_sync` enqueues
// whatever else the caller reads there), and the emit pass into the scanner's match or line arena.  The batch is
// uploaded (batch_upload, b.a.counts zero) and the tile scratch sized.  sfirst[nfiles + 1] receives every file's record
// range; *tt the records, the newlines and the launches.  Afterwards tile_matches / tile_newlines hold the exclusive
// record and newline prefix of the batch tiles.
template <typename BeforeSync = int (&)()>
int select_lines_batch(ugx_scanner* s, const ugx_pattern* p, const Batch& b, bool lines, uint32_t flags, const char* who,
                       uint64_t* sfirst, ugx_totals* tt, BeforeSync&& before_sync = no_setup)
{
  const uint64_t nfiles = b.nfiles, ntiles = b.tf.size();
  ugx::BatchRecordArgs r;
  r.tile_matches = s->tile_matches.p;
  r.tile_newlines = s->tile_newlines.p;
  r.strip_counts = s->strip_counts.p;
  r.out = nullptr;
  r.lout = nullptr;
  r.out_cap = 0;
  // a prefilter that admits no candidate (config 3) searches no line: no match records, and the inverted line
  // records are every line
  r.lflags = flags | (p->never ? ugx::SCAN_LINES_NEVER : 0u);
  CU(ugx::launch_scan_batch_records(p->dev, b.dbuf, b.a, r, lines, false, s->sm_count, s->stream));
  CU(ugx::launch_tile_prefix(s->tile_matches.p, s->tile_newlines.p, ntiles, s->totals, s->stream));
  CU(cudaMemcpyAsync(s->h_totals, s->totals, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
  CU(cudaMemcpyAsync(sfirst + 1, b.a.counts, nfiles * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
  TRY(before_sync());
  CU(cudaStreamSynchronize(s->stream));
  tt->launches += 2;
  const uint64_t nrec = s->h_totals[ugx::SLOT_MATCHES];
  sfirst[0] = 0;
  for (uint64_t f = 0; f < nfiles; ++f)
    sfirst[f + 1] += sfirst[f];
  if (sfirst[nfiles] != nrec)
    return fail(UGX_E_CUDA, std::string(who) + ": per-file record counts disagree with the total");
  TRY(lines ? s->lines.ensure(nrec) : s->records.ensure(nrec));
  if (nrec > 0)
  {
    r.out = lines ? nullptr : s->records.p;
    r.lout = lines ? s->lines.p : nullptr;
    r.out_cap = nrec;
    CU(ugx::launch_scan_batch_records(p->dev, b.dbuf, b.a, r, lines, true, s->sm_count, s->stream));
    tt->launches += 1;
  }
  (lines ? s->lines_n : s->records_n) = nrec;
  tt->matches = nrec;
  tt->newlines = s->h_totals[ugx::SLOT_NEWLINES];
  return UGX_OK;
}

// match records (lines == false) or line records of a batch: select_lines_batch, and with ctx the context stage.
// first[nfiles + 1] receives every file's record range, *n_out the number of records, out[cap] the records (out ==
// NULL with cap == 0: they stay on the device).
int batch_records(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, const uint64_t* begins,
                  const uint64_t* lens, uint64_t nfiles, bool lines, uint32_t flags, uint64_t* first, void* out, uint64_t cap,
                  uint64_t* n_out, ugx_totals* totals, const Context* ctx = nullptr)
{
  if (n_out)
    *n_out = 0;
  const char* who = ctx ? "ugx_find_context_batch" : lines ? "ugx_find_lines_batch" : "ugx_find_all_batch";
  if (s == nullptr || p == nullptr || (buf == nullptr && nbytes != 0) ||
      (nfiles != 0 && (begins == nullptr || lens == nullptr || first == nullptr)))
    return fail(UGX_E_INVALID, std::string(who) + ": bad argument");
  TRY(check_scan(who, s, p, buf, nbytes, flags));
  ugx_totals tt{};
  tt.flags = UGX_TOT_NEWLINES;
  if (totals)
    *totals = tt;
  if (first != nullptr)
    first[0] = 0;
  uint64_t& arena_n = lines ? s->lines_n : s->records_n;
  if (nfiles == 0)
  {
    arena_n = 0;
    return UGX_OK;
  }
  return guarded(UGX_E_NOMEM, nullptr, [&]() -> int {
    Batch b;
    TRY(begin_batch(s, who, buf, nbytes, begins, lens, nfiles, arena_n, first, nfiles + 1, tt, b));
    if (b.dbuf == nullptr)
      return UGX_OK; // only empty files: no lines, no records
    // with context, first[] receives the printed lines' ranges and the selected records' ranges go to sfirst
    std::vector<uint64_t> ctx_first;
    uint64_t* sfirst = first;
    if (ctx != nullptr)
    {
      ctx_first.assign(nfiles + 1, 0);
      sfirst = ctx_first.data();
    }
    TRY(select_lines_batch(s, p, b, lines, flags, who, sfirst, &tt));
    const uint64_t nrec = tt.matches, nl_total = tt.newlines;
    if (ctx != nullptr)
    {
      // every file's first batch tile: the tiles are ordered by file
      std::vector<uint64_t> ftile(nfiles + 1, 0);
      for (uint64_t f = 0; f < nfiles; ++f)
        ftile[f + 1] = ftile[f] + (lens[f] + ugx::SCAN_TILE - 1) / ugx::SCAN_TILE;
      ugx::ContextArgs c{};
      c.buf = b.dbuf;
      c.nl_total = nl_total;
      c.nfiles = nfiles;
      c.begins = b.a.begins;
      c.lens = b.a.lens;
      c.tile_nl = s->tile_newlines.p;
      c.ntiles = b.tf.size();
      TRY(context_stage(s, p, *ctx, flags, c, sfirst, ftile, first, &tt));
    }
    tt.matches = nrec;
    tt.newlines = nl_total;
    tt.kernel = UGX_K_BATCH;
    TRY(end_scan(s, tt, totals));
    return lines ? copy_out(s, s->lines.p, sizeof(ugx_line), arena_n, out, cap, n_out, true, "record buffer too small")
                 : copy_out(s, s->records.p, sizeof(ugx_match), arena_n, out, cap, n_out, true, "record buffer too small");
  });
}

// Boolean line queries over a batch: every term's batch selection (select_lines_batch, flags 0) marked into one term
// mask per line of the batch, the lines numbered across the files from the first term's newline prefix, then the
// clauses (bool_lines.cu).  want_records = false stops after the count: counts[nfiles] (ugx_count_lines_bool_batch);
// otherwise first[nfiles + 1] and the records as in ugx_find_lines_batch.
int bool_batch(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns, const ugx_bool_clause* clauses,
               uint32_t nclauses, const void* buf, uint64_t nbytes, const uint64_t* begins, const uint64_t* lens,
               uint64_t nfiles, uint32_t flags, bool want_records, uint64_t* counts, uint64_t* first, ugx_line* out,
               uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  const char* who = want_records ? "ugx_find_lines_bool_batch" : "ugx_count_lines_bool_batch";
  if (n_out)
    *n_out = 0;
  TRY(bool_check(s, patterns, npatterns, clauses, nclauses, buf, nbytes, flags));
  // the per-file result: counts[nfiles], or first[nfiles + 1] with the records
  uint64_t* per_file = want_records ? first : counts;
  const uint64_t at = want_records ? 1 : 0;
  if (nfiles != 0 && (begins == nullptr || lens == nullptr || per_file == nullptr))
    return fail(UGX_E_INVALID, std::string(who) + ": bad argument");
  ugx_totals tt{};
  tt.flags = UGX_TOT_NEWLINES;
  tt.kernel = UGX_K_BOOL_LINES;
  if (totals)
    *totals = tt;
  if (want_records && first != nullptr)
    first[0] = 0;
  if (nfiles == 0)
  {
    s->lines_n = 0;
    return UGX_OK;
  }
  return guarded(UGX_E_NOMEM, nullptr, [&]() -> int {
    Batch b;
    const uint64_t nf1 = nfiles + 1;
    TRY(begin_batch(s, who, buf, nbytes, begins, lens, nfiles, s->lines_n, per_file, nfiles + at, tt, b,
                    [&] { return s->bool_files.ensure(3 * nf1); }));
    if (b.dbuf == nullptr)
      return UGX_OK; // only empty files: no lines
    // every file's lines, then lb[] (its first global line, lb[nfiles] = the batch's lines); its newlines; its
    // selected lines
    uint64_t* lb = s->bool_files.p;
    uint64_t* fnl = lb + nf1;
    unsigned long long* fsel = reinterpret_cast<unsigned long long*>(fnl + nf1);
    std::vector<uint64_t> term_first(nf1);
    uint64_t nlines = 0;
    for (uint32_t j = 0; j < npatterns; ++j)
    {
      if (j > 0)
        CU(cudaMemsetAsync(b.a.counts, 0, nfiles * sizeof(uint64_t), s->stream));
      ugx_totals t{};
      TRY(select_lines_batch(s, patterns[j], b, true, 0, who, term_first.data(), &t, [&]() -> int {
        if (j > 0)
          return UGX_OK;
        // the line table from this term's newline prefix, read in the synchronise that sizes its arena
        CU(cudaMemsetAsync(lb, 0, 2 * nf1 * sizeof(uint64_t), s->stream));
        CU(ugx::launch_bool_batch_lines(b.dbuf, b.a, s->tile_newlines.p, s->totals + ugx::SLOT_NEWLINES, lb, fnl,
                                        s->stream));
        CU(ugx::launch_tile_prefix(lb, fnl, nf1, s->totals + ugx::SLOT_BATCH_LINES, s->stream));
        CU(cudaMemcpyAsync(s->h_totals + ugx::SLOT_BATCH_LINES, s->totals + ugx::SLOT_BATCH_LINES,
                           2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        return UGX_OK;
      }));
      tt.launches += t.launches;
      if (j == 0)
      {
        tt.launches += 2;
        tt.newlines = t.newlines;
        nlines = s->h_totals[ugx::SLOT_BATCH_LINES];
        TRY(s->bool_mask.ensure(nlines));
        CU(cudaMemsetAsync(s->bool_mask.p, 0, nlines * sizeof(uint32_t), s->stream));
      }
      if (s->lines_n > 0)
      {
        CU(ugx::launch_bool_batch_mark(s->lines.p, s->lines_n, s->tile_matches.p, b.a, lb, s->bool_mask.p, 1u << j,
                                       s->sm_count, s->stream));
        tt.launches += 1;
      }
    }
    s->lines_n = 0;
    const ugx::BoolQuery q = bool_query(clauses, nclauses, flags);
    const uint64_t nlb = ugx::bool_line_blocks(nlines);
    TRY(s->bool_pos.ensure(2 * nlb + (want_records ? nlines : 0)));
    CU(cudaMemsetAsync(fsel, 0, nfiles * sizeof(unsigned long long), s->stream));
    ugx::BoolArgs a{};
    a.buf = b.dbuf;
    a.files = b.a;
    a.nfiles = nfiles;
    a.lb = lb;
    a.nlines = nlines;
    a.mask = s->bool_mask.p;
    a.fsel = fsel;
    a.blk = s->bool_pos.p;
    a.nblocks = nlb;
    a.tile_nl = s->tile_newlines.p;
    a.eol = s->bool_pos.p + 2 * nlb;
    CU(ugx::launch_bool_batch_count(a, q, s->stream));
    CU(ugx::launch_tile_prefix(a.blk, a.blk + nlb, nlb, s->totals, s->stream));
    CU(cudaMemcpyAsync(per_file + at, fsel, nfiles * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
    TRY(read_totals(s, 1));
    tt.launches += 2;
    const uint64_t nsel = s->h_totals[ugx::SLOT_MATCHES];
    tt.matches = nsel;
    if (want_records)
    {
      for (uint64_t f = 0; f < nfiles; ++f)
        first[f + 1] += first[f];
      if (first[nfiles] != nsel)
        return fail(UGX_E_CUDA, std::string(who) + ": per-file line counts disagree with the total");
      if (nsel > 0)
      {
        TRY(s->lines.ensure(nsel));
        a.out = s->lines.p;
        CU(ugx::launch_bool_batch_index(a, s->stream));
        CU(ugx::launch_bool_batch_emit(a, q, s->stream));
        tt.launches += 2;
        s->lines_n = nsel;
      }
    }
    TRY(end_scan(s, tt, totals));
    return want_records ? copy_out(s, s->lines.p, sizeof(ugx_line), s->lines_n, out, cap, n_out, true,
                                   "record buffer too small")
                        : UGX_OK;
  });
}

} // namespace

extern "C" {

int ugx_count_batch(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, const uint64_t* begins,
                    const uint64_t* lens, uint64_t nfiles, int mode, uint64_t* counts, ugx_totals* totals)
{
  if (s == nullptr || p == nullptr || (buf == nullptr && nbytes != 0) || (nfiles != 0 && (begins == nullptr || lens == nullptr || counts == nullptr)) ||
      (mode != UGX_MODE_LINES && mode != UGX_MODE_MATCHES))
    return fail(UGX_E_INVALID, "ugx_count_batch: bad argument");
  TRY(check_scan("ugx_count_batch", s, p, buf, nbytes));
  ugx_totals tt{};
  if (totals)
    *totals = tt;
  if (nfiles == 0)
    return UGX_OK;
  return guarded(UGX_E_NOMEM, nullptr, [&]() -> int {
    Batch b;
    TRY(batch_tiles("ugx_count_batch", nbytes, begins, lens, nfiles, b));
    memset(counts, 0, nfiles * sizeof(uint64_t));
    if (b.tf.empty() || p->never)
      return UGX_OK; // only empty files, or a prefilter that admits no candidate (config 3): nothing matches
    TRY(begin_scan(s, buf, nbytes, tt, nullptr, &b.dbuf, [&] { return batch_upload(s, begins, lens, nfiles, b); }));
    CU(ugx::launch_scan_batch(p->dev, b.dbuf, b.a, mode, s->sm_count, s->stream));
    CU(cudaEventRecord(s->ev1, s->stream)); // the counts' copy is not kernel time
    CU(cudaMemcpyAsync(counts, b.a.counts, nfiles * 8, cudaMemcpyDeviceToHost, s->stream));
    TRY(end_scan(s, tt, nullptr, 0, true));
    for (uint64_t f = 0; f < nfiles; ++f)
      tt.matches += counts[f];
    tt.launches = 1;
    tt.kernel = UGX_K_BATCH;
    if (totals)
      *totals = tt;
    return UGX_OK;
  });
}

int ugx_find_all_batch(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, const uint64_t* begins,
                       const uint64_t* lens, uint64_t nfiles, uint64_t* first, ugx_match* out, uint64_t cap,
                       uint64_t* n_out, ugx_totals* totals)
{
  return batch_records(s, p, buf, nbytes, begins, lens, nfiles, false, 0, first, out, cap, n_out, totals);
}

int ugx_find_lines_batch(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, const uint64_t* begins,
                         const uint64_t* lens, uint64_t nfiles, uint32_t flags, uint64_t* first, ugx_line* out,
                         uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  return batch_records(s, p, buf, nbytes, begins, lens, nfiles, true, flags, first, out, cap, n_out, totals);
}

int ugx_find_context_batch(ugx_scanner* s, const ugx_pattern* p, const void* buf, uint64_t nbytes, const uint64_t* begins,
                           const uint64_t* lens, uint64_t nfiles, uint32_t flags, uint32_t before, uint32_t after,
                           uint64_t* first, ugx_line* out, uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  const Context ctx{before, after};
  return batch_records(s, p, buf, nbytes, begins, lens, nfiles, true, flags, first, out, cap, n_out, totals, &ctx);
}

int ugx_count_lines_bool_batch(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns,
                               const ugx_bool_clause* clauses, uint32_t nclauses, const void* buf, uint64_t nbytes,
                               const uint64_t* begins, const uint64_t* lens, uint64_t nfiles, uint32_t flags,
                               uint64_t* counts, ugx_totals* totals)
{
  return bool_batch(s, patterns, npatterns, clauses, nclauses, buf, nbytes, begins, lens, nfiles, flags, false, counts,
                    nullptr, nullptr, 0, nullptr, totals);
}

int ugx_find_lines_bool_batch(ugx_scanner* s, const ugx_pattern* const* patterns, uint32_t npatterns,
                              const ugx_bool_clause* clauses, uint32_t nclauses, const void* buf, uint64_t nbytes,
                              const uint64_t* begins, const uint64_t* lens, uint64_t nfiles, uint32_t flags,
                              uint64_t* first, ugx_line* out, uint64_t cap, uint64_t* n_out, ugx_totals* totals)
{
  return bool_batch(s, patterns, npatterns, clauses, nclauses, buf, nbytes, begins, lens, nfiles, flags, true, nullptr,
                    first, out, cap, n_out, totals);
}

int ugx_check_text(ugx_scanner* s, const void* buf, uint64_t nbytes, ugx_text_info* out)
{
  if (s == nullptr || out == nullptr || (buf == nullptr && nbytes != 0))
    return fail(UGX_E_INVALID, "null argument");
  memset(out, 0, sizeof(*out));
  out->is_utf8 = 1;
  ugx_totals tt{};
  const uint8_t* dbuf;
  unsigned long long* dflags = s->totals + ugx::SLOT_UTF8;
  TRY(begin_scan(s, buf, nbytes, tt, nullptr, &dbuf, [&]() -> int {
    CU(cudaMemsetAsync(dflags, 0, sizeof(unsigned long long), s->stream));
    return UGX_OK;
  }));
  if (dbuf == nullptr)
    return UGX_OK;
  CU(ugx::launch_utf8_check(dbuf, nbytes, reinterpret_cast<unsigned int*>(dflags), s->sm_count, s->stream));
  CU(cudaMemcpyAsync(s->h_totals + ugx::SLOT_UTF8, dflags, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
  TRY(end_scan(s, tt, nullptr));
  const unsigned int f = static_cast<unsigned int>(s->h_totals[ugx::SLOT_UTF8]);
  out->is_utf8 = (f & 1u) == 0;
  out->has_nul = (f & 2u) != 0;
  out->kernel_ms = tt.kernel_ms;
  out->launches = 1;
  return UGX_OK;
}

int ugx_count_newlines(ugx_scanner* s, const void* buf, uint64_t nbytes, ugx_totals* totals)
{
  if (s == nullptr || (buf == nullptr && nbytes != 0))
    return fail(UGX_E_INVALID, "null argument");
  ugx_totals tt{};
  tt.flags = UGX_TOT_NEWLINES;
  const uint8_t* dbuf;
  TRY(begin_scan(s, buf, nbytes, tt, totals, &dbuf));
  if (dbuf == nullptr)
    return UGX_OK;
  TRY(newline_pass(s, dbuf, nbytes, tt));
  return end_scan(s, tt, totals, READ_NEWLINES);
}

} // extern "C"
