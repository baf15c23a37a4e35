// device_pattern.cuh — the compiled pattern as the kernels see it, and the per-position
// building blocks shared by every scan kernel: predictors, candidate predicates, the dense
// DFA step and the META-aware opcode interpreter.
//
// Reference semantics restated here (paths into /root/reference):
//   predict_match PM4 / PMH     include/reflex/pattern.h:366-401, hashes :1274-1282
//   advance_* candidate tests   lib/matcher.cpp:957-3549 (position-local form, DESIGN.md)
//   DFA interpreter             lib/matcher.cpp:94-546
//   word-boundary predicates    include/reflex/matcher.h:1194-1319
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/ugrep_b200.h"
#include "filter_plan.hpp"
#include "ptx.cuh"

namespace ugx {

constexpr uint32_t D_OP_HALT = 0x00FFFFFFu;
constexpr uint32_t D_IDX_HALT = 0xFFFFu;
constexpr uint32_t D_IDX_LONG = 0xFFFEu;
constexpr uint32_t D_NONE = 0xFFFFFFFFu;
constexpr uint32_t D_DEAD = 0xFFFFu;
constexpr int D_EOF = -1;

struct DevPattern {
  uint32_t adv, len, min, pin, lcp, lcs, one, bol, lbk, lbm, flags;
  uint32_t nstates, ncls, has_meta, to_start, nop, n_word_ranges, table_bytes;
  uint32_t first_acc, first_leaf, acc0; // state numbering (pattern_host.hpp); acc0: the start state accepts
  uint32_t covers;         // proven at upload: every match start passes cand() (pattern_host.hpp prefilter_covers_matches)
  uint32_t pin_a[8], pin_b[8], cbk[8], fst[8]; // 256-bit sets
  uint8_t chr[256];
  const uint8_t* cls;      // [256] byte -> class
  const uint16_t* next;    // [nstates * ncls]
  const uint32_t* accept;  // [nstates]
  const uint32_t* opc;     // [nop + 2] opcode words (META interpreter only)
  const uint8_t* pred;     // [4096] pma_ when min < 4, else pmh_
  const uint8_t* tap;      // [2048]
  const int* word_ranges;  // [2 * n_word_ranges]
  FilterPlan plan;         // first-stage filter of the position-parallel kernels
  // k-gram viability of an anchored attempt (pattern_host.hpp Viability; span_scan.cu)
  uint32_t via_k, via_stride, via_words, via_pair_bytes;
  uint32_t via_bytes;        // via_bits holds one BYTE per entry (small tables: one lookup, no shift / mask per position)
  const uint32_t* via_ids;   // [512] t01 / t23 interleaved: one 64-bit lookup per text byte
  const uint32_t* via_bits;  // [via_words] (a multiple of 4 words)
  const uint8_t* via_pair;   // [via_pair_bytes] (a multiple of 16 bytes)
  // line-resetting search automaton of `-c` (pattern_host.hpp SearchDfa, stream_search.cu); search_ok = 0: not built
  uint32_t search_ok, search_depth, search_ncls, search_bytes; // search_bytes: the table, padded to 16 bytes
  const uint8_t* search_cls;    // [256]
  const uint16_t* search_next;  // [search_bytes / 2] pre-multiplied row offsets, MATCHED = 0
};

// the tables a kernel actually reads (shared-memory copies when staged, else the global ones)
struct Tables {
  const uint8_t* cls;
  const uint16_t* next;
  const uint8_t* pred;
  const uint8_t* tap;
};

// one DFA transition with the lookups by shared-space address (LDS with a 32-bit address and the pattern's constants in
// registers; through the generic pointers of Tables the same transition compiles to LD.E with 64-bit address arithmetic
// and re-reads of the parameter bank — three times the instructions).  The class map is always staged; the table is
// read from global memory when it does not fit (next_s == 0).
struct Stepper {
  uint32_t cls_s, next_s, ncls;
  const uint16_t* gnext;
  __device__ __forceinline__ Stepper(const Tables& T, uint32_t ncls_, bool staged)
      : cls_s(smem_u32(T.cls)), next_s(staged ? smem_u32(T.next) : 0u), ncls(ncls_), gnext(T.next)
  {
    // opaque to the compiler, which otherwise rebuilds the shared-window addresses from special registers per use
    asm volatile("" : "+r"(cls_s), "+r"(next_s), "+r"(ncls));
  }
  __device__ __forceinline__ uint32_t operator()(uint32_t state, uint32_t ch) const
  {
    const uint32_t idx = state * ncls + lds_u8(cls_s + ch);
    return next_s != 0 ? lds_u16(next_s + 2 * idx) : static_cast<uint32_t>(__ldg(gnext + idx));
  }
  // the same with the table's place known at compile time (no branch per transition)
  template <bool STAGED>
  __device__ __forceinline__ uint32_t at(uint32_t state, uint32_t ch) const
  {
    const uint32_t idx = state * ncls + lds_u8(cls_s + ch);
    return STAGED ? lds_u16(next_s + 2 * idx) : static_cast<uint32_t>(__ldg(gnext + idx));
  }
};

__device__ __forceinline__ bool bit256(const uint32_t* set, uint32_t c) { return (set[c >> 5] >> (c & 31)) & 1u; }
__device__ __forceinline__ uint32_t hash3(uint32_t h, uint32_t b) { return ((h << 3) ^ b) & (UGX_HASH - 1); }
__device__ __forceinline__ uint32_t bihash(uint32_t a, uint32_t b) { return (a ^ (b << 6)) & (UGX_BTAP - 1); }

// ---- text access: one buffer in global memory; reads past the end see the caller's NUL slot ----
struct Text {
  const uint8_t* __restrict__ b;
  uint64_t end;
  __device__ __forceinline__ uint32_t at(uint64_t i) const { return i < end ? __ldg(b + i) : 0u; }
  __device__ __forceinline__ uint32_t raw(uint64_t i) const { return __ldg(b + i); }
};

__device__ __forceinline__ bool pm4(const Text& t, const uint8_t* pma, uint64_t k)
{
  uint32_t c0 = t.at(k), c1 = t.at(k + 1), c2 = t.at(k + 2), c3 = t.at(k + 3);
  uint32_t h1 = hash3(c0, c1), h2 = hash3(h1, c2), h3 = hash3(h2, c3);
  uint32_t q = (pma[c0] & 0xc0u) | (pma[h1] & 0x30u) | (pma[h2] & 0x0cu) | (pma[h3] & 0x03u);
  uint32_t r = ((((((q >> 2) | q) >> 2) | q) >> 1) | q) & 0xffu;
  return r != 0xffu;
}

__device__ __forceinline__ bool pmh(const Text& t, const uint8_t* tab, uint64_t k, uint32_t n)
{
  uint32_t h = t.at(k);
  uint32_t f = tab[h] & 1u;
  uint32_t bit = 2;
  for (uint32_t j = 1; j < n; ++j, bit <<= 1)
  {
    h = hash3(h, t.at(k + j));
    f |= tab[h] & bit;
    if (j == 3 && f != 0)
      return false;
  }
  return f == 0;
}

__device__ __forceinline__ uint32_t tapbit(const Text& t, const uint8_t* tap, uint64_t k, uint32_t j)
{
  return (tap[bihash(t.at(k), t.at(k + 1))] >> j) & 1u;
}

__device__ __forceinline__ bool literal_at(const Text& t, const DevPattern& P, uint64_t k)
{
  if (k + P.len > t.end)
    return false;
  for (uint32_t i = 0; i < P.len; ++i)
    if (t.raw(k + i) != P.chr[i])
      return false;
  return true;
}

// cand(k): can the reference's advance routine stop at byte k?  One case per routine family.
__device__ __forceinline__ bool cand(const Text& t, const DevPattern& P, const Tables& T, uint64_t k)
{
  const uint64_t end = t.end;
  const uint32_t min = P.min, len = P.len, lcp = P.lcp, lcs = P.lcs;
  switch (P.adv)
  {
    case UGX_ADV_PIN1_ONE:
      return t.raw(k) == P.chr[0] && (k + 4 > end || pm4(t, T.pred, k));
    case UGX_ADV_PIN1_PMA:
      if (k + lcp >= end || t.raw(k + lcp) != P.chr[0])
        return false;
      return k + 4 > end || (t.at(k + lcs) == P.chr[1] && pm4(t, T.pred, k));
    case UGX_ADV_PIN1_PMH:
      if (k + lcp >= end || t.raw(k + lcp) != P.chr[0])
        return false;
      return k + min > end || (t.at(k + lcs) == P.chr[1] && pmh(t, T.pred, k, min));
    case UGX_ADV_PIN_ONE:
      if (k + 4 > end)
        return true;
      return bit256(P.pin_a, t.raw(k)) && pm4(t, T.pred, k);
    case UGX_ADV_PIN_PMA:
      if (k + min > end)
        return false;
      if (k + 4 > end)
        return true;
      return bit256(P.pin_a, t.raw(k + lcp)) && bit256(P.pin_b, t.raw(k + lcs)) && pm4(t, T.pred, k);
    case UGX_ADV_PIN_PMH:
      if (k + min > end)
        return false;
      return bit256(P.pin_a, t.raw(k + lcp)) && bit256(P.pin_b, t.raw(k + lcs)) && pmh(t, T.pred, k, min);
    case UGX_ADV_MIN1:
      if (tapbit(t, T.tap, k, 0))
        return false;
      return k + 4 >= end || pm4(t, T.pred, k);
    case UGX_ADV_MIN2:
      if (k + 2 > end)
        return false;
      if (tapbit(t, T.tap, k, 0) || tapbit(t, T.tap, k + 1, 1))
        return false;
      return k + 5 > end || pm4(t, T.pred, k);
    case UGX_ADV_MIN3:
      if (k + 3 > end)
        return false;
      if (tapbit(t, T.tap, k, 0) || tapbit(t, T.tap, k + 1, 1) || tapbit(t, T.tap, k + 2, 2))
        return false;
      return k + 5 > end || pm4(t, T.pred, k);
    case UGX_ADV_MIN4:
      if (k + min > end)
        return false;
      for (uint32_t j = 0; j < min; ++j)
        if (tapbit(t, T.tap, k + j, j))
          return false;
      return pmh(t, T.pred, k, min);
    case UGX_ADV_PMA:
      if (k + 7 <= end)
        return pm4(t, T.pred, k);
      if (tapbit(t, T.tap, k, 0))
        return false;
      return k + 4 >= end || pm4(t, T.pred, k);
    case UGX_ADV_CHAR:
      return t.raw(k) == P.chr[0];
    case UGX_ADV_CHAR_PMA:
      return t.raw(k) == P.chr[0] && (k + 5 > end || pm4(t, T.pred, k + 1));
    case UGX_ADV_CHAR_PMH:
      return t.raw(k) == P.chr[0] && (k + 1 + min > end || pmh(t, T.pred, k + 1, min));
    case UGX_ADV_STRING:
      return literal_at(t, P, k);
    case UGX_ADV_STRING_PMA:
      if (k + len + min > end || !literal_at(t, P, k))
        return false;
      return k + len + 4 > end || pm4(t, T.pred, k + len);
    case UGX_ADV_STRING_PMH:
      if (k + len + min > end || !literal_at(t, P, k))
        return false;
      return pmh(t, T.pred, k + len, min);
    case UGX_ADV_NONE:
      // advance_none (lib/matcher.cpp:957-960; option N with min_ == 0, :804) never moves the cursor: find() then
      // attempts the DFA at every position in turn, which is what "every position is a candidate" gives
      return true;
    default:
      return false;
  }
}

// ---- word characters ----
__device__ __forceinline__ bool is_alnum_ascii(int c)
{
  return (c >= '0' && c <= '9') || (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z');
}

__device__ inline bool is_word_cp(const DevPattern& P, int c)
{
  int lo = 0, hi = static_cast<int>(P.n_word_ranges) - 1;
  while (lo <= hi)
  {
    int mid = (lo + hi) >> 1;
    if (c < __ldg(P.word_ranges + 2 * mid))
      hi = mid - 1;
    else if (c > __ldg(P.word_ranges + 2 * mid + 1))
      lo = mid + 1;
    else
      return true;
  }
  return false;
}

// reflex::utf8(), include/reflex/utf8.h:138-215 (invalid -> U+FFFD)
__device__ inline int decode_utf8(const Text& t, uint64_t i)
{
  int c = t.at(i);
  if (c < 0x80)
    return c;
  int c1 = t.at(i + 1);
  if (c < 0xC0 || (c == 0xC0 && c1 != 0x80) || c == 0xC1 || (c1 & 0xC0) != 0x80)
    return 0xFFFD;
  c1 &= 0x3F;
  if (c < 0xE0)
    return ((c & 0x1F) << 6) | c1;
  int c2 = t.at(i + 2);
  if ((c == 0xE0 && c1 < 0x20) || (c2 & 0xC0) != 0x80)
    return 0xFFFD;
  c2 &= 0x3F;
  if (c < 0xF0)
    return ((c & 0x0F) << 12) | (c1 << 6) | c2;
  int c3 = t.at(i + 3);
  if ((c == 0xF0 && c1 < 0x10) || (c == 0xF4 && c1 >= 0x10) || c >= 0xF5 || (c3 & 0xC0) != 0x80)
    return 0xFFFD;
  return ((c & 0x07) << 18) | (c1 << 12) | (c2 << 6) | (c3 & 0x3F);
}

// ---- the matcher state a find() needs (AbstractMatcher fields, absmatcher.h:1632-1660) ----
struct Cursor {
  uint64_t cur, pos, txt;
  uint32_t len;
  int got;
  uint32_t cap;
};

// AbstractMatcher::set_current (absmatcher.h:1576).  `got_` (the byte before the cursor) is only read by the META
// predicates and by option W: scans without either skip the load (need_got false).
__device__ __forceinline__ void set_current(const Text& t, Cursor& m, uint64_t loc, bool need_got = true)
{
  m.pos = m.cur = loc;
  if (need_got)
    m.got = loc > 0 ? static_cast<int>(t.raw(loc - 1)) : '\n';
}

__device__ __forceinline__ int get_ch(const Text& t, Cursor& m) { return m.pos < t.end ? static_cast<int>(t.raw(m.pos++)) : D_EOF; }
__device__ __forceinline__ int peek_ch(const Text& t, const Cursor& m) { return m.pos < t.end ? static_cast<int>(t.raw(m.pos)) : D_EOF; }

__device__ inline bool at_wb(const Text& t, const DevPattern& P, const Cursor& m)
{
  int c = m.got;
  if (c == '\n')
    return true;
  if (c == '_')
    return false;
  if ((c & 0xC0) == 0x80 && m.cur > 0)
  {
    uint64_t k = m.cur - 1;
    if (k > 0 && (t.raw(--k) & 0xC0) == 0x80)
      if (k > 0 && (t.raw(--k) & 0xC0) == 0x80)
        if (k > 0)
          --k;
    return !is_word_cp(P, decode_utf8(t, k));
  }
  return !is_alnum_ascii(c);
}

__device__ inline bool at_we(const Text& t, const DevPattern& P, int c, uint64_t k)
{
  if (c == D_EOF)
    return true;
  if (c == '_')
    return false;
  if ((c & 0xC0) == 0xC0)
    return !is_word_cp(P, decode_utf8(t, k));
  return !is_alnum_ascii(c);
}

__device__ inline bool at_bw(const Text& t, const DevPattern& P, const Cursor& m)
{
  uint64_t i = m.txt + m.len;
  int c = t.at(i);
  if (c == '_')
    return true;
  if ((c & 0xC0) == 0xC0)
    return is_word_cp(P, decode_utf8(t, i));
  return is_alnum_ascii(c);
}

__device__ inline bool at_ew(const Text& t, const DevPattern& P, const Cursor& m, int c)
{
  uint64_t k = m.pos + (c == D_EOF);
  c = k > 1 ? static_cast<int>(t.raw(k - 2)) : m.got;
  if (c == '\n')
    return false;
  if (c == '_')
    return true;
  if ((c & 0xC0) == 0x80 && k > 2)
  {
    k -= 3;
    if ((t.raw(k) & 0xC0) == 0x80)
      if (k > 0 && (t.raw(--k) & 0xC0) == 0x80)
        if (k > 0)
          --k;
    return is_word_cp(P, decode_utf8(t, k));
  }
  return is_alnum_ascii(c);
}

__device__ inline bool meta_holds(const Text& t, const DevPattern& P, const Cursor& m, uint32_t code, int ch, bool bol)
{
  switch (code)
  {
    case 0x0c: return ch == D_EOF;
    case 0x0b: return false;
    case 0x0a: return ch == D_EOF || ch == '\n' || (ch == '\r' && peek_ch(t, m) == '\n');
    case 0x09: return bol;
    case 0x08: return at_we(t, P, ch, m.pos) && at_ew(t, P, m, ch);
    case 0x07: return !at_we(t, P, ch, m.pos) && !at_ew(t, P, m, ch);
    case 0x06: return !at_bw(t, P, m) && !at_wb(t, P, m);
    case 0x05: return at_bw(t, P, m) && at_wb(t, P, m);
    case 0x04: return at_we(t, P, ch, m.pos) != at_ew(t, P, m, ch);
    case 0x03: return at_bw(t, P, m) != at_wb(t, P, m);
    case 0x02: return at_we(t, P, ch, m.pos) == at_ew(t, P, m, ch);
    case 0x01: return at_bw(t, P, m) == at_wb(t, P, m);
    default: return false;
  }
}

__device__ __forceinline__ bool d_op_is_goto(uint32_t op) { return (op << 8) >= (op & 0xff000000u); }

} // namespace ugx
