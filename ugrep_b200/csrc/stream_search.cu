// stream_search.cu — count_lines_search_kernel: `ugrep -c` as one left-to-right pass of the line-resetting search
// automaton (pattern_host.hpp SearchDfa, DESIGN.md §4.3a) instead of candidates, queues and rounds of anchored attempts.
//
// Why it is exact: on the streaming route with DevPattern::covers, a line counts iff some interior position in it
// starts a non-empty anchored match (stream_count.cu).  The automaton is MATCHED after byte k iff some attempt started
// earlier in the line has decided "match" by byte k, so the success bit of byte k is "state == MATCHED" and a line
// counts iff it has a success — attributed to the accepting byte instead of the start byte, both in the same line.
// An attempt decides within D bytes (the decision depth), so the state at x is determined, MATCHED aside, by bytes
// [x - (D - 1), x): a lane that starts from the empty set D - 1 bytes before its segment reaches, at the first byte
// where the line's first match decides, the same transition into MATCHED as a pass from the line start.
//
// Work decomposition: the regions, their schedule, the line state with its carry arithmetic, the region summaries and
// the epilogue are those of stream_common.cuh.  A warp walks its 16 KiB region in 2 KiB blocks; lane l owns the 64
// contiguous bytes [64 l, 64 l + 64) of a block (four LDG.128; the next block is in flight while this one runs).  The
// D - 1 warm-up bytes come from lane l - 1 by shuffle (lane 0: one 16-byte load before the block, or '\n' bytes at the
// buffer's start, which leave the empty set).  Per byte: one class lookup and one transition in shared memory.
//
// The end of the buffer.  count_lines_stream_kernel skips the candidate predicate only on interior spans
// (sbase + SC_SPAN + 24 <= n): from the first other span, p0, a position counts iff it passes cand() AND starts a
// match.  So the automaton's success bits are dropped from p0 on, and the lanes whose segments reach p0 - (D - 1) take
// the positions there one by one (tail_successes): an attempt from p in [p0 - (D - 1), p0) that matches, and
// cand(p) && attempt(p) for p >= p0, mark p itself.  Attempts from before p0 - (D - 1) decide before p0, where the
// automaton still sees them.  Only the last launch of a buffer has such lanes, and only in its last one or two blocks.
#include "device_pattern.cuh"
#include "ptx.cuh"
#include "scan_kernels.hpp"
#include "stream_common.cuh"

namespace ugx {

namespace {

constexpr int SS_THREADS = 512;
constexpr uint32_t SS_BLOCK = 2048; // bytes per block: 32 lanes x 64

// resolve_span (stream_common.cuh) for 64-byte lane segments: the same carry arithmetic with the carry out of bit 63
// taken from the 64-bit add, and the same three ballots across lanes
__device__ __forceinline__ void resolve_span64(LineState& L, uint64_t nl, uint64_t succ)
{
  const uint64_t s = succ & ~nl;
  const uint64_t sum = s + ~nl;
  const uint32_t g = sum < s ? 1u : 0u;                       // success after the last newline (or anywhere, if none)
  const uint64_t v = sum & nl;                                // newlines that end a segment with a success
  const uint64_t first = nl & (0ull - nl);
  const bool has = nl != 0;
  const bool hs = has ? (v & first) != 0 : g != 0;            // success before the first newline
  L.lcount += __popcll(v & ~first) + (has ? g : 0u);          // lines that start inside this segment
  const uint32_t NL = __ballot_sync(0xffffffffu, has);
  const uint32_t H = __ballot_sync(0xffffffffu, hs);
  const uint32_t G = __ballot_sync(0xffffffffu, g != 0);
  const uint32_t A = G | ~NL;
  const uint64_t carry = static_cast<uint64_t>(A) + G + L.cin;
  const uint32_t C = static_cast<uint32_t>(carry) ^ A ^ G;   // bit l: the line open at lane l's first byte already counted
  if (!L.seen_nl)
  {
    const uint32_t headlanes = NL != 0 ? (((NL & (0u - NL)) << 1) - 1u) : 0xffffffffu;
    if ((H & headlanes) != 0)
      L.head = true;
  }
  L.ucount += __popc(H & ~C);
  L.cin = static_cast<uint32_t>(carry >> 32);
  if (NL != 0)
    L.seen_nl = true;
}

__device__ __forceinline__ uint32_t word_of(const uint4 (&v)[4], int i)
{
  const uint4 q = v[i >> 2];
  return (i & 3) == 0 ? q.x : (i & 3) == 1 ? q.y : (i & 3) == 2 ? q.z : q.w;
}

// one transition: pre-multiplied row offset + class, then the next row offset.  The table follows the 256-byte class map
// in shared memory, so one base address serves both lookups (the offset folds into the LDS).
__device__ __forceinline__ uint32_t search_step(uint32_t cls_s, uint32_t st, uint32_t byte)
{
  return lds_u16(cls_s + 256 + 2 * (st + lds_u8(cls_s + byte)));
}

__device__ __forceinline__ uint32_t newline_mask16(uint4 q) { return newline_mask_exact4(q.x, q.y, q.z, q.w); }

__device__ __forceinline__ void load_segment(uint4 (&v)[4], const uint8_t* __restrict__ p)
{
#pragma unroll
  for (int j = 0; j < 4; ++j)
    v[j] = __ldg(reinterpret_cast<const uint4*>(p) + j);
}

// the same where the segment may reach past the valid bytes: bytes at or past n read as zero (never newlines)
__device__ __forceinline__ void load_segment_guarded(uint4 (&v)[4], const uint8_t* __restrict__ buf, uint64_t n, uint64_t at)
{
#pragma unroll
  for (int j = 0; j < 4; ++j)
    v[j] = load_chunk_guarded(buf, n, at + 16 * j);
}

// does an anchored attempt at `pos` give a non-empty match?  The decision of attempt_table (stream_count.cu): the first
// accepting state, dead state or leaf reached decides (acc0 is 0 on this route).
__device__ __forceinline__ bool attempt_matches(const Text& t, const DevPattern& P, uint64_t pos)
{
  uint32_t state = 0;
  for (uint64_t p = pos; p < t.end; ++p)
  {
    const uint32_t nxt = __ldg(P.next + state * P.ncls + __ldg(P.cls + t.raw(p)));
    if (nxt >= P.first_acc)
    {
      if (nxt == D_DEAD)
        return false;
      if (nxt < P.first_leaf)
        return true;
      return (__ldg(P.accept + nxt) & 0x7fffffffu) != 0; // leaf: accepting unless it is a dead end
    }
    state = nxt;
  }
  return false;
}

// the success mask of a segment [seg, seg + 64) that reaches p0 - (D - 1): the automaton's bits before p0, and the
// positions from p0 - (D - 1) on evaluated as count_lines_stream_kernel evaluates them at the end of the buffer.
// (called in the last blocks of a buffer only)
__device__ __forceinline__ uint64_t tail_successes(const DevPattern& P, const uint8_t* __restrict__ buf, uint64_t n, uint64_t seg,
                                                uint64_t p0, uint32_t dm1, uint64_t succ)
{
  const Text t{buf, n};
  Tables T;
  T.cls = P.cls;
  T.next = P.next;
  T.pred = P.pred;
  T.tap = P.tap;
  succ &= p0 <= seg ? 0ull : p0 - seg >= 64 ? ~0ull : (1ull << (p0 - seg)) - 1;
  for (uint32_t k = 0; k < 64 && seg + k < n; ++k)
  {
    const uint64_t p = seg + k;
    if (p + dm1 < p0)
      continue;
    if ((p < p0 || cand(t, P, T, p)) && attempt_matches(t, P, p))
      succ |= 1ull << k;
  }
  return succ;
}

// the automaton over one lane's 64 bytes of the block at blk (in v): warm-up over the D - 1 bytes before the segment
// (from the previous lane; lane 0: one 16-byte load, or '\n' bytes at the buffer's start), then one step per byte.
// `between` runs after the warm-up (the hot loop issues the next block's loads there).  Returns bit k = MATCHED after
// byte k.
template <class Between>
__device__ __forceinline__ uint64_t segment_successes(uint32_t cls_s, uint32_t empty, uint32_t skip, uint32_t lane,
                                                      const uint8_t* __restrict__ buf, uint64_t blk, const uint4 (&v)[4],
                                                      Between&& between)
{
  uint4 wu;
  wu.x = __shfl_up_sync(0xffffffffu, v[3].x, 1);
  wu.y = __shfl_up_sync(0xffffffffu, v[3].y, 1);
  wu.z = __shfl_up_sync(0xffffffffu, v[3].z, 1);
  wu.w = __shfl_up_sync(0xffffffffu, v[3].w, 1);
  if (lane == 0)
    wu = blk >= 16 ? __ldg(reinterpret_cast<const uint4*>(buf + blk - 16)) : make_uint4(0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au);
  uint32_t st = empty;
#pragma unroll
  for (uint32_t i = 0; i < 16; ++i)
    if (i >= skip)
    {
      const uint32_t w = i < 4 ? wu.x : i < 8 ? wu.y : i < 12 ? wu.z : wu.w;
      st = search_step(cls_s, st, (w >> (8 * (i & 3))) & 0xffu);
    }
  between();
  uint32_t s_lo = 0, s_hi = 0;
#pragma unroll
  for (int i = 0; i < 64; ++i)
  {
    st = search_step(cls_s, st, (word_of(v, i >> 2) >> (8 * (i & 3))) & 0xffu);
    if (i < 32)
      s_lo |= (st == 0 ? 1u : 0u) << i;
    else
      s_hi |= (st == 0 ? 1u : 0u) << (i - 32);
  }
  return (static_cast<uint64_t>(s_hi) << 32) | s_lo;
}

// the same automaton for a region near the end of the buffer, one byte at a time from memory (a rolled loop: a second
// unrolled copy of the one above would crowd the registers of the hot loop)
__device__ __forceinline__ uint64_t tail_segment_successes(uint32_t cls_s, uint32_t empty, uint32_t dm1,
                                                           const uint8_t* __restrict__ buf, uint64_t n, uint64_t seg)
{
  uint32_t st = empty;
  for (uint64_t p = seg > dm1 ? seg - dm1 : 0; p < seg && p < n; ++p)
    st = search_step(cls_s, st, __ldg(buf + p));
  uint64_t succ = 0;
#pragma unroll 1
  for (uint32_t k = 0; k < 64 && seg + k < n; ++k)
  {
    st = search_step(cls_s, st, __ldg(buf + seg + k));
    if (st == 0)
      succ |= 1ull << k;
  }
  return succ;
}

// newline mask of the segment, line resolution, newline count
template <bool WANT_NL>
__device__ __forceinline__ void block_resolve(LineState& L, uint32_t& region_nl, const uint4 (&v)[4], uint64_t succ)
{
  const uint64_t nl = static_cast<uint64_t>(newline_mask16(v[0]) | (newline_mask16(v[1]) << 16)) |
                      (static_cast<uint64_t>(newline_mask16(v[2]) | (newline_mask16(v[3]) << 16)) << 32);
  resolve_span64(L, nl, succ);
  if (WANT_NL)
    region_nl += __popc(static_cast<uint32_t>(nl)) + __popc(static_cast<uint32_t>(nl >> 32));
}

} // namespace

template <bool WANT_NL>
#ifndef UGX_SEARCH_MINB
#define UGX_SEARCH_MINB 1 // one CTA per SM: at 64 registers (two CTAs) the loop spills
#endif
__global__ void __launch_bounds__(SS_THREADS, UGX_SEARCH_MINB)
count_lines_search_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, StreamArgs a)
{
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t* s_cls = smem;
  uint16_t* s_next = reinterpret_cast<uint16_t*>(smem + 256);
  for (uint32_t i = threadIdx.x; i < 16; i += blockDim.x)
    reinterpret_cast<uint4*>(s_cls)[i] = __ldg(reinterpret_cast<const uint4*>(P.search_cls) + i);
  for (uint32_t i = threadIdx.x; i < P.search_bytes / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(s_next)[i] = __ldg(reinterpret_cast<const uint4*>(P.search_next) + i);
  __syncthreads();

  uint32_t cls_s = smem_u32(s_cls);
  uint32_t empty = P.search_ncls;                     // the empty set's row offset
  uint32_t skip = 16 - (P.search_depth - 1);          // warm-up: the last D - 1 of the 16 bytes before the segment
  uint32_t lane = threadIdx.x & 31;
  asm volatile("" : "+r"(cls_s), "+r"(empty), "+r"(skip), "+r"(lane));

  // the first position of the spans count_lines_stream_kernel does not treat as interior
  const uint64_t p0 = n < SC_SPAN + 24 ? 0 : ((n - SC_SPAN - 24) / SC_SPAN + 1) * SC_SPAN;
  const uint64_t nregions = a.region_end;
  unsigned long long my_lines = 0, my_newlines = 0;
  uint32_t warp_uniform_lines = 0;
  RegionSchedule sched;
  sched.init(a.ticket, a.region_end - a.region_begin);
  uint64_t r = a.region_begin + sched.next(lane);
  // a region is interior when every lane of it runs the automaton alone (its segments end before p0 - (D - 1))
  auto interior = [&](uint64_t reg) { return reg * SC_REGION + SC_REGION + 16 <= p0; };
  uint4 v[4];
  if (r < nregions && interior(r))
    load_segment(v, buf + r * SC_REGION + lane * 64);
  while (r < nregions)
  {
    const uint64_t rbase = r * SC_REGION;
    if (rbase >= n)
      break; // defensive: a region range that does not match the valid bytes must not spin
    const uint64_t rnext = a.region_begin + sched.next(lane);
    const bool have_next = rnext < nregions && interior(rnext); // the first block of the next region is prefetched
    LineState L;
    L.cin = 1;
    L.seen_nl = false;
    L.watch = true;
    L.head = false;
    L.ucount = 0;
    L.lcount = 0;
    uint32_t region_nl = 0; // WANT_NL: newlines of this region
    if (interior(r))
    {
      // interior region: the automaton alone; the next block is in flight while this one runs
#pragma unroll 1
      for (uint32_t b = 0; b < SC_REGION / SS_BLOCK; ++b)
      {
        const uint64_t blk = rbase + static_cast<uint64_t>(b) * SS_BLOCK;
        const bool last = b + 1 == SC_REGION / SS_BLOCK;
        uint4 nv[4];
        const uint64_t succ = segment_successes(cls_s, empty, skip, lane, buf, blk, v, [&] {
          if (!last || have_next)
            load_segment(nv, buf + (last ? rnext * SC_REGION : blk + SS_BLOCK) + lane * 64);
        });
        block_resolve<WANT_NL>(L, region_nl, v, succ);
        if (!last || have_next)
        {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            v[j] = nv[j];
        }
      }
    }
    else
    {
      // a region that reaches p0 - (D - 1): blocks loaded one at a time, the lanes near the end take their positions
      // one by one
#pragma unroll 1
      for (uint64_t blk = rbase; blk < rbase + SC_REGION && blk < n; blk += SS_BLOCK)
      {
        load_segment_guarded(v, buf, n, blk + lane * 64);
        const uint64_t seg = blk + lane * 64;
        uint64_t succ = tail_segment_successes(cls_s, empty, 16 - skip, buf, n, seg);
        if (seg + 64 + (16 - skip) > p0)
          succ = tail_successes(P, buf, n, seg, p0, 16 - skip, succ);
        block_resolve<WANT_NL>(L, region_nl, v, succ);
      }
      if (have_next)
        load_segment(v, buf + rnext * SC_REGION + lane * 64);
    }
    // publish the region: bit 0 has newline, bit 1 head success, bit 2 carry out
    if (lane == 0)
    {
      const uint32_t g = L.seen_nl ? L.cin : (L.head ? 1u : 0u);
      a.region_sum[r] = static_cast<uint8_t>((L.seen_nl ? 1u : 0u) | (L.head ? 2u : 0u) | (g << 2));
    }
    my_lines += L.lcount;
    my_newlines += region_nl;
    warp_uniform_lines += L.ucount;
    r = rnext;
  }
  stream_epilogue(a, nregions, my_lines, my_newlines, warp_uniform_lines);
}

cudaError_t launch_count_lines_search(const DevPattern& P, const uint8_t* buf, uint64_t n, const StreamArgs& a, bool want_nl,
                                      int sm_count, cudaStream_t st)
{
  auto kern = want_nl ? count_lines_search_kernel<true> : count_lines_search_kernel<false>;
  const size_t smem = 256 + P.search_bytes;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, UGX_MAX_DYN_SMEM);
  if (e != cudaSuccess)
    return e;
  int per_sm = 1;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SS_THREADS, smem);
  if (e != cudaSuccess)
    return e;
  kern<<<stream_grid((a.region_end - a.region_begin) * SC_REGION, sm_count, per_sm, SS_THREADS), SS_THREADS, smem, st>>>(
      P, buf, n, a);
  return cudaGetLastError();
}

} // namespace ugx
