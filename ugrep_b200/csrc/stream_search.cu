// stream_search.cu — count_lines_search_kernel: `ugrep -c` as one left-to-right pass of the line-resetting search
// automaton (pattern_host.hpp SearchDfa, DESIGN.md §4.3a) instead of candidates, queues and rounds of anchored attempts.
//
// Why it is exact: on the streaming route with DevPattern::covers, a line counts iff some interior position in it
// starts a non-empty anchored match (stream_count.cu).  The automaton is MATCHED after byte k iff some attempt started
// earlier in the line has decided "match" by byte k, so the success bit of byte k is "state == MATCHED" and a line
// counts iff it has a success — attributed to the accepting byte instead of the start byte, both in the same line.
// An attempt decides within D bytes (the decision depth), so the state at x is determined, MATCHED aside, by bytes
// [x - (D - 1), x): a lane that starts from the empty set D - 1 bytes before its stretch reaches, at the first byte
// where the line's first match decides, the same transition into MATCHED as a pass from the line start.
//
// Work decomposition: the regions, their schedule, the line state with its carry arithmetic, the region summaries and
// the epilogue are those of stream_common.cuh.  A warp splits its 16 KiB region into rounds of 64 lane stretches of
// SS_S contiguous bytes; in a round lane l runs two automata side by side, one over stretch l of the round's first half
// and one over stretch l of its second half, so every lane keeps two independent chains of shared-memory lookups in
// flight.  Each automaton starts from the empty set D - 1 bytes before its stretch (one 16-byte load) and carries its
// state across the stretch's 32-byte steps; the lane resolves its lines per step on its own (stretch_step), and the
// warp chains its 32 stretches of each half once per round with three ballots (combine_stretches).  The next step's
// 32 bytes of both stretches are loaded while the current step runs.  Per byte: one class lookup and one transition
// in shared memory.
//
// The end of the buffer.  count_lines_stream_kernel skips the candidate predicate only on interior spans
// (sbase + SC_SPAN + 24 <= n): from the first other span, p0, a position counts iff it passes cand() AND starts a
// match.  So the automaton's success bits are dropped from p0 on, and the steps that reach p0 - (D - 1) take the
// positions there one by one (tail_successes): an attempt from p in [p0 - (D - 1), p0) that matches, and
// cand(p) && attempt(p) for p >= p0, mark p itself.  Attempts from before p0 - (D - 1) decide before p0, where the
// automaton still sees them.  Only the last launch of a buffer has such regions, and only its last one or two.
#include "device_pattern.cuh"
#include "ptx.cuh"
#include "scan_kernels.hpp"
#include "stream_common.cuh"

namespace ugx {

namespace {

constexpr int SS_THREADS = 512;
#ifndef UGX_SEARCH_S
#define UGX_SEARCH_S 256
#endif
constexpr uint32_t SS_S = UGX_SEARCH_S;           // bytes per lane stretch
constexpr uint32_t SS_STEP = 32;                  // bytes per step of a stretch (one 32-byte load)
constexpr uint32_t SS_STEPS = SS_S / SS_STEP;
constexpr uint32_t SS_HALF = 32 * SS_S;           // one chain of a round: 32 lanes x SS_S
constexpr uint32_t SS_ROUNDS = SC_REGION / (2 * SS_HALF);
static_assert(SS_S % SS_STEP == 0 && SC_REGION % (2 * SS_HALF) == 0, "a region is a whole number of rounds of 64 stretches");

// one lane's automaton over its stretch, and what the lane knows of the stretch's lines.  f: bit 0 the stretch has a
// newline so far, bit 1 a success before its first newline, bit 2 a success after its last newline (or anywhere, if it
// has none) — one register, for the hot loop's two stretches
struct Stretch {
  uint32_t st; // automaton state (row offset)
  uint32_t f;
};

// one step of a stretch: bit k of nl / succ = byte k is a newline / the automaton is MATCHED after it.  The carry
// arithmetic of resolve_span (stream_common.cuh) inside the lane, continued from the steps before: lines that start
// inside the stretch and have a success in it are counted here, once.
__device__ __forceinline__ void stretch_step(Stretch& T, uint32_t& lcount, uint32_t nl, uint32_t succ)
{
  const uint32_t s = succ & ~nl;
  const uint32_t sum = s + ~nl;
  const uint32_t g = sum < s ? 1u : 0u;                      // success after the step's last newline (or anywhere)
  const uint32_t v = sum & nl;                               // newlines that end a piece with a success
  const uint32_t first = nl & (0u - nl);
  const uint32_t has = nl != 0 ? 1u : 0u;
  const uint32_t hs = has ? ((v & first) != 0 ? 1u : 0u) : g; // success before the step's first newline
  const uint32_t tnl = T.f & 1u, topen = (T.f >> 2) & 1u;
  lcount += (tnl & hs & ~topen) + (has ? __popc(v & ~first) + g : 0u);
  const uint32_t head = (T.f >> 1) & 1u | (~tnl & hs);
  const uint32_t open = has ? g : (topen | hs);
  T.f = (tnl | has) | (head << 1) | (open << 2);
}

// the warp's 32 stretches, in lane order, into the region's line state: the carry across lanes of resolve_span
__device__ __forceinline__ void combine_stretches(LineState& L, const Stretch& T)
{
  const uint32_t NL = __ballot_sync(0xffffffffu, (T.f & 1u) != 0);
  const uint32_t H = __ballot_sync(0xffffffffu, (T.f & 2u) != 0);
  const uint32_t G = __ballot_sync(0xffffffffu, (T.f & 4u) != 0);
  const uint32_t A = G | ~NL;
  const uint64_t carry = static_cast<uint64_t>(A) + G + L.cin;
  const uint32_t C = static_cast<uint32_t>(carry) ^ A ^ G;   // bit l: the line open at stretch l's first byte already counted
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

// one transition.  The class lookup does not depend on the state, so the shared address of the byte's column is formed
// beside it, and the chain from one state to the next is one LDS.U16 and one IADD3.  The table starts at a 512-byte
// boundary (tbl_s), so the column's address is tbl_s | 2 cls; written as one sum instead, ptxas re-associates it and
// puts two adds on the chain.
__device__ __forceinline__ uint32_t search_step(uint32_t cls_s, uint32_t tbl_s, uint32_t st, uint32_t byte)
{
  const uint32_t col = tbl_s | (lds_u8(cls_s + byte) << 1);
  return lds_u16(col + 2 * st);
}

__device__ __forceinline__ uint32_t newline_mask16(uint4 q) { return newline_mask_exact4(q.x, q.y, q.z, q.w); }

__device__ __forceinline__ uint32_t byte_of(uint4 q, int i)
{
  const uint32_t w = (i >> 2) == 0 ? q.x : (i >> 2) == 1 ? q.y : (i >> 2) == 2 ? q.z : q.w;
  return (w >> (8 * (i & 3))) & 0xffu;
}

// the 16 bytes before `at` (the automaton's warm-up); '\n' before the buffer's start, which leaves the empty set
__device__ __forceinline__ uint4 warm_bytes(const uint8_t* __restrict__ buf, uint64_t at)
{
  return at >= 16 ? __ldg(reinterpret_cast<const uint4*>(buf + at - 16)) : make_uint4(0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au);
}

// the automaton from the empty set over the last D - 1 of the 16 bytes in w (skip = 16 - (D - 1))
__device__ __forceinline__ uint32_t warm_up(uint32_t cls_s, uint32_t tbl_s, uint32_t empty, uint32_t skip, uint4 w)
{
  uint32_t st = empty;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i >= static_cast<int>(skip))
      st = search_step(cls_s, tbl_s, st, byte_of(w, i));
  return st;
}

// one 32-byte step of a stretch in one load (LDG.256: `p` 32-byte aligned).  A warp's loads of a step touch 32 lines
// (one per stretch); two 16-byte loads instead would touch them twice, and the L1 wavefronts of those loads take from
// the same pipe as the automaton's lookups.
__device__ __forceinline__ void load_step32(uint4 (&v)[2], const uint8_t* p)
{
  asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(v[0].x), "=r"(v[0].y), "=r"(v[0].z), "=r"(v[0].w), "=r"(v[1].x), "=r"(v[1].y), "=r"(v[1].z), "=r"(v[1].w)
      : "l"(p));
}

__device__ __forceinline__ uint32_t newline_mask32(const uint4 (&v)[2]) { return newline_mask16(v[0]) | (newline_mask16(v[1]) << 16); }

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

// the success mask of a step [seg, seg + 32) that reaches p0 - (D - 1): the automaton's bits before p0, and the
// positions from p0 - (D - 1) on evaluated as count_lines_stream_kernel evaluates them at the end of the buffer.
// (called in the last regions of a buffer only)
__device__ __forceinline__ uint32_t tail_successes(const DevPattern& P, const uint8_t* __restrict__ buf, uint64_t n, uint64_t seg,
                                                uint64_t p0, uint32_t dm1, uint32_t succ)
{
  const Text t{buf, n};
  Tables T;
  T.cls = P.cls;
  T.next = P.next;
  T.pred = P.pred;
  T.tap = P.tap;
  succ &= p0 <= seg ? 0u : p0 - seg >= 32 ? ~0u : (1u << (p0 - seg)) - 1;
  for (uint32_t k = 0; k < SS_STEP && seg + k < n; ++k)
  {
    const uint64_t p = seg + k;
    if (p + dm1 < p0)
      continue;
    if ((p < p0 || cand(t, P, T, p)) && attempt_matches(t, P, p))
      succ |= 1u << k;
  }
  return succ;
}

// a region that reaches p0 - (D - 1): its stretches one after the other, the automaton byte by byte from memory (a
// rolled loop: a second unrolled copy of the hot loop would crowd its registers), the steps near the end of the buffer
// through tail_successes
template <bool WANT_NL>
__device__ __forceinline__ void tail_region(const DevPattern& P, uint32_t cls_s, uint32_t tbl_s, uint32_t empty, uint32_t dm1,
                                            const uint8_t* __restrict__ buf, uint64_t n, uint64_t p0, uint64_t rbase,
                                            uint32_t lane, LineState& L, uint32_t& region_nl)
{
#pragma unroll 1
  for (uint32_t h = 0; h < 2 * SS_ROUNDS; ++h)
  {
    const uint64_t base = rbase + static_cast<uint64_t>(h) * SS_HALF + lane * SS_S;
    Stretch T{empty, 0u};
    for (uint64_t p = base > dm1 ? base - dm1 : 0; p < base && p < n; ++p)
      T.st = search_step(cls_s, tbl_s, T.st, __ldg(buf + p));
#pragma unroll 1
    for (uint64_t seg = base; seg < base + SS_S && seg < n; seg += SS_STEP)
    {
      const uint4 v[2] = {load_chunk_guarded(buf, n, seg), load_chunk_guarded(buf, n, seg + 16)}; // zero past n
      const uint32_t nl = newline_mask32(v);
      uint32_t succ = 0;
#pragma unroll 1
      for (uint32_t k = 0; k < SS_STEP && seg + k < n; ++k)
      {
        T.st = search_step(cls_s, tbl_s, T.st, __ldg(buf + seg + k));
        if (T.st == 0)
          succ |= 1u << k;
      }
      if (seg + SS_STEP + dm1 > p0)
        succ = tail_successes(P, buf, n, seg, p0, dm1, succ);
      stretch_step(T, L.lcount, nl, succ);
      if (WANT_NL)
        region_nl += __popc(nl);
    }
    combine_stretches(L, T);
  }
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
  // the class map, then the table at the next 512-byte boundary of the shared space (search_step)
  uint8_t* s_cls = smem;
  const uint32_t tbl_off = ((smem_u32(smem) + 256 + 511) & ~511u) - smem_u32(smem);
  uint16_t* s_next = reinterpret_cast<uint16_t*>(smem + tbl_off);
  for (uint32_t i = threadIdx.x; i < 16; i += blockDim.x)
    reinterpret_cast<uint4*>(s_cls)[i] = __ldg(reinterpret_cast<const uint4*>(P.search_cls) + i);
  for (uint32_t i = threadIdx.x; i < P.search_bytes / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(s_next)[i] = __ldg(reinterpret_cast<const uint4*>(P.search_next) + i);
  __syncthreads();

  uint32_t cls_s = smem_u32(s_cls);
  uint32_t tbl_s = smem_u32(s_next);
  uint32_t empty = P.search_ncls;                     // the empty set's row offset
  uint32_t skip = 16 - (P.search_depth - 1);          // warm-up: the last D - 1 of the 16 bytes before a stretch
  uint32_t lane = threadIdx.x & 31;
  asm volatile("" : "+r"(cls_s), "+r"(tbl_s), "+r"(empty), "+r"(skip), "+r"(lane));
  // the scanned buffers are 16-byte aligned (capi.cu); the hot loop's steps take one 32-byte load where they can
  const bool aligned32 = (reinterpret_cast<uintptr_t>(buf) & 31) == 0;

  // the first position of the spans count_lines_stream_kernel does not treat as interior
  const uint64_t p0 = n < SC_SPAN + 24 ? 0 : ((n - SC_SPAN - 24) / SC_SPAN + 1) * SC_SPAN;
  const uint64_t nregions = a.region_end;
  unsigned long long my_lines = 0, my_newlines = 0;
  uint32_t warp_uniform_lines = 0;
  RegionSchedule sched;
  sched.init(a.ticket, a.region_end - a.region_begin);
  uint64_t r = a.region_begin + sched.next(lane);
  // a region is interior when its stretches and their warm-up bytes end before p0 - (D - 1)
  auto interior = [&](uint64_t reg) { return reg * SC_REGION + SC_REGION + 16 <= p0; };
  // the current step of both chains and the warm-up bytes of the stretches to come, loaded a step ahead
  uint4 va[2], vb[2], wa, wb;
  if (r < nregions && interior(r))
  {
    const uint64_t at = r * SC_REGION + lane * SS_S;
    wa = warm_bytes(buf, at);
    wb = warm_bytes(buf, at + SS_HALF);
#pragma unroll
    for (int j = 0; j < 2; ++j)
    {
      va[j] = __ldg(reinterpret_cast<const uint4*>(buf + at) + j);
      vb[j] = __ldg(reinterpret_cast<const uint4*>(buf + at + SS_HALF) + j);
    }
  }
  while (r < nregions)
  {
    const uint64_t rbase = r * SC_REGION;
    if (rbase >= n)
      break; // defensive: a region range that does not match the valid bytes must not spin
    const uint64_t rnext = a.region_begin + sched.next(lane);
    const bool have_next = rnext < nregions && interior(rnext); // the first step of the next region is prefetched
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
#pragma unroll 1
      for (uint32_t k = 0; k < SS_ROUNDS; ++k)
      {
        Stretch A{warm_up(cls_s, tbl_s, empty, skip, wa), 0u};
        Stretch B{warm_up(cls_s, tbl_s, empty, skip, wb), 0u};
        const uint8_t* pa = buf + rbase + static_cast<uint64_t>(k) * 2 * SS_HALF + lane * SS_S;
#pragma unroll 1
        for (uint32_t s = 0; s < SS_STEPS; ++s)
        {
          // the step after this one: the next bytes of the stretches, or the first ones of the next round's or
          // the next region's stretches (with their warm-up bytes)
          const bool last = s + 1 == SS_STEPS;
          const bool more = !last || k + 1 < SS_ROUNDS || have_next;
          const uint8_t* pn = !last ? pa + SS_STEP
                              : k + 1 < SS_ROUNDS ? buf + rbase + static_cast<uint64_t>(k + 1) * 2 * SS_HALF + lane * SS_S
                                                   : buf + rnext * SC_REGION + lane * SS_S;
          if (last)
          {
            // (defined on every path, so that the warm-up bytes are not live across the steps)
            wa = more ? warm_bytes(buf, pn - buf) : make_uint4(0, 0, 0, 0);
            wb = more ? warm_bytes(buf, pn - buf + SS_HALF) : make_uint4(0, 0, 0, 0);
          }
          uint32_t sa = 0, sb = 0;
          const uint32_t nla = newline_mask32(va), nlb = newline_mask32(vb);
#pragma unroll
          for (int j = 0; j < 2; ++j)
          {
#pragma unroll
            for (int i = 0; i < 16; ++i)
            {
              A.st = search_step(cls_s, tbl_s, A.st, byte_of(va[j], i));
              B.st = search_step(cls_s, tbl_s, B.st, byte_of(vb[j], i));
              sa |= (A.st == 0 ? 1u : 0u) << (16 * j + i);
              sb |= (B.st == 0 ? 1u : 0u) << (16 * j + i);
            }
          }
          if (more && aligned32)
          {
            load_step32(va, pn);
            load_step32(vb, pn + SS_HALF);
          }
          else if (more)
          {
#pragma unroll
            for (int j = 0; j < 2; ++j)
            {
              va[j] = __ldg(reinterpret_cast<const uint4*>(pn) + j);
              vb[j] = __ldg(reinterpret_cast<const uint4*>(pn + SS_HALF) + j);
            }
          }
          stretch_step(A, L.lcount, nla, sa);
          stretch_step(B, L.lcount, nlb, sb);
          if (WANT_NL)
            region_nl += __popc(nla) + __popc(nlb);
          pa = pn;
        }
        combine_stretches(L, A);
        combine_stretches(L, B);
      }
    }
    else
    {
      tail_region<WANT_NL>(P, cls_s, tbl_s, empty, 16 - skip, buf, n, p0, rbase, lane, L, region_nl);
      // (defined on every path, so that the prefetch registers are not live across the tail path)
      const uint4 z = make_uint4(0, 0, 0, 0);
      const uint64_t at = rnext * SC_REGION + lane * SS_S;
      wa = have_next ? warm_bytes(buf, at) : z;
      wb = have_next ? warm_bytes(buf, at + SS_HALF) : z;
#pragma unroll
      for (int j = 0; j < 2; ++j)
      {
        va[j] = have_next ? __ldg(reinterpret_cast<const uint4*>(buf + at) + j) : z;
        vb[j] = have_next ? __ldg(reinterpret_cast<const uint4*>(buf + at + SS_HALF) + j) : z;
      }
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
  const size_t smem = 256 + 496 + P.search_bytes; // the table's start rounded up to 512 bytes (the base is 16-aligned)
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
