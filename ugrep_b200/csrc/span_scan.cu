// span_scan.cu — span_scan_kernel: `ugrep -c -o` (count matches) and `ugrep -o -n -b` (match records) as a
// streaming pass in which every DFA attempt is taken OUT of the sequential find loop, for patterns with or without
// look-back, and in which lines of any length are scanned by many warps at once.
//
// The rule it implements (checked against the oracle's find loop on the CPU, tests/test_span_rule.py).  For a
// pattern without META edges, without option W and whose start state does not accept, successive calls of
// Matcher::match(FIND) (lib/matcher.cpp:42-750) over a buffer return exactly the chain
//
//     c -> the first p >= c with p in A and D(p) > 0;   c := p + D(p)
//
//   D(p) = length of the longest match of the DFA anchored at p (0 = none): a function of the text alone;
//   A    = { p : some prefilter candidate k >= p has only look-back bytes (cbk_) in [p, k) } — the positions the
//          look-back / retry rules (lib/matcher.cpp:54-70, 627-658) can attempt: after a candidate k the matcher
//          walks back over the cbk_ run below k and then tries every position of that run up to k in increasing
//          order (first by its retry budget, then — budget spent — by advancing again with the floor one byte on),
//          so within one find() the attempted positions are A at or after the cursor, in order.  Without look-back
//          A is the candidate set.  A is position-local: A(p) = cand(p) | (cbk(p) & A(p + 1)), a carry chain that
//          runs from high to low addresses.
//
// Work decomposition.  The buffer is cut into 16 KiB regions; a warp owns the matches that START in its region.  It
// walks the region in 512-byte spans, lane l holding chunk l (16 bytes + halo) of the span:
//   1. masks    candidate / look-back / newline bits of the 16 positions (register window, tile_phase_a.cuh);
//   2. A        the carry chain within the lane (a 16-bit add), across lanes (a 64-bit add of two ballots) and across
//               spans (the next span's masks are evaluated one iteration ahead);
//   3. D        the positions of A are compacted into a per-warp queue and handed out one per lane, so the attempts
//               run with full warps whatever their distribution; results go to a per-warp table in shared memory;
//   4. chain    every lane resolves its own successes assuming the cursor reaches it before its first success; one
//               shuffle checks the assumption for all lanes; spans in which a match straddles into a lane's first
//               success (rare) are resolved lane after lane instead.
// The chain state at a region start comes from the 512 bytes before it (the "window"): after a newline in the window
// the chain is fresh (no match crosses a newline: no DFA in scope has a '\n' transition); without one it is taken fresh
// from the window's first success, which is right unless a match that starts before the window reaches beyond that
// point — every region publishes the farthest end of its matches and the final kernel checks exactly that condition;
// a violation (a match longer than 512 bytes straddling a region start inside a line longer than 512 bytes) makes the
// caller fall back to the line-at-a-time kernels for this buffer.  Hence a 1 GiB line is scanned by all warps.
//
// End of the buffer.  A failed attempt that read up to the end of the buffer makes the reference continue byte by
// byte without its prefilter (lib/matcher.cpp:623 `if (!at_end())`, :709-713).  Only attempts in the last line can
// do that.  The last line (when it is at most 64 KiB long) is therefore left to one thread of the final kernel, which
// runs the line-at-a-time form (find_in_line) on it; a longer last line stays with the spans and an attempt that
// fails at the end of the buffer raises the same fallback flag.
#include "block_scan.cuh"
#include "device_pattern.cuh"
#include "line_match.cuh"
#include "ptx.cuh"
#include "scan_kernels.hpp"
#include "stream_common.cuh"
#include "tile_phase_a.cuh"
#include "viability.cuh"

namespace ugx {

namespace {

constexpr uint32_t SP_SPAN = 512;
constexpr int SP_SPANS = SC_REGION / SP_SPAN; // spans per region
constexpr uint32_t SP_LONG = 0xffffu;         // D(p) is kept in 16 bits
constexpr uint64_t SP_NO_V = ~0ull;           // region needs no validation (its chain starts after a newline)
constexpr uint32_t SP_FAR_SPANS = 2048;       // longest look-ahead over a run of look-back bytes (1 MiB): beyond it the
                                              // buffer goes to the line-at-a-time kernels, where ONE thread walks the line —
                                              // far worse than looking ahead

struct SpanMasks {
  uint32_t cand, cbk, nl, via; // 16 bits each: bit k = byte k of the lane's chunk
};

// masks of the chunk at `base` (16-byte aligned); positions at or past `limit` read as nothing
__device__ __forceinline__ SpanMasks eval_masks(const Text& t, const DevPattern& P, const Tables& T, const uint8_t* s_flags,
                                                const ViaTables& via, uint64_t base, uint64_t limit, bool want_cand,
                                                bool want_cbk, bool want_via)
{
  SpanMasks m;
  m.cand = m.cbk = m.nl = m.via = 0;
  if (base >= limit)
    return m;
  Window W;
  const bool interior = load_window(t.b, t.end, base, W);
  if (want_cand)
    m.cand = interior ? chunk_cand_fast(W, t, P, T, base) : chunk_cand_generic(t, P, T, base);
  m.nl = newline_mask16(W);
  if (want_cbk)
  {
#pragma unroll
    for (int k = 0; k < 16; ++k)
      m.cbk |= static_cast<uint32_t>(s_flags[UGX_WB(W, k)] & 1u) << k;
  }
  // positions whose next bytes cannot start a match (the last bytes of the buffer are left to the attempt)
  m.via = (want_via && interior) ? viable16(via, W) : 0xffffu;
  if (base + 16 > limit)
  {
    const uint32_t valid = (1u << (limit - base)) - 1u;
    m.cand &= valid;
    m.cbk &= valid;
    m.nl &= valid;
    m.via &= valid;
  }
  return m;
}

// A(p) = C(p) | (R(p) & A(p + 1)) over the 16 positions of a chunk; cin = A(position 16); cout = A(position 0)
__device__ __forceinline__ uint32_t flood16(uint32_t C, uint32_t R, uint32_t cin, uint32_t& cout)
{
  const uint32_t c = __brev(C) >> 16, r = __brev(R) >> 16; // reversed: the carry now runs upwards
  const uint32_t a = c | r;
  const uint32_t sum = a + c + cin;
  const uint32_t K = sum ^ a ^ c;                         // carry into every bit
  cout = (K >> 16) & 1u;
  return __brev((c | (r & K)) & 0xffffu) >> 16;
}

// lane-level carry behaviour of a span: G = lanes whose position 0 is in A whatever comes in, Pp = lanes that only
// pass the carry on (all 16 bytes look-back bytes, no candidate)
struct SpanCarry {
  uint32_t G, Pp;
  // A(first position of the span) given the carry into its last lane
  __device__ __forceinline__ uint32_t out(uint32_t cin) const
  {
    const uint32_t g = __brev(G), a = g | __brev(Pp);
    return static_cast<uint32_t>((static_cast<uint64_t>(a) + g + cin) >> 32);
  }
  // the carry into lane `lane`
  __device__ __forceinline__ uint32_t into(uint32_t cin, uint32_t lane) const
  {
    const uint32_t g = __brev(G), a = g | __brev(Pp);
    const uint32_t K = static_cast<uint32_t>(static_cast<uint64_t>(a) + g + cin) ^ a ^ g;
    return (K >> (31u - lane)) & 1u;
  }
};

__device__ __forceinline__ SpanCarry span_carry(const SpanMasks& m)
{
  uint32_t g;
  flood16(m.cand, m.cbk, 0u, g);
  SpanCarry c;
  c.G = __ballot_sync(0xffffffffu, g != 0);
  c.Pp = __ballot_sync(0xffffffffu, m.cbk == 0xffffu && m.cand == 0);
  return c;
}

// the candidate test at one position, for the lazy form of the attempt set (PM4 / bitap prefilters, whose masks cost
// several table lookups per byte: they are evaluated only where a viable position asks)
__device__ __forceinline__ bool cand_at(const Text& t, const DevPattern& P, const Tables& T, uint64_t q)
{
  if (P.adv == UGX_ADV_PMA && q + 12 <= t.end)
  {
    const uint8_t* p = t.b + q;
    const uint32_t sh = (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(p)) & 3u) * 8;
    const uint32_t* a = reinterpret_cast<const uint32_t*>(p - (sh >> 3));
    return pm4_x(T.pred, __funnelshift_r(__ldg(a), __ldg(a + 1), sh));
  }
  return cand(t, P, T, q);
}

// p in A?  (A(p) = cand(p) | (cbk(p) & A(p + 1)), walked forwards from p)
__device__ __forceinline__ bool in_attempt_set(const Text& t, const DevPattern& P, const Tables& T, const uint8_t* s_flags,
                                               uint64_t pos, uint32_t& bad)
{
  uint64_t q = pos;
  for (uint32_t steps = 0;; ++steps)
  {
    if (q >= t.end)
      return false;
    if (cand_at(t, P, T, q))
      return true;
    if (P.lbk == 0 || (s_flags[t.raw(q)] & 1u) == 0)
      return false;
    if (steps >= SP_FAR_SPANS * SP_SPAN)
    {
      bad |= 4u; // a look-back run longer than the bound: the buffer goes to the line-at-a-time kernels
      return false;
    }
    ++q;
  }
}

// the longest anchored match at offset `off` of the span at `sp` (16-byte aligned): (accept << 16) | length, 0 = none.
// The first 8 bytes come from three aligned 32-bit loads and are stepped through unrolled; `bad`: bit 1 a match too long
// for the table, bit 0 the attempt failed after reading up to the end of the buffer (see the file header)
__device__ __forceinline__ uint32_t longest_in_span(const DevPattern& P, const Stepper& step, const uint8_t* __restrict__ sp,
                                                    uint32_t off, uint32_t rel_end, uint32_t& bad)
{
  const uint32_t first_acc = P.first_acc, first_leaf = P.first_leaf;
  uint32_t state = 0, pp = off;
  // States are numbered so that [first_acc, first_leaf) accept and have byte edges, and ids >= first_leaf have no byte
  // edges (the interpreter halts there before reading; accepting unless a dead end): the walk only remembers the last
  // state of either kind and where it was, the accept word is looked up once, afterwards.
  uint32_t acc_state = 0, acc_len = 0, leaf_state = 0, leaf_len = 0;
  bool stop = false;
  auto special = [&](uint32_t nx) { // nx >= first_acc
    if (nx == D_DEAD)
      stop = true;
    else if (nx >= first_leaf)
    {
      leaf_state = nx;
      leaf_len = pp - off;
      stop = true;
    }
    else
    {
      acc_state = nx;
      acc_len = pp - off;
    }
  };
  if (off + 12 <= rel_end)
  {
    const uint32_t sh = (off & 3u) * 8;
    const uint32_t* a = reinterpret_cast<const uint32_t*>(sp + (off & ~3u));
    const uint32_t l0 = __ldg(a), l1 = __ldg(a + 1), l2 = __ldg(a + 2);
    const uint32_t lo = __funnelshift_r(l0, l1, sh), hi = __funnelshift_r(l1, l2, sh);
#pragma unroll
    for (int i = 0; i < 8; ++i)
    {
      if (!stop)
      {
        const uint32_t nx = step(state, __byte_perm(i < 4 ? lo : hi, 0, 0x4440 + (i & 3)));
        ++pp;
        if (nx >= first_acc)
          special(nx);
        state = nx;
      }
    }
  }
  while (!stop && pp < rel_end)
  {
    const uint32_t nx = step(state, __ldg(sp + pp));
    ++pp;
    if (nx >= first_acc)
      special(nx);
    state = nx;
  }
  uint32_t best = 0;
  if (leaf_state != 0)
  {
    const uint32_t acc = __ldg(P.accept + leaf_state) & 0x7fffffffu;
    if (acc != 0)
    {
      if (leaf_len >= SP_LONG || acc >= 0x8000u)
        bad |= 2u;
      best = ((acc & 0x7fffu) << 16) | (leaf_len & 0xffffu);
    }
  }
  if (best == 0 && acc_state != 0)
  {
    const uint32_t acc = __ldg(P.accept + acc_state) & 0x7fffffffu;
    if (acc_len >= SP_LONG || acc >= 0x8000u)
      bad |= 2u;
    best = ((acc & 0x7fffu) << 16) | (acc_len & 0xffffu);
  }
  if (best == 0 && pp >= rel_end)
    bad |= 1u;
  return best;
}

} // namespace

// the start of the buffer's last line, if that line is at most SPAN_TAIL_MAX bytes long: tail[0] = its offset, else n
__global__ void __launch_bounds__(32) last_line_kernel(const uint8_t* __restrict__ buf, uint64_t n, uint64_t* __restrict__ tail)
{
  const uint32_t lane = threadIdx.x;
  uint64_t t0 = n;
  if (n > 0)
  {
    // the last byte does not end a PREVIOUS line even when it is a newline: search [n - 1 - MAX, n - 1)
    const uint64_t hi = n - 1;
    const uint64_t lo = hi > SPAN_TAIL_MAX ? hi - SPAN_TAIL_MAX : 0;
    uint64_t at = hi;
    bool found = false;
    while (at > lo && !found)
    {
      const uint64_t from = at - lo > 32 * 8 ? at - 32 * 8 : lo; // 256 bytes per step
      uint32_t best = 0;
      bool mine = false;
      for (uint64_t i = from + lane * 8; i < at && i < from + lane * 8 + 8; ++i)
        if (__ldg(buf + i) == '\n')
        {
          mine = true;
          best = static_cast<uint32_t>(i - from);
        }
      const uint32_t any = __ballot_sync(0xffffffffu, mine);
      if (any != 0)
      {
        const uint32_t src = 31u - __clz(any);
        t0 = from + __shfl_sync(0xffffffffu, best, src) + 1;
        found = true;
      }
      at = from;
    }
    if (!found)
      t0 = lo == 0 ? 0 : n; // the whole buffer is one short line, or the last line is too long to set aside
  }
  if (lane == 0)
    tail[0] = t0;
}

// per region: {matches that start in it, newlines in it, farthest match ends, validation point}; with a.sel_bits, also
// the selected match starts of every chunk (16 bits per 16 text bytes) for span_emit_kernel
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS >= 512 ? 1 : 4)
span_scan_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, SpanArgs a)
{
  constexpr uint32_t NWARPS = THREADS / 32;
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  uint8_t* s_cls = smem;
  uint8_t* s_pred = s_cls + 256;
  uint8_t* s_tap = s_pred + UGX_HASH;
  uint8_t* s_flags = s_tap + UGX_BTAP;                                     // [256] bit 0: look-back byte
  uint32_t* s_dtab = reinterpret_cast<uint32_t*>(s_flags + 256);           // [NWARPS][512] (accept << 16) | length
  uint32_t* s_succ = s_dtab + NWARPS * SP_SPAN;                            // [NWARPS][16] success bits of the span
  uint16_t* s_queue = reinterpret_cast<uint16_t*>(s_succ + NWARPS * 16);   // [NWARPS][512] attempt positions
  uint8_t* s_via = reinterpret_cast<uint8_t*>(s_queue + NWARPS * SP_SPAN);
  uint16_t* s_next = reinterpret_cast<uint16_t*>(s_via + (a.use_via ? via_smem_bytes(P) : 0));
  stage_tables_bulk(&s_bar, s_cls, P.cls, s_pred, P.pred, s_tap, P.tap, s_next, P.next,
                    a.stage_table ? ((P.table_bytes + 15) / 16) * 16 : 0);
  const ViaTables via = via_stage(P, s_via, a.use_via != 0);
  for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x)
    s_flags[i] = bit256(P.cbk, i) ? 1u : 0u;
  for (uint32_t i = threadIdx.x; i < NWARPS * 16; i += blockDim.x)
    s_succ[i] = 0;
  __syncthreads();
  Tables T;
  T.cls = s_cls;
  T.pred = s_pred;
  T.tap = s_tap;
  T.next = a.stage_table ? s_next : P.next;
  const Text t{buf, n};
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t* dtab = s_dtab + wid * SP_SPAN;
  uint32_t* succ = s_succ + wid * 16;
  uint16_t* queue = s_queue + wid * SP_SPAN;
  const Stepper step(T, P.ncls, a.stage_table != 0);
  const bool has_lb = P.lbk != 0;
  // lazy attempt set: the prefilter's masks cost table lookups per byte (PM4 at every byte, bitap), and the viability
  // table is there to name the few positions worth asking about — membership in A is then decided per viable position
  const bool lazy_fam = via.on && (P.adv == UGX_ADV_PMA || P.adv == UGX_ADV_MIN1 || P.adv == UGX_ADV_MIN2 ||
                                   P.adv == UGX_ADV_MIN3 || P.adv == UGX_ADV_MIN4);
  const bool cover = P.covers != 0 && a.no_cover == 0;
  // with `cover` (every match start passes the candidate test) the viability table alone may name the positions worth an
  // attempt: taken, region by region, when a measurement shows it at least as selective as the candidate masks
  bool via_only = false;
  const uint64_t limit = __ldcg(a.tail); // spans own [0, limit): the last line belongs to the final kernel
  const uint64_t nregions = (limit + SC_REGION - 1) / SC_REGION;
  const uint64_t total_warps = static_cast<uint64_t>(gridDim.x) * NWARPS;
  uint32_t bad = 0; // bit 0: an attempt failed at the end of the buffer, bit 1: a match too long for the table
  uint32_t probe_tick = 0;
  bool via_keep = false;

  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * NWARPS + wid; r < nregions; r += total_warps)
  {
    const uint64_t rb = r * SC_REGION;
    uint64_t m_run = 0, nl_run = 0;   // matches / newlines of the region so far (warp-uniform)
    uint64_t emain = 0, elast = 0;    // lane-private: farthest end of a success that starts in spans 0..30 / span 31
    uint64_t vpoint = SP_NO_V;
    int64_t cursor = 0;               // chain cursor, relative to the current span's base (warp-uniform)
    uint64_t far_base = 0;            // look-ahead cache: the carry out of the run that ends in the span at far_base
    uint32_t far_val = 0;
    // masks of the first span to process (the window before the region, or span 0 of region 0) and of the one after
    int s = r == 0 ? 0 : -1;
    // The viability table costs two lookups per byte.  The lazy form lives on it; the mask form measures on the first
    // span of every region how many attempts it spares and keeps it only where that pays (a warp-round of attempts).
    // (the measurement is repeated every eighth region of a warp; in between its last answer stands)
    const bool probe_now = via.on && !lazy_fam && (probe_tick++ & 7u) == 0;
    const bool lazy = lazy_fam || (via_only && !probe_now);
    const bool mask_lb = has_lb && !lazy;
    bool via_r = via.on && (lazy || probe_now || via_keep);
    bool probing = probe_now;
    SpanMasks cur = eval_masks(t, P, T, s_flags, via, rb + static_cast<int64_t>(s) * SP_SPAN + lane * 16, limit, !lazy, mask_lb, via_r);
    for (; s < SP_SPANS; ++s)
    {
      const uint64_t sbase = rb + static_cast<int64_t>(s) * SP_SPAN;
      if (sbase >= limit)
        break;
      // ---- 1. masks of the next span (needed now for the carry into this one; they become `cur` afterwards)
      const SpanMasks nxt = eval_masks(t, P, T, s_flags, via, sbase + SP_SPAN + lane * 16, limit, !lazy, mask_lb, via_r);
      // ---- 2. the attempt set of this span (lazy form: the viable positions, membership decided in step 3)
      uint32_t a16 = lazy ? cur.via : cur.cand;
      if (mask_lb)
      {
        const SpanCarry cn = span_carry(nxt);
        uint32_t cin_span = cn.out(0);
        if (cn.out(1) != cin_span)
        {
          // 512 look-back bytes in a row without a candidate: look further ahead until the run ends.  The answer holds
          // for every span up to there (they all just pass the carry on), so it is kept; the look-ahead is bounded —
          // a longer run leaves the buffer to the line-at-a-time kernels.
          if (far_base <= sbase + SP_SPAN)
          {
            far_val = 0;
            far_base = limit;
            uint32_t steps = 0;
            for (uint64_t fb = sbase + 2 * SP_SPAN; fb < limit; fb += SP_SPAN)
            {
              if (++steps > SP_FAR_SPANS)
              {
                bad |= 4u;
                break;
              }
              const SpanMasks far = eval_masks(t, P, T, s_flags, via, fb + lane * 16, limit, true, true, false);
              const SpanCarry cf = span_carry(far);
              const uint32_t o0 = cf.out(0);
              if (cf.out(1) == o0)
              {
                far_val = o0;
                far_base = fb;
                break;
              }
            }
          }
          cin_span = far_val;
        }
        const SpanCarry cc = span_carry(cur);
        uint32_t unused;
        a16 = flood16(cur.cand, cur.cbk, cc.into(cin_span, lane), unused);
      }
      if (!lazy)
      {
        if (probing)
        {
          probing = false;
          via_keep = __reduce_add_sync(0xffffffffu, __popc(a16 & ~cur.via)) >= 32u;
          via_only = cover && via_keep && __reduce_add_sync(0xffffffffu, __popc(cur.via & ~a16)) <= 16u;
          via_r = via_keep;
        }
        a16 &= cur.via; // a position that cannot start a match needs no attempt (its D is 0 either way)
      }
      // ---- 3. D(p) for the positions of A: compaction, then rounds of one position per lane (longest_in_span)
      {
        const uint32_t cnt = __popc(a16);
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1)
        {
          const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
          if (lane >= static_cast<uint32_t>(d))
            incl += y;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t at = incl - cnt;
        uint32_t todo = a16;
        while (todo != 0)
        {
          const uint32_t k = __ffs(todo) - 1;
          todo &= todo - 1;
          queue[at++] = static_cast<uint16_t>(lane * 16 + k);
        }
        __syncwarp();
        const uint8_t* __restrict__ sp = buf + sbase;
        const uint32_t rel_end = n - sbase > 0x7fffffffull ? 0x7fffffffu : static_cast<uint32_t>(n - sbase);
        // rounds of 32 positions, one per lane (the viability table leaves less than a round per span on config 5)
        for (uint32_t qb = 0; qb < total; qb += 32)
        {
          if (qb + lane < total)
          {
            const uint32_t off = queue[qb + lane];
            // (a position that starts a match is in A when `cover` holds — away from the end of the buffer, where the
            // prefilters' clauses differ — and one that does not start a match does not count either way)
            if (!lazy || (cover && sbase + off + 32 <= t.end) || in_attempt_set(t, P, T, s_flags, sbase + off, bad))
            {
              uint32_t best;
              if (P.one)
              {
                // the candidate test was the exact literal (lib/matcher.cpp:71-83)
                if (P.len >= SP_LONG)
                  bad |= 2u;
                best = (1u << 16) | P.len;
              }
              else
                best = longest_in_span(P, step, sp, off, rel_end, bad);
              if (best != 0)
              {
                dtab[off] = best;
                atomicOr(&succ[off >> 5], 1u << (off & 31));
              }
            }
          }
          __syncwarp();
        }
        __syncwarp();
      }
      uint32_t succ16 = (succ[lane >> 1] >> (16 * (lane & 1))) & 0xffffu;
      __syncwarp();
      if (lane < 16)
        succ[lane] = 0;
      // ---- the window before the region: only the chain state at the region start is wanted
      if (s < 0)
      {
        const uint32_t NL = __ballot_sync(0xffffffffu, cur.nl != 0);
        if (NL != 0)
        {
          // fresh after the window's last newline
          const uint32_t ln = 31u - __clz(NL);
          const uint32_t xb = 31u - __clz(__shfl_sync(0xffffffffu, cur.nl, ln));
          if (lane < ln)
            succ16 = 0;
          else if (lane == ln)
            succ16 &= ~((2u << xb) - 1u);
          cursor = static_cast<int64_t>(ln * 16 + xb + 1);
        }
        else
        {
          // fresh from the window's first success: to be validated against earlier regions' farthest match end
          const uint32_t S = __ballot_sync(0xffffffffu, succ16 != 0);
          uint64_t v = rb;
          if (S != 0)
          {
            const uint32_t fl = __ffs(S) - 1;
            v = sbase + fl * 16 + (__ffs(__shfl_sync(0xffffffffu, succ16, fl)) - 1);
          }
          vpoint = v;
          cursor = 0;
        }
      }
      // ---- 4. the chain over this span's successes
      const uint32_t S = __ballot_sync(0xffffffffu, succ16 != 0);
      uint32_t sel = 0;
      int64_t e_out = 0;
      uint64_t far_end = 0;
      if (S != 0)
      {
        // every lane on its own, assuming the cursor is at or before its first success
        const int32_t lbase = static_cast<int32_t>(lane * 16);
        {
          int32_t e = 0;
          uint32_t m = succ16;
          while (m != 0)
          {
            const int32_t k = __ffs(m) - 1;
            m &= m - 1;
            const int32_t p = lbase + k;
            const int32_t end = p + static_cast<int32_t>(dtab[p] & 0xffffu);
            if (static_cast<uint64_t>(end) > far_end)
              far_end = end;
            if (p >= e)
            {
              sel |= 1u << k;
              e = end;
            }
          }
          e_out = e;
        }
        // the cursor that really reaches me: the previous success lane's, or the span's
        const uint32_t before = S & ((1u << lane) - 1u);
        const uint32_t pl = before != 0 ? 31u - __clz(before) : lane;
        const int64_t e_prev = __shfl_sync(0xffffffffu, e_out, pl);
        const int64_t e_in = before != 0 ? e_prev : cursor;
        const int32_t p1 = lbase + (__ffs(succ16) - 1);
        const bool ok = succ16 == 0 || e_in <= p1;
        if (!__all_sync(0xffffffffu, ok))
        {
          // a match straddles into some lane's first success: lane after lane from the first such lane
          const uint32_t first_bad = __ffs(__ballot_sync(0xffffffffu, !ok)) - 1;
          const uint32_t lower = S & ((1u << first_bad) - 1u);
          int64_t e = lower != 0 ? __shfl_sync(0xffffffffu, e_out, 31u - __clz(lower)) : cursor;
          uint32_t rest = S & ~((1u << first_bad) - 1u);
          while (rest != 0)
          {
            const uint32_t L = __ffs(rest) - 1;
            rest &= rest - 1;
            if (lane == L)
            {
              sel = 0;
              int64_t ee = e;
              uint32_t m = succ16;
              while (m != 0)
              {
                const int32_t k = __ffs(m) - 1;
                m &= m - 1;
                const int32_t p = lbase + k;
                if (p >= ee)
                {
                  sel |= 1u << k;
                  ee = p + static_cast<int32_t>(dtab[p] & 0xffffu);
                }
              }
              e_out = ee;
            }
            e = __shfl_sync(0xffffffffu, e_out, L);
          }
          cursor = e;
        }
        else
        {
          const int64_t last_e = __shfl_sync(0xffffffffu, e_out, 31u - __clz(S));
          cursor = last_e > cursor ? last_e : cursor;
        }
      }
      if (s >= 0)
      {
        // ---- ownership: the matches that start in spans 0..31 of this region
        const uint32_t nsel = __popc(sel);
        if (far_end != 0)
        {
          const uint64_t fe = sbase + far_end;
          if (s == SP_SPANS - 1)
            elast = fe > elast ? fe : elast;
          else
            emain = fe > emain ? fe : emain;
        }
        m_run += nsel;            // lane-private; reduced after the region
        nl_run += __popc(cur.nl);
        if (a.sel_bits != nullptr)
          a.sel_bits[(sbase >> 4) + lane] = static_cast<uint16_t>(sel);
      }
      __syncwarp(); // dtab / queue are rewritten by the next span
      cursor -= SP_SPAN;
      cur = nxt;
    }
    {
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
      {
        m_run += __shfl_down_sync(0xffffffffu, m_run, d);
        nl_run += __shfl_down_sync(0xffffffffu, nl_run, d);
        const uint64_t x = __shfl_down_sync(0xffffffffu, emain, d), y = __shfl_down_sync(0xffffffffu, elast, d);
        emain = x > emain ? x : emain;
        elast = y > elast ? y : elast;
      }
      if (lane == 0)
      {
        a.reg_matches[r] = m_run;
        a.reg_newlines[r] = nl_run;
        a.reg_emain[r] = emain;
        a.reg_elast[r] = elast;
        a.reg_v[r] = vpoint;
      }
    }
  }
  if (bad != 0)
    atomicOr(a.flags, bad);
}

// one anchored attempt for a known match start: (accept << 16) | length of the longest match
__device__ __forceinline__ uint32_t longest_at(const Text& t, const DevPattern& P, const Stepper& step, uint64_t pos)
{
  if (P.one)
    return (1u << 16) | P.len;
  uint32_t state = 0, best = 0;
  uint64_t p = pos;
  for (;;)
  {
    if (p >= t.end)
      break;
    const uint32_t nx = step(state, t.raw(p++));
    if (nx == D_DEAD)
      break;
    if (nx >= P.first_acc)
    {
      const uint32_t acc = __ldg(P.accept + nx);
      if ((acc & 0x7fffffffu) != 0)
        best = ((acc & 0x7fffu) << 16) | static_cast<uint32_t>((p - pos) & 0xffffu);
      if (acc & 0x80000000u)
        break;
    }
    state = nx;
  }
  return best;
}

// the records: span_scan_kernel left the selected match starts of every chunk in a.sel_bits and the final kernel turned
// the regions' counts into prefixes, so this pass only reads the text for its newlines (line numbers), re-runs the DFA
// at the few selected positions for length and accept index, and writes every record to its final place — input
// order, no atomics, no reorder pass.
template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS >= 512 ? 1 : 4)
span_emit_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, SpanArgs a)
{
  constexpr uint32_t NWARPS = THREADS / 32;
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  uint8_t* s_cls = smem;
  uint8_t* s_pred = s_cls + 256;
  uint8_t* s_tap = s_pred + UGX_HASH;
  uint16_t* s_next = reinterpret_cast<uint16_t*>(s_tap + UGX_BTAP);
  stage_tables_bulk(&s_bar, s_cls, P.cls, s_pred, P.pred, s_tap, P.tap, s_next, P.next,
                    a.stage_table ? ((P.table_bytes + 15) / 16) * 16 : 0);
  __syncthreads();
  Tables T;
  T.cls = s_cls;
  T.pred = s_pred;
  T.tap = s_tap;
  T.next = a.stage_table ? s_next : P.next;
  const Stepper step(T, P.ncls, a.stage_table != 0);
  const Text t{buf, n};
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint64_t limit = __ldcg(a.tail);
  const uint64_t nregions = (limit + SC_REGION - 1) / SC_REGION;
  const uint64_t total_warps = static_cast<uint64_t>(gridDim.x) * NWARPS;
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * NWARPS + wid; r < nregions; r += total_warps)
  {
    const uint64_t rb = r * SC_REGION;
    uint64_t idx0 = a.reg_matches[r];
    uint64_t line0 = a.reg_newlines[r] + 1 + a.base_line;
    for (int s = 0; s < SP_SPANS; ++s)
    {
      const uint64_t sbase = rb + static_cast<uint64_t>(s) * SP_SPAN;
      if (sbase >= limit)
        break;
      const uint64_t base = sbase + lane * 16;
      uint32_t nl = 0, sel = 0;
      if (base < limit)
      {
        const uint4 v = load_chunk_guarded(buf, n, base);
        nl = newline_mask_exact4(v.x, v.y, v.z, v.w);
        if (base + 16 > limit)
          nl &= (1u << (limit - base)) - 1u;
        sel = a.sel_bits[(sbase >> 4) + lane];
      }
      const uint32_t nsel = __popc(sel), nnl = __popc(nl);
      uint32_t mi = nsel, ni = nnl;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1)
      {
        const uint32_t y = __shfl_up_sync(0xffffffffu, mi, d), z = __shfl_up_sync(0xffffffffu, ni, d);
        if (lane >= static_cast<uint32_t>(d))
        {
          mi += y;
          ni += z;
        }
      }
      uint64_t idx = idx0 + (mi - nsel);
      const uint64_t lno = line0 + (ni - nnl);
      while (sel != 0)
      {
        const uint32_t k = __ffs(sel) - 1;
        sel &= sel - 1;
        const uint32_t d = longest_at(t, P, step, base + k);
        ugx_match rec;
        rec.line = lno + __popc(nl & ((1u << k) - 1u));
        rec.offset = base + k + a.base_offset;
        rec.len = d & 0xffffu;
        rec.cap = d >> 16;
        if (idx < a.out_cap)
          a.out[idx] = rec;
        ++idx;
      }
      idx0 += __shfl_sync(0xffffffffu, mi, 31);
      line0 += __shfl_sync(0xffffffffu, ni, 31);
    }
  }
}

// one CTA: exclusive prefixes of the regions' match / newline counts, the validation of the regions' chain starts,
// and the buffer's last line (line-at-a-time form, one thread).
// totals: [0] matches, [1] newlines, [2] fallback flag (1 = the spans' result is not valid), [3] matches before the
// last line, [4] newlines before the last line
template <bool EMIT>
__global__ void __launch_bounds__(1024)
span_final_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, SpanArgs a,
                  unsigned long long* __restrict__ totals)
{
  __shared__ uint64_t s_m[1024];  // inclusive prefix maximum of the farthest match ends over the tile (carry included)
  __shared__ uint64_t s_em[1024]; // emain of the tile's regions
  __shared__ uint64_t s_wf[32];
  __shared__ uint32_t s_wx[33], s_wy[33];
  __shared__ uint32_t s_viol;
  const uint64_t limit = a.tail[0];
  const uint64_t nreg = (limit + SC_REGION - 1) / SC_REGION;
  if (!EMIT)
  {
    // One pass over the regions in tiles of blockDim.x consecutive regions (coalesced loads), per tile three block
    // scans: exclusive sums of matches and newlines (they become the regions' record / line bases) and an inclusive
    // maximum of the farthest match ends.
    // Region i's chain start is valid when no success that starts before its window ends after its validation point:
    // far2 = the farthest end over regions <= i - 2 (window and all), prev_main = over spans 0..30 of region i - 1.
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, B = blockDim.x;
    if (tid == 0)
      s_viol = 0;
    uint64_t rx = 0, ry = 0;     // matches / newlines of the regions before the tile
    uint64_t all1 = 0, all2 = 0; // farthest end over the regions <= base - 1 / <= base - 2
    uint64_t pmain = 0;          // emain of region base - 1
    bool viol = false;
    // (the next tile's five values are loaded while this one is scanned: a tile is otherwise one round trip to memory
    // plus eight barriers, 3.7 us measured)
    uint64_t nx_m = 0, nx_n = 0, nx_em = 0, nx_el = 0, nx_v = SP_NO_V;
    if (tid < nreg)
    {
      nx_m = a.reg_matches[tid];
      nx_n = a.reg_newlines[tid];
      nx_em = a.reg_emain[tid];
      nx_el = a.reg_elast[tid];
      nx_v = a.reg_v[tid];
    }
    for (uint64_t base = 0; base < nreg; base += B)
    {
      const uint64_t i = base + tid;
      const bool in = i < nreg;
      const uint32_t cm = static_cast<uint32_t>(nx_m); // at most one per byte of a 16 KiB region
      const uint32_t cn = static_cast<uint32_t>(nx_n);
      const uint64_t em = nx_em, el = nx_el, v = nx_v;
      nx_m = nx_n = nx_em = nx_el = 0;
      nx_v = SP_NO_V;
      if (i + B < nreg)
      {
        nx_m = a.reg_matches[i + B];
        nx_n = a.reg_newlines[i + B];
        nx_em = a.reg_emain[i + B];
        nx_el = a.reg_elast[i + B];
        nx_v = a.reg_v[i + B];
      }
      uint64_t m = em > el ? em : el;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1)
      {
        const uint64_t y = __shfl_up_sync(0xffffffffu, m, d);
        if (lane >= static_cast<uint32_t>(d) && y > m)
          m = y;
      }
      if (lane == 31)
        s_wf[wid] = m;
      uint32_t tx, ty;
      const uint32_t ex = block_excl_scan(cm, s_wx, &tx); // (synchronises: s_wf is complete afterwards)
      const uint32_t ey = block_excl_scan(cn, s_wy, &ty);
      uint64_t before_warp = all1;
      for (uint32_t w = 0; w < wid; ++w)
        before_warp = s_wf[w] > before_warp ? s_wf[w] : before_warp;
      m = before_warp > m ? before_warp : m;
      s_m[tid] = m;
      s_em[tid] = em;
      __syncthreads();
      if (in)
      {
        const uint64_t far2 = tid >= 2 ? s_m[tid - 2] : (tid == 1 ? all1 : all2);
        const uint64_t prev_main = tid >= 1 ? s_em[tid - 1] : pmain;
        const uint64_t before = far2 > prev_main ? far2 : prev_main;
        if (v != SP_NO_V && before > v)
          viol = true;
        a.reg_matches[i] = rx + ex;
        a.reg_newlines[i] = ry + ey;
      }
      // carries (only used when another tile follows, i.e. this one was full)
      const uint64_t n1 = s_m[B - 1], n2 = s_m[B - 2], nm = s_em[B - 1];
      __syncthreads();
      all1 = n1;
      all2 = n2;
      pmain = nm;
      rx += tx;
      ry += ty;
    }
    if (viol)
      atomicOr(&s_viol, 1u);
    if (tid == 0)
    {
      totals[3] = rx;
      totals[4] = ry;
    }
    __syncthreads();
  }
  // ---- the last line: Matcher::match(FIND) again and again from its start (find_in_line)
  if (threadIdx.x == 0)
  {
    Tables T;
    T.cls = P.cls;
    T.next = P.next;
    T.pred = P.pred;
    T.tap = P.tap;
    const Text t{buf, n};
    uint64_t tail_matches = 0;
    const uint64_t before = totals[3];
    if (limit < n)
    {
      const uint64_t last = n - 1;
      const uint64_t lno = totals[4] + 1 + a.base_line;
      const CandMap cm{nullptr, 0, 0};
      Cursor m;
      set_current(t, m, limit);
      for (;;)
      {
        const uint32_t cap = find_in_line<false>(t, P, T, cm, m, last);
        if (cap == 0)
          break;
        if (EMIT)
        {
          ugx_match rec;
          rec.line = lno;
          rec.offset = m.txt + a.base_offset;
          rec.len = m.len;
          rec.cap = cap;
          if (before + tail_matches < a.out_cap)
            a.out[before + tail_matches] = rec;
        }
        ++tail_matches;
      }
    }
    if (!EMIT)
    {
      totals[0] = before + tail_matches;
      totals[1] = totals[4] + ((limit < n && buf[n - 1] == '\n') ? 1 : 0);
      totals[2] = (s_viol != 0 || (*a.flags) != 0) ? 1 : 0;
    }
  }
}

// ---- line records (ugx_find_lines) from the selected match starts ----
//
// A line is on the `ugrep -c` loop's list when it holds a selected start: the chain is fresh after every newline (no
// match crosses one), so the first selected start at or after a line's start is the match the loop's find() returns
// from there, and the loop then skips to the next line.  A line belongs to the region that holds its '\n'.  The count
// pass knows, per region, every owned line but the first; the first one began at or before the region start, and
// whether it matches also depends on the regions before: span_lines_final_kernel carries "last newline before the
// region" (max) and "first selected start since then" (a minimum that restarts at every region with a newline) over
// all regions, so a line over thousands of regions comes out of one prefix.

namespace {
constexpr uint64_t SL_NONE = ~0ull;
}

// count pass (EMIT = false): per region the SpanLinesArgs count values; emit pass: the records of the owned lines in
// their final slots (bases and carries from span_lines_final_kernel), and the last line's record from thread 0
template <bool EMIT, int THREADS>
__global__ void __launch_bounds__(THREADS, 4)
span_lines_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, SpanLinesArgs a)
{
  constexpr uint32_t NWARPS = THREADS / 32;
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  Tables T;
  if (EMIT)
  {
    // longest_at at the first selected start of every matching line
    uint8_t* s_cls = smem;
    uint8_t* s_pred = s_cls + 256;
    uint8_t* s_tap = s_pred + UGX_HASH;
    uint16_t* s_next = reinterpret_cast<uint16_t*>(s_tap + UGX_BTAP);
    stage_tables_bulk(&s_bar, s_cls, P.cls, s_pred, P.pred, s_tap, P.tap, s_next, P.next,
                      a.stage_table ? ((P.table_bytes + 15) / 16) * 16 : 0);
    __syncthreads();
    T.cls = s_cls;
    T.pred = s_pred;
    T.tap = s_tap;
    T.next = a.stage_table ? s_next : P.next;
  }
  const Text t{buf, n};
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const bool inv = a.invert != 0;
  const uint64_t limit = __ldcg(a.limit);
  const uint64_t nregions = (limit + SC_REGION - 1) / SC_REGION;
  const uint64_t total_warps = static_cast<uint64_t>(gridDim.x) * NWARPS;
  if (EMIT && blockIdx.x == 0 && threadIdx.x == 0 && a.tail[6] != 0)
  {
    const Stepper step(T, P.ncls, a.stage_table != 0);
    ugx_line rec;
    rec.line = a.tail[0];
    rec.bol = a.tail[1] + a.base_offset;
    rec.eol = a.tail[2] + a.base_offset;
    rec.offset = a.tail[3] + a.base_offset;
    uint64_t lc = a.tail[4];
    if (lc == SL_NONE)
    {
      const uint32_t d = longest_at(t, P, step, a.tail[3]);
      lc = (static_cast<uint64_t>(d >> 16) << 32) | (d & 0xffffu);
    }
    rec.len = static_cast<uint32_t>(lc);
    rec.cap = static_cast<uint32_t>(lc >> 32);
    if (a.tail[5] < a.out_cap)
      a.out[a.tail[5]] = rec;
  }
  for (uint64_t r = static_cast<uint64_t>(blockIdx.x) * NWARPS + wid; r < nregions; r += total_warps)
  {
    const uint64_t rb = r * SC_REGION;
    // warp-uniform state at the current span: first selected start since the last newline, start of the current line
    uint64_t first = EMIT ? a.reg_fa[r] : SL_NONE;
    uint64_t bol = EMIT ? a.reg_bol[r] : 0;
    uint64_t idx0 = EMIT ? a.reg_m[r] : 0;
    uint64_t line0 = EMIT ? a.reg_nl[r] + 1 + a.base_line : 0;
    uint64_t nl_run = 0, fb = SL_NONE;
    uint32_t m_run = 0; // lane-private: matching owned lines but the region's first
    for (int s = 0; s < SP_SPANS; ++s)
    {
      const uint64_t sbase = rb + static_cast<uint64_t>(s) * SP_SPAN;
      if (sbase >= limit)
        break;
      const uint64_t base = sbase + lane * 16;
      uint32_t nl = 0, sel = 0;
      if (base < limit)
      {
        const uint4 v = load_chunk_guarded(buf, n, base);
        nl = newline_mask_exact4(v.x, v.y, v.z, v.w);
        sel = a.sel_bits[(sbase >> 4) + lane];
        if (base + 16 > limit)
        {
          nl &= (1u << (limit - base)) - 1u;
          sel &= (1u << (limit - base)) - 1u;
        }
      }
      // per lane: the first selected start after its last newline (of the whole chunk without one), the start of the
      // line after its last newline, its newlines; then inclusive scans over the lanes (the first one restarts at every
      // lane with a newline)
      const uint32_t hb = nl != 0 ? 31u - __clz(nl) : 0u;
      const uint32_t after = nl != 0 ? sel & ~((2u << hb) - 1u) : sel;
      uint64_t v = after != 0 ? base + __ffs(after) - 1 : SL_NONE;
      uint64_t lp = nl != 0 ? base + hb + 1 : 0;
      uint32_t f = nl != 0 ? 1u : 0u, cnt = __popc(nl);
#pragma unroll
      for (int d = 1; d < 32; d <<= 1)
      {
        const uint64_t yv = __shfl_up_sync(0xffffffffu, v, d), yl = __shfl_up_sync(0xffffffffu, lp, d);
        const uint32_t yf = __shfl_up_sync(0xffffffffu, f, d), yc = __shfl_up_sync(0xffffffffu, cnt, d);
        if (lane >= static_cast<uint32_t>(d))
        {
          if (f == 0)
            v = yv < v ? yv : v;
          f |= yf;
          lp = yl > lp ? yl : lp;
          cnt += yc;
        }
      }
      uint64_t ev = __shfl_up_sync(0xffffffffu, v, 1), el = __shfl_up_sync(0xffffffffu, lp, 1);
      uint32_t ef = __shfl_up_sync(0xffffffffu, f, 1), ec = __shfl_up_sync(0xffffffffu, cnt, 1);
      if (lane == 0)
      {
        ev = SL_NONE;
        el = 0;
        ef = 0;
        ec = 0;
      }
      const uint64_t c_in = ef != 0 ? ev : (first < ev ? first : ev); // positions grow: the minimum is the earliest
      const uint64_t b_in = el > bol ? el : bol;
      // the lines that end in my chunk, in order: first match = the carry, else the first selected start on the line
      uint64_t fb_lane = SL_NONE;
      uint32_t my_recs = 0;
      uint64_t my_idx = 0;
      for (int pass = 0; pass < (EMIT ? 2 : 1); ++pass)
      {
        if (EMIT && pass == 1)
        {
          const uint32_t ex = warp_excl_scan(my_recs, lane);
          my_idx = idx0 + ex;
          idx0 += __shfl_sync(0xffffffffu, ex + my_recs, 31);
        }
        uint64_t c = c_in, lb = b_in;
        uint32_t from = 0, j = 0, mm = nl;
        while (mm != 0)
        {
          const uint32_t k = __ffs(mm) - 1;
          mm &= mm - 1;
          const uint32_t seg = sel & ((1u << k) - 1u) & ~((1u << from) - 1u);
          const uint64_t fm = c != SL_NONE ? c : (seg != 0 ? base + __ffs(seg) - 1 : SL_NONE);
          if (!EMIT)
          {
            if (nl_run == 0 && ec == 0 && j == 0)
              fb_lane = fm; // the region's first owned line: the final kernel adds what came before
            else
              m_run += fm != SL_NONE ? 1u : 0u;
          }
          else if ((fm != SL_NONE) != inv)
          {
            if (pass == 0)
              ++my_recs;
            else
            {
              ugx_line rec;
              rec.line = line0 + ec + j;
              rec.bol = lb + a.base_offset;
              rec.eol = base + k + a.base_offset;
              if (inv)
              {
                rec.offset = rec.bol;
                rec.len = 0;
                rec.cap = 0;
              }
              else
              {
                const Stepper step(T, P.ncls, a.stage_table != 0);
                const uint32_t d = longest_at(t, P, step, fm);
                rec.offset = fm + a.base_offset;
                rec.len = d & 0xffffu;
                rec.cap = d >> 16;
              }
              if (my_idx < a.out_cap)
                a.out[my_idx] = rec;
              ++my_idx;
            }
          }
          c = SL_NONE;
          from = k + 1;
          lb = base + k + 1;
          ++j;
        }
      }
      if (!EMIT && nl_run == 0)
      {
        const uint32_t any = __ballot_sync(0xffffffffu, nl != 0);
        if (any != 0)
          fb = __shfl_sync(0xffffffffu, fb_lane, __ffs(any) - 1);
      }
      const uint64_t v31 = __shfl_sync(0xffffffffu, v, 31), l31 = __shfl_sync(0xffffffffu, lp, 31);
      const uint32_t f31 = __shfl_sync(0xffffffffu, f, 31), c31 = __shfl_sync(0xffffffffu, cnt, 31);
      first = f31 != 0 ? v31 : (first < v31 ? first : v31);
      bol = l31 > bol ? l31 : bol;
      nl_run += c31;
      line0 += c31;
    }
    if (!EMIT)
    {
      const uint32_t m_tot = __reduce_add_sync(0xffffffffu, m_run);
      if (lane == 0)
      {
        a.reg_nl[r] = nl_run;
        a.reg_m[r] = m_tot;
        a.reg_bol[r] = bol;
        a.reg_fb[r] = fb;
        a.reg_fa[r] = first;
      }
    }
  }
}

// one CTA over the regions in tiles of blockDim.x: the carries (last newline, first selected start since it) into every
// region, its number of records (the first owned line matches when it has a selected start before the region's first
// newline or the carry has one), record and line bases; then the buffer's last line: the line after the last newline
// when the spans own the end of the buffer, or the set-aside last line (one find_in_line from its start)
__global__ void __launch_bounds__(1024)
span_lines_final_kernel(const __grid_constant__ DevPattern P, const uint8_t* __restrict__ buf, uint64_t n, SpanLinesArgs a,
                        unsigned long long* __restrict__ totals)
{
  __shared__ uint64_t s_v[32], s_l[32];
  __shared__ uint32_t s_f[32];
  __shared__ uint32_t s_wx[33], s_wy[33];
  __shared__ uint64_t s_carry[2];
  const uint64_t limit = a.limit[0];
  const uint64_t nreg = (limit + SC_REGION - 1) / SC_REGION;
  const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, B = blockDim.x;
  uint64_t c_nl = 0, c_rec = 0, c_bol = 0, c_first = SL_NONE; // over the regions before the tile
  for (uint64_t base = 0; base < nreg; base += B)
  {
    const uint64_t i = base + tid;
    const bool in = i < nreg;
    const uint64_t nl = in ? a.reg_nl[i] : 0, m = in ? a.reg_m[i] : 0, fb = in ? a.reg_fb[i] : SL_NONE;
    uint64_t v = in ? a.reg_fa[i] : SL_NONE, l = in ? a.reg_bol[i] : 0;
    uint32_t f = nl != 0 ? 1u : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
      const uint64_t yv = __shfl_up_sync(0xffffffffu, v, d), yl = __shfl_up_sync(0xffffffffu, l, d);
      const uint32_t yf = __shfl_up_sync(0xffffffffu, f, d);
      if (lane >= static_cast<uint32_t>(d))
      {
        if (f == 0)
          v = yv < v ? yv : v;
        f |= yf;
        l = yl > l ? yl : l;
      }
    }
    if (lane == 31)
    {
      s_v[wid] = v;
      s_l[wid] = l;
      s_f[wid] = f;
    }
    __syncthreads();
    uint64_t pv = c_first, pl = c_bol; // everything before my warp
    for (uint32_t w = 0; w < wid; ++w)
    {
      pv = s_f[w] != 0 ? s_v[w] : (s_v[w] < pv ? s_v[w] : pv);
      pl = s_l[w] > pl ? s_l[w] : pl;
    }
    uint64_t ev = __shfl_up_sync(0xffffffffu, v, 1), el = __shfl_up_sync(0xffffffffu, l, 1);
    uint32_t ef = __shfl_up_sync(0xffffffffu, f, 1);
    if (lane == 0)
    {
      ev = SL_NONE;
      el = 0;
      ef = 0;
    }
    const uint64_t first_in = ef != 0 ? ev : (pv < ev ? pv : ev);
    const uint64_t bol_in = el > pl ? el : pl;
    const uint32_t matched = nl == 0 ? 0u : static_cast<uint32_t>(m) + ((fb != SL_NONE || first_in != SL_NONE) ? 1u : 0u);
    const uint32_t recs = a.invert != 0 ? static_cast<uint32_t>(nl) - matched : matched;
    uint32_t tx, ty;
    const uint32_t ex = block_excl_scan(recs, s_wx, &tx);
    const uint32_t ey = block_excl_scan(static_cast<uint32_t>(nl), s_wy, &ty);
    if (in)
    {
      a.reg_nl[i] = c_nl + ey;
      a.reg_m[i] = c_rec + ex;
      a.reg_bol[i] = bol_in;
      a.reg_fa[i] = first_in;
    }
    if (tid == B - 1)
    {
      s_carry[0] = f != 0 ? v : (pv < v ? pv : v);
      s_carry[1] = l > pl ? l : pl;
    }
    __syncthreads();
    c_first = s_carry[0];
    c_bol = s_carry[1];
    c_nl += ty;
    c_rec += tx;
    __syncthreads();
  }
  if (tid == 0)
  {
    uint64_t present = 0, tbol = 0, teol = 0, off = SL_NONE, lc = 0, tail_nl = 0;
    if (limit < n)
    {
      // the set-aside last line: the `ugrep -c` loop's first find() from its start
      Tables T;
      T.cls = P.cls;
      T.next = P.next;
      T.pred = P.pred;
      T.tap = P.tap;
      const Text t{buf, n};
      const CandMap cm{nullptr, 0, 0};
      Cursor m;
      set_current(t, m, limit);
      const uint32_t cap = find_in_line<false>(t, P, T, cm, m, n - 1);
      tail_nl = buf[n - 1] == '\n' ? 1 : 0;
      present = 1;
      tbol = limit;
      teol = tail_nl != 0 ? n - 1 : n;
      if (cap != 0)
      {
        off = m.txt;
        lc = (static_cast<uint64_t>(cap) << 32) | m.len;
      }
    }
    else if (n > 0 && buf[n - 1] != '\n')
    {
      // an unterminated line the spans own: carried like a region's first line (longest_at runs in the emit pass)
      present = 1;
      tbol = c_bol;
      teol = n;
      off = c_first;
      lc = SL_NONE;
    }
    const bool rec = present != 0 && (off != SL_NONE) != (a.invert != 0);
    a.tail[0] = c_nl + 1 + a.base_line;
    a.tail[1] = tbol;
    a.tail[2] = teol;
    a.tail[3] = a.invert != 0 ? tbol : off;
    a.tail[4] = a.invert != 0 ? 0 : lc;
    a.tail[5] = c_rec;
    a.tail[6] = rec ? 1 : 0;
    totals[0] = c_rec + (rec ? 1 : 0);
    totals[1] = c_nl + tail_nl;
  }
}

// ---- host side ----

bool span_scan_eligible(const DevPattern& P)
{
  return P.has_meta == 0 && (P.flags & UGX_OPT_W) == 0 && P.acc0 == 0 && P.adv != UGX_ADV_NONE &&
         (P.lbk == 0 || P.lbk == 0xffff);
}

static int span_threads(const DevPattern& P)
{
  if (P.table_bytes <= 24 * 1024)
    return 256;
  if (P.table_bytes <= 110 * 1024)
    return 1024;
  if (P.table_bytes <= 160 * 1024)
    return 512;
  return 256; // the table stays in global memory / L2
}

static size_t span_smem_bytes(const DevPattern& P, bool stage, bool use_via, int threads)
{
  return 256 + UGX_HASH + UGX_BTAP + 256 + static_cast<size_t>(threads / 32) * (SP_SPAN * 4 + 64 + SP_SPAN * 2) +
         (use_via ? via_smem_bytes(P) : 0) + (stage ? ((P.table_bytes + 15) / 16) * 16 : 0);
}

template <bool EMIT, int THREADS>
static cudaError_t launch_span_one(const DevPattern& P, const uint8_t* buf, uint64_t n, SpanArgs a, size_t smem, int sm_count,
                                   cudaStream_t st)
{
  auto kern = EMIT ? span_emit_kernel<THREADS> : span_scan_kernel<THREADS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, UGX_MAX_DYN_SMEM);
  if (e != cudaSuccess)
    return e;
  int per_sm = 1;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
  if (e != cudaSuccess)
    return e;
  if (per_sm < 1)
    per_sm = 1;
  uint64_t g = static_cast<uint64_t>(sm_count) * per_sm;
  const uint64_t need = ((n + SC_REGION - 1) / SC_REGION + THREADS / 32 - 1) / (THREADS / 32);
  if (g > need)
    g = need;
  if (g == 0)
    g = 1;
  kern<<<static_cast<int>(g), THREADS, smem, st>>>(P, buf, n, a);
  return cudaGetLastError();
}

cudaError_t launch_last_line(const uint8_t* buf, uint64_t n, uint64_t* tail, cudaStream_t st)
{
  last_line_kernel<<<1, 32, 0, st>>>(buf, n, tail);
  return cudaGetLastError();
}

cudaError_t launch_span_scan(const DevPattern& P, const uint8_t* buf, uint64_t n, SpanArgs a, bool emit, int sm_count,
                             cudaStream_t st)
{
  const int threads = span_threads(P);
  // the viability tables are small and spare most attempts: they get shared memory before the transition table does
  const bool use_via = P.via_k != 0 && span_smem_bytes(P, false, true, threads) <= static_cast<size_t>(UGX_MAX_DYN_SMEM);
  const bool stage = P.table_bytes <= 160 * 1024 &&
                     span_smem_bytes(P, true, use_via, threads) <= static_cast<size_t>(UGX_MAX_DYN_SMEM);
  const size_t smem = emit ? 256 + UGX_HASH + UGX_BTAP + (stage ? ((P.table_bytes + 15) / 16) * 16 : 0)
                           : span_smem_bytes(P, stage, use_via, threads);
  a.stage_table = stage ? 1u : 0u;
  a.use_via = use_via ? 1u : 0u;
#define UGX_SPAN_GO(EMITF)                                                        \
  do                                                                              \
  {                                                                               \
    if (threads == 1024)                                                          \
      return launch_span_one<EMITF, 1024>(P, buf, n, a, smem, sm_count, st);      \
    if (threads == 512)                                                           \
      return launch_span_one<EMITF, 512>(P, buf, n, a, smem, sm_count, st);       \
    return launch_span_one<EMITF, 256>(P, buf, n, a, smem, sm_count, st);         \
  } while (0)
  if (emit)
    UGX_SPAN_GO(true);
  UGX_SPAN_GO(false);
#undef UGX_SPAN_GO
}

cudaError_t launch_span_final(const DevPattern& P, const uint8_t* buf, uint64_t n, const SpanArgs& a, bool emit,
                              unsigned long long* totals, cudaStream_t st)
{
  if (emit)
    span_final_kernel<true><<<1, 32, 0, st>>>(P, buf, n, a, totals); // the last line's records: one thread
  else
    span_final_kernel<false><<<1, 1024, 0, st>>>(P, buf, n, a, totals);
  return cudaGetLastError();
}

cudaError_t launch_span_lines(const DevPattern& P, const uint8_t* buf, uint64_t n, SpanLinesArgs a, bool emit, int sm_count,
                              cudaStream_t st)
{
  constexpr int THREADS = 256;
  // the emit pass runs longest_at once per matching line: the transition table is staged when it fits
  const bool stage = emit && 256 + UGX_HASH + UGX_BTAP + ((P.table_bytes + 15) / 16) * 16 <= static_cast<uint32_t>(UGX_MAX_DYN_SMEM);
  const size_t smem = emit ? 256 + UGX_HASH + UGX_BTAP + (stage ? ((P.table_bytes + 15) / 16) * 16 : 0) : 0;
  a.stage_table = stage ? 1u : 0u;
  auto kern = emit ? span_lines_kernel<true, THREADS> : span_lines_kernel<false, THREADS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, UGX_MAX_DYN_SMEM);
  if (e != cudaSuccess)
    return e;
  int per_sm = 1;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
  if (e != cudaSuccess)
    return e;
  if (per_sm < 1)
    per_sm = 1;
  uint64_t g = static_cast<uint64_t>(sm_count) * per_sm;
  const uint64_t need = ((n + SC_REGION - 1) / SC_REGION + THREADS / 32 - 1) / (THREADS / 32);
  if (g > need)
    g = need;
  if (g == 0)
    g = 1;
  kern<<<static_cast<int>(g), THREADS, smem, st>>>(P, buf, n, a);
  return cudaGetLastError();
}

cudaError_t launch_span_lines_final(const DevPattern& P, const uint8_t* buf, uint64_t n, const SpanLinesArgs& a,
                                    unsigned long long* totals, cudaStream_t st)
{
  span_lines_final_kernel<<<1, 1024, 0, st>>>(P, buf, n, a, totals);
  return cudaGetLastError();
}

} // namespace ugx
